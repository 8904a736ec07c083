#!/bin/bash
# round 2: per-phase cycle counts of the softmax warps (build with -DESF_ATTN_TIMING; clock64 around the loop phases)
set -u
cd "$(dirname "$0")/../.."
O=gpurun_out/r2_s34
mkdir -p $O
export ESF_NVCC_EXTRA=-DESF_ATTN_TIMING
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1 || { tail -5 $O/build.log; exit 1; }
for d in 8 32; do
  echo "== d = $d"; python tools/prof_attn.py $d 8 56 4 1 2>&1 | grep -E "^warp|attn tc" | sort | head -20
done | tee $O/timing.txt
