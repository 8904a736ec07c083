#!/bin/bash
# round 2: temporal-band stem kernel -- kernel tests and time against the banded stem at the headline shape:
#   gpurun -- 'bash tools/sessions/r2_s24_stem_tband.sh'                                  tests + A/B (+ BENCH=1: bench)
set -u
cd "$(dirname "$0")/../.."
O=gpurun_out/r2_s24
mkdir -p $O
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1 || { tail -5 $O/build.log; exit 1; }
if [ "${TESTS:-1}" = 1 ]; then
  timeout 600 python -m pytest tests/test_gpu_kernels.py -x -q -m gpu -k "stem" > $O/pytest.log 2>&1; echo "pytest rc $?"; tail -3 $O/pytest.log
fi
{
  python tools/prof_stem.py 64 20 1
  python tools/prof_stem.py 64 20
} | tee $O/stem_ab.txt
if [ "${BENCH:-0}" = 1 ]; then
  timeout 900 python bench.py --steps 10 --warmup 3 --no-extra-configs > $O/bench.json 2> $O/bench.err; echo "bench rc $?"
  tail -1 $O/bench.json | cut -c1-200
fi
