#!/bin/bash
# round 2: ncu --set full of the temporal-band stem at the headline shape
set -u
cd "$(dirname "$0")/../.."
O=gpurun_out/r2_s26
mkdir -p $O
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1 || { tail -5 $O/build.log; exit 1; }
python tools/prof_stem.py 64 20 | tee $O/time.txt
python tools/prof_stem.py 64 20 1 | tee -a $O/time.txt
timeout 600 ncu --set full --clock-control none --import-source on -k regex:stem_tband -s 2 -c 1 -o $O/stem_tband_b64 -f python tools/prof_stem.py 64 3 > $O/ncu.log 2>&1; tail -2 $O/ncu.log
