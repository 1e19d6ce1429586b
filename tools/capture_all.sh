#!/bin/bash
# usage: gpurun --timeout 2400 -- 'bash tools/capture_all.sh <tag>'   (tests + breakdown + bench, then the ncu capture)
# (every step under its own timeout: a hung kernel must not eat the GPU budget)
set -u
T=$1
O=gpurun_out
mkdir -p $O
timeout 1000 python -m pytest tests -m gpu -q -x --timeout 240 > $O/${T}_pytest.log 2>&1; echo "pytest rc=$?"; tail -6 $O/${T}_pytest.log
timeout 200 python tools/kernel_breakdown.py --cfg 1 3 4b 5 > $O/${T}_breakdown.md 2> $O/${T}_breakdown.err; echo "breakdown rc=$?"; cut -d'|' -f2-9,13- $O/${T}_breakdown.md; tail -3 $O/${T}_breakdown.err
timeout 300 python bench.py --no-cpu-baseline > $O/${T}_bench.json 2> $O/${T}_bench.err; echo "bench rc=$?"; cut -c1-200 $O/${T}_bench.json
bash tools/capture_prof.sh ${T}p
