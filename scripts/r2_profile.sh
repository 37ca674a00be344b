#!/bin/bash
# round-2 profiling pass on a B200 in one run: launch list, ncu --set full of the hot kernels.
# outputs under gpurun_out/ (summaries are copied to profiles/ afterwards)
set -x
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
# 1. launch list of the default bench command
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file gpurun_out/r2_launches.csv python bench.py --steps 2 --warmup 1 --no-e2e --no-cpu-baseline > gpurun_out/r2_launches_bench.log 2>&1
# 2. full capture of the fragment kernels and of the partitioned aggregate
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_frag_ -c 3 -o gpurun_out/r2_frag python bench.py --steps 1 --warmup 1 --no-e2e --no-cpu-baseline > gpurun_out/r2_frag_ncu.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_aggp -c 4 -o gpurun_out/r2_aggp python tools/groupby_highcard.py --rows 200000000 --keys 20000000 --reps 1 > gpurun_out/r2_aggp_ncu.log 2>&1
ls -la gpurun_out | tail -12
