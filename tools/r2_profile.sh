#!/bin/bash
# Second GPU call of round 2 (after the first decided which kernel variant stays): the ncu evidence bench.py's
# roofline object refers to.  One GPU; ncu replays kernels, so nothing printed by these commands is a bench value.
#   gpurun --timeout 1800 -- 'bash tools/r2_profile.sh'
# then here:  python tools/ncu_summary.py gpurun_out/r2_tick13.ncu-rep > profiles/r2_ncu_tick13.txt   (etc.)
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
# 1. launch list of the bench command (share of the step per kernel)
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file gpurun_out/r2_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline > gpurun_out/r2_launches.log 2>&1
# 2. DRAM bytes of every tick launch of one run (bench.py's roofline.traffic: mean per launch) — tick t is the t-th tick_kernel launch
ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum -k regex:tick_kernel --clock-control none --csv \
    --log-file gpurun_out/r2_traffic_ncu.csv python tools/tick_profile.py --runs 1 > gpurun_out/r2_traffic.log 2>&1
# 3. full captures: plateau tick 13, ramp tick 9 (compaction path), second-wave tick 18, tail tick 28
for t in 13 9 18 28; do
  ncu --set full --clock-control none --import-source on -k regex:tick_kernel --launch-skip $t --launch-count 1 -f -o gpurun_out/r2_tick$t \
      python tools/tick_profile.py --runs 1 > gpurun_out/r2_ncu_tick$t.log 2>&1
done
ls -la gpurun_out/*.ncu-rep
