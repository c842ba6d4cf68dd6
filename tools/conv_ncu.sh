#!/bin/bash
# GPU box: full ncu capture of one frontend_tc_kernel and one head_tc_kernel launch of the driver workload.
set -u
mkdir -p gpurun_out
unset AFT_B200_LIB
for k in frontend_tc_kernel head_tc_kernel; do
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:$k -s 10 -c 1 -f -o gpurun_out/r02_$k python bench.py --steps 1 --warmup 3 --no-cpu-baseline --e2e-steps 0 --no-extra > gpurun_out/r02_${k}_ncu.log 2>&1
  tail -1 gpurun_out/r02_${k}_ncu.log | cut -c1-160
done
