#!/bin/bash
# GPU box: the round's evidence files (launch list, full ncu capture of the encoder kernel, one bench line with the CPU arm).
set -u
mkdir -p gpurun_out
unset AFT_B200_LIB
timeout 600 python bench.py --steps 5 --warmup 3 > gpurun_out/r02_bench_1gpu_final.json 2> gpurun_out/r02_bench_1gpu_final.err
tail -c 600 gpurun_out/r02_bench_1gpu_final.json
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r02_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu-baseline --e2e-steps 0 --no-extra > gpurun_out/r02_launches.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:encoder_kernel -s 2 -c 1 -f -o gpurun_out/r02_encoder python bench.py --steps 1 --warmup 3 --no-cpu-baseline --e2e-steps 0 --no-extra > gpurun_out/r02_encoder_ncu.log 2>&1
tail -2 gpurun_out/r02_encoder_ncu.log | cut -c1-200

timeout 600 python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/r02_bench_reference.json 2> gpurun_out/r02_bench_reference.err
tail -c 400 gpurun_out/r02_bench_reference.json
timeout 300 python tools/gates_report.py 2>&1 | tail -1 | tee gpurun_out/r02_gates_report.json
TARGETS=bf16 tools/sanitize.sh memcheck synccheck
