#!/bin/bash
# GPU box with N GPUs: the sharded default bench (config 3) and BASELINE configs[4] as independent replicas.
set -u
N=${1:-8}
mkdir -p gpurun_out
unset AFT_B200_LIB
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus $N --steps 5 --warmup 3 --no-cpu-baseline > gpurun_out/r02_bench_${N}gpu.json 2> gpurun_out/r02_bench_${N}gpu.err
grep "^{" gpurun_out/r02_bench_${N}gpu.json | tail -1 | cut -c1-3000
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29513 tools/config5_mgpu.py 64 2 > gpurun_out/r02_config5_${N}gpu.json 2> gpurun_out/r02_config5_${N}gpu.err
grep "^{" gpurun_out/r02_config5_${N}gpu.json | tail -1; tail -3 gpurun_out/r02_config5_${N}gpu.err
