#!/bin/bash
# GPU box with N GPUs: the default sharded bench (config 3, global batch 65536) -> gpurun_out/r02_bench_${N}gpu.json
set -u
N=${1:-2}
mkdir -p gpurun_out
unset AFT_B200_LIB
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus $N --steps 5 --warmup 3 --no-cpu-baseline > gpurun_out/r02_bench_${N}gpu.json 2> gpurun_out/r02_bench_${N}gpu.err
python - <<PY
import json
d=json.loads([l for l in open("gpurun_out/r02_bench_${N}gpu.json").read().strip().splitlines() if l.startswith("{")][-1])
print("N=$N value %.0f e2e %.0f ms %.2f" % (d["value"], d["e2e"]["value"], d["ms_per_step"]), d["stages_ms_per_step"], d["collectives"])
PY
