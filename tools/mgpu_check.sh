#!/bin/bash
# N GPUs: the sharded bench at 8192 estimates per rank (the per-rank load of the 8-GPU run).
set -u
N=${1:-2}
mkdir -p gpurun_out
unset AFT_B200_LIB
timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus $N --global-batch $((8192*N)) --steps 6 --warmup 3 --no-cpu-baseline > gpurun_out/mgpu_${N}.json 2> gpurun_out/mgpu_${N}.err
python - <<PY
import json
try:
    d=json.loads([l for l in open("gpurun_out/mgpu_${N}.json").read().strip().splitlines() if l.startswith("{")][-1])
    print("N=$N value %.0f e2e %.0f ms %.2f" % (d["value"], d["e2e"]["value"], d["ms_per_step"]), d["stages_ms_per_step"], d["collectives"])
except Exception as e:
    print("failed", e); print(open("gpurun_out/mgpu_${N}.err").read()[-800:])
PY
