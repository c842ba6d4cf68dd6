#!/bin/bash
# GPU box: parity of the bf16 forward, conv-kernel timeline (tl build) and a short bench of both workloads.
set -u
mkdir -p gpurun_out
unset AFT_B200_LIB
tag=${1:-conv}
timeout 300 python tools/tc_check.py fwd 2>&1 | tail -4
if [ -f adafortitran_b200/lib/libaft_b200_tl.so ]; then
  AFT_B200_LIB=$PWD/adafortitran_b200/lib/libaft_b200_tl.so timeout 300 python tools/tc_check.py timeline 2>&1 | grep CONV
fi
for wl in ada forti; do
  timeout 400 python bench.py --workload $wl --steps 4 --warmup 3 --no-cpu-baseline --e2e-steps 0 --no-extra > gpurun_out/${tag}_$wl.json 2> gpurun_out/${tag}_$wl.err
  python - <<PY
import json
try:
    d=json.loads(open("gpurun_out/${tag}_$wl.json").read().strip().splitlines()[-1])
    print("$wl", "est/s %.0f" % d["value"], "ms %.2f" % d["ms_per_step"], "stages", {k: round(x,2) for k,x in d["stages_ms_per_step"].items()}, "frac %.4f" % d["roofline"]["frac"])
except Exception as e:
    print("bench $wl failed", e); print(open("gpurun_out/${tag}_$wl.err").read()[-600:])
PY
done
