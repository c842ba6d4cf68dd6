"""LinearEstimator training on the GPU (reference shape 24 -> 1680, fp32).

Measures, in one run on one card:
  * aft_linear_backward kernel time (CUDA events over repeated calls), with and without grad_x, at batch 262144 (the
    forward's row in profiles/r02_aux_kernels.json) and 65536, against the computed bounds: HBM (grad_y + x, + grad_x
    when computed) and fp32 FMA on the CUDA cores (148 SMs x 128 lanes x 2 FLOP x max SM clock);
  * a full training step (forward, MSE loss, backward, torch.optim.Adam) of LinearEstimator with trainable = True, in
    samples/s, and the same step with stock nn.Linear fp32 autograd (TF32 off) as a comparison arm.
Every working set is larger than the 126 MB L2 (grad_y alone is 440 MB at 65536 and 1.76 GB at 262144), so each pass
reads grad_y from HBM.

  python tools/linear_train_bench.py --out profiles/r05_linear_train.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from adafortitran_b200 import LinearEstimator, ModelConfig, SystemConfig, _capi  # noqa: E402
from tests import util  # noqa: E402

IN, OUT = 24, 1680
HBM_GBS = 6551.0   # measured copy bandwidth of the B200 this project uses as its HBM peak (DESIGN §7)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=30)
    name, power, clock = (s.strip() for s in r.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def timed_ms(fn, min_s):
    """Mean ms per call over a window of at least min_s seconds (CUDA events), after warm-up."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n, total = 0, 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while total < min_s * 1e3:
        k = max(1, n or 5)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        n += k
    return total / n


def kernel_rows(batch, clock_mhz, min_s):
    lib = _capi.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    w = torch.randn(OUT, IN, device="cuda") / IN ** 0.5
    x = torch.randn(batch, IN, device="cuda")
    gy = torch.randn(batch, OUT, device="cuda")
    gw, gb, gx = torch.empty(OUT, IN, device="cuda"), torch.empty(OUT, device="cuda"), torch.empty(batch, IN, device="cuda")
    need = lib.aft_linear_backward_workspace_bytes(batch, IN, OUT)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    fma_peak = 148 * 128 * 2 * clock_mhz * 1e6
    rows = []
    for with_x in (False, True):
        call = lambda: _capi.check(lib.aft_linear_backward(vp(w), vp(x), vp(gy), vp(gw), vp(gb), vp(gx if with_x else None),
                                                           batch, IN, OUT, vp(ws), need, st))
        ms = timed_ms(call, min_s)
        nbytes = batch * 4 * (OUT + IN + (IN if with_x else 0))
        flop = batch * 2 * OUT * IN * (2 if with_x else 1)
        rate = batch / ms * 1e3
        hbm_rate = HBM_GBS * 1e9 / (nbytes / batch)
        fma_rate = fma_peak / (flop / batch)
        bound = "fma" if fma_rate < hbm_rate else "hbm"
        rows.append({"batch": batch, "grad_x": with_x, "ms": ms, "samples_per_s": rate,
                     "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / ms / 1e6, "flop": flop,
                     "achieved_tflops": flop / ms / 1e9, "bound": bound,
                     "bound_samples_per_s": min(hbm_rate, fma_rate), "fraction_of_bound": rate / min(hbm_rate, fma_rate),
                     "fraction_of_hbm": nbytes / ms / 1e6 / HBM_GBS, "launches_per_call": 3 if with_x else 2})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def step_rows(batch, min_s):
    """One training step per call: forward, MSE, backward, Adam; ours vs stock nn.Linear fp32 autograd."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    ours = LinearEstimator(SystemConfig(**util.SYS), ModelConfig(**dict(util.FORTI, model_type="linear", device="cuda")))
    ours.trainable = True
    ours.train()
    stock = torch.nn.Linear(IN, OUT).cuda()
    stock.load_state_dict({"weight": ours.linear.weight.detach().clone(), "bias": ours.linear.bias.detach().clone()})
    x = torch.randn(batch, 12, 2, device="cuda")
    t = torch.randn(batch, 120, 14, device="cuda")
    arms = {"ours": (ours, lambda m: m(x)), "torch_nn_linear_fp32": (stock, lambda m: m(x.reshape(batch, IN)).reshape(batch, 120, 14))}
    out = {}
    for name, (m, fwd) in arms.items():
        opt = torch.optim.Adam(m.parameters(), lr=1e-4)

        def step():
            opt.zero_grad(set_to_none=True)
            torch.nn.functional.mse_loss(fwd(m), t).backward()
            opt.step()
        ms = timed_ms(step, min_s)
        out[name] = {"batch": batch, "ms_per_step": ms, "samples_per_s": batch / ms * 1e3}
        print(name, json.dumps(out[name]), flush=True)
    out["speedup_vs_torch"] = out["ours"]["samples_per_s"] / out["torch_nn_linear_fp32"]["samples_per_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--window", type=float, default=2.0, help="seconds per timed window")
    args = ap.parse_args()
    gpu = card()
    t0 = time.time()
    res = {"gpu": gpu, "shape": {"in_dim": IN, "out_dim": OUT}, "hbm_gbs_assumed": HBM_GBS,
           "fma_peak_tflops": 148 * 128 * 2 * gpu["max_sm_clock_mhz"] * 1e6 / 1e12,
           "working_set": "larger than the 126 MB L2 at every batch: grad_y is 440 MB at 65536, 1.76 GB at 262144",
           "backward_kernels": [], "training_step": []}
    for batch in (262144, 65536):
        res["backward_kernels"] += kernel_rows(batch, gpu["max_sm_clock_mhz"], args.window)
    for batch in (65536, 262144):
        res["training_step"].append(step_rows(batch, args.window))
    res["wall_s"] = time.time() - t0
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
