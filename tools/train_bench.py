"""Training-step benchmark: AdaFortiTran default config, dropout 0.1, one full step (training forward, the reference loss
-- MSE over concatenated real / imaginary parts --, backward, torch.optim.Adam.step) at several batch sizes.

Arms, interleaved window by window on the same card:
  ours  : AdaFortiTranEstimator with trainable = True (aft_forward_train / aft_backward, fp32 CUDA cores)
  torch : the same model in stock PyTorch fp32 autograd -- the reference under baseline/_ref when present, else
          oracle/torch_port.py in train mode (TF32 off, torch's default)

Timing: CUDA events around forward / backward / optimizer of every step, warm-up steps first, windows of at least
--window seconds.  FLOPs are counted from the shapes below (a training step = 3x the forward's multiply-adds x 2).

  python tools/train_bench.py --out profiles/r03_train_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import aft_oracle as O  # noqa: E402
from tests import util  # noqa: E402

L, S, D, FF, PIX, NP = 6, 280, 128, 256, 1680, 24


def forward_flops_per_sample(layers=L, in_dim=12):
    conv = 2 * PIX * 9 * (1 * 8 + 8 * 32 + 32 * 8 + 8 * 1)
    per_seq = (2 * NP * PIX + 2 * conv + 2 * S * in_dim * D + 2 * S * D * 6
               + layers * (2 * S * D * 3 * D + 2 * 2 * S * S * D + 2 * S * D * D + 2 * 2 * S * D * FF))
    return 2 * per_seq


def saved_bytes_per_sample(layers=L):
    per_seq = NP + PIX + S * D + layers * S * (D + 3 * D + D + 4 + D + D + FF + D)
    return 4 * (2 * per_seq + 3)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def make_batch(n, seed):
    pilots, snr, ds, dop = O.synthetic_batch(n, seed=seed)
    _, h = O.synthetic_channel(n, 15.0, 100.0, 600.0, seed=seed)
    dev = torch.device("cuda")
    return (torch.from_numpy(pilots).to(dev), [torch.from_numpy(np.asarray(v, np.float32)).to(dev) for v in (snr, ds, dop)],
            torch.from_numpy(h).to(dev))


def loss_fn(est, truth):
    return torch.nn.functional.mse_loss(torch.cat([est.real, est.imag], 1), torch.cat([truth.real, truth.imag], 1))


class Ours:
    name = "ours"

    def __init__(self):
        torch.manual_seed(0)
        self.model = util.make_model("ada", device="cuda")
        self.model.trainable = True
        self.model.train()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=5e-4)

    def forward(self, pilots, cond):
        z = torch.zeros_like(cond[0])
        return self.model(pilots, (z, cond[0], cond[1], cond[2], z, None))


class Stock:
    def __init__(self):
        torch.manual_seed(0)
        ref = os.path.join(ROOT, "baseline", "_ref")
        if os.path.isdir(os.path.join(ref, "src", "models")):
            sys.path.insert(0, ref)
            from src.config.schemas import ModelConfig, SystemConfig  # the reference's own
            from src.models import AdaFortiTranEstimator
            self.name = "reference (baseline/_ref)"
            self.model = AdaFortiTranEstimator(SystemConfig(**util.SYS), ModelConfig(**dict(util.ADA, device="cuda"))).cuda()
            self.kind = "ref"
        else:
            from oracle.torch_port import TorchPort
            self.name = "oracle/torch_port.py (stock PyTorch)"
            self.model = TorchPort(util.ada_weights()).cuda()
            self.kind = "port"
        self.model.train()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=5e-4)

    def forward(self, pilots, cond):
        c = [v.reshape(-1, 1) for v in cond]
        if self.kind == "ref":
            z = torch.zeros_like(c[0])
            return self.model(pilots, (z, c[0], c[1], c[2], z, None))
        return torch.complex(self.model._real(pilots.real, c), self.model._real(pilots.imag, c))


def window(arm, batch, seconds):
    pilots, cond, truth = batch
    ev = lambda: torch.cuda.Event(enable_timing=True)
    steps, fwd, bwd, opt = 0, 0.0, 0.0, 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    start = ev()
    start.record()
    while True:
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        loss = loss_fn(arm.forward(pilots, cond), truth)
        e1.record()
        arm.opt.zero_grad(set_to_none=True)
        loss.backward()
        e2.record()
        arm.opt.step()
        e3.record()
        e3.synchronize()
        fwd += e0.elapsed_time(e1)
        bwd += e1.elapsed_time(e2)
        opt += e2.elapsed_time(e3)
        steps += 1
        if time.perf_counter() - t0 >= seconds:
            break
    end = ev()
    end.record()
    end.synchronize()
    total = start.elapsed_time(end)
    return dict(steps=steps, ms_per_step=total / steps, fwd_ms=fwd / steps, bwd_ms=bwd / steps, opt_ms=opt / steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="32,256,1024")
    ap.add_argument("--window", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_train_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_bench: no CUDA device (this measurement runs on the GPU only)")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    arms = [Ours(), Stock()]
    from adafortitran_b200 import _capi
    res = dict(card=card(), torch=torch.__version__, config="AdaFortiTran default, dropout 0.1, Adam 5e-4, MSE(re|im)",
               stock_arm=arms[1].name, forward_flops_per_sample=forward_flops_per_sample(),
               step_flops_per_sample=3 * forward_flops_per_sample(), saved_bytes_per_sample=saved_bytes_per_sample(), rows=[])
    for b in [int(x) for x in args.batches.split(",")]:
        batch = make_batch(b, seed=b)
        for arm in arms:        # warm-up
            for _ in range(3):
                window(arm, batch, 0.0)
        per = {a.name: [] for a in arms}
        for _ in range(args.rounds):
            for arm in arms:
                per[arm.name].append(window(arm, batch, args.window))
        row = dict(batch=b, workspace_bytes=int(_capi.lib().aft_train_workspace_bytes(arms[0].model._handle, b)))
        for arm in arms:
            w = min(per[arm.name], key=lambda r: r["ms_per_step"])
            w["samples_per_s"] = b / (w["ms_per_step"] / 1e3)
            w["tflops"] = res["step_flops_per_sample"] * b / (w["ms_per_step"] / 1e3) / 1e12
            w["windows_ms_per_step"] = [r["ms_per_step"] for r in per[arm.name]]
            row["ours" if arm is arms[0] else "torch"] = w
        row["speedup"] = row["ours"]["samples_per_s"] / row["torch"]["samples_per_s"]
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
        del batch
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("written", args.out)


if __name__ == "__main__":
    main()
