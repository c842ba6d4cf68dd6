"""Data-parallel training-step benchmark: full Adam steps of AdaFortiTran (default config, dropout 0.1, the reference's
MSE over concatenated real / imaginary parts) through ``distributed.ShardedTrainer`` on the GPUs of one node.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29514 \\
      tools/train_mgpu.py [--out profiles/r04_train_mgpu.json]

One launch measures one world size N, at two global batches:
  weak   : 256 samples per GPU (global batch 256 N)
  strong : global batch 2048 (2048 / N per GPU)
Timing is the window method of tools/train_bench.py: warm-up steps, then windows of at least --window seconds (the step
count of a window is fixed by rank 0 from the warm-up and broadcast, so every rank runs the same collectives), CUDA
events around each window on every rank, the slowest rank's time, the best of --rounds windows.  Rank 0 merges one row
per (N, kind) into --out, so launches at N = 1, 2, 4, 8 fill one file; efficiency = throughput / (N x the N = 1
throughput of the same kind; for strong scaling the N = 1 run of batch 2048).
"""
import argparse
import json
import math
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from adafortitran_b200 import distributed as D  # noqa: E402
from tests import util  # noqa: E402
from tools.train_bench import card, make_batch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-gpu", type=int, default=256)
    ap.add_argument("--strong", type=int, default=2048)
    ap.add_argument("--window", type=float, default=3.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_train_mgpu.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_mgpu: no CUDA device (this measurement runs on the GPU only)")
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)
    model = util.make_model("ada", device=f"cuda:{local}")
    model.trainable = True
    model.train()
    trainer = D.ShardedTrainer(model)
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    nparams = sum(p.numel() for p in trainer.params)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def slowest(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rows = []
    for kind, global_batch in (("weak", args.per_gpu * world), ("strong", args.strong)):
        lo, hi = D.shard_range(global_batch, rank, world)
        pilots, cond, truth = make_batch(global_batch, seed=global_batch)     # the same global batch on every rank
        z = torch.zeros(hi - lo, device=dev)
        shard = (pilots[lo:hi], (z, cond[0][lo:hi], cond[1][lo:hi], cond[2][lo:hi], z, None), truth[lo:hi])

        def step():
            trainer.step(*shard, global_batch)
            opt.step()

        for _ in range(3):
            step()
        sync()
        t0 = time.perf_counter()
        for _ in range(3):
            step()
        sync()
        per = slowest((time.perf_counter() - t0) / 3)
        steps = max(3, math.ceil(args.window / per))
        windows = []
        for _ in range(args.rounds):
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            e1.synchronize()
            windows.append(slowest(e0.elapsed_time(e1)) / steps)
        ms = min(windows)
        row = dict(kind=kind, n_gpus=world, global_batch=global_batch, per_gpu=hi - lo if rank == 0 else None,
                   steps_per_window=steps, ms_per_step=ms, windows_ms_per_step=windows,
                   samples_per_s=global_batch / (ms / 1e3), allreduce_floats=nparams + 1,
                   allreduce_bytes=4 * (nparams + 1))
        rows.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
        del shard, pilots, cond, truth
        torch.cuda.empty_cache()

    if rank == 0:
        res = json.load(open(args.out)) if os.path.exists(args.out) else {}
        res.update(card=card(), torch=torch.__version__, nccl=".".join(map(str, torch.cuda.nccl.version())),
                   config="AdaFortiTran default, dropout 0.1, Adam 5e-4, MSE(re|im), ShardedTrainer (one NCCL SUM "
                          "all-reduce of all gradients per step)")
        res.setdefault("rows", [])
        res["rows"] = [r for r in res["rows"] if r["n_gpus"] != world] + rows
        res["rows"].sort(key=lambda r: (r["kind"], r["n_gpus"]))
        base = {r["kind"]: r["samples_per_s"] for r in res["rows"] if r["n_gpus"] == 1}
        for r in res["rows"]:
            if r["kind"] in base:
                r["efficiency"] = r["samples_per_s"] / (r["n_gpus"] * base[r["kind"]])
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        print("written", args.out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
