#!/usr/bin/env python
"""bench.py -- channel estimates / second of the AdaFortiTran / FortiTran inference forward on B200.

    python bench.py --gpus N --steps K --warmup W                      # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K --warmup W     # the UNMODIFIED reference on the host CPU

Workloads (BASELINE.json `configs`):
  --workload ada   (default) configs[2]: AdaFortiTran default config, bf16, GLOBAL batch 65536 sharded over the N
                   GPUs (strong scaling: B/N samples per rank), SNR / delay-spread / Doppler metadata.
  --workload forti configs[1]: FortiTran default config, bf16, batch 16384 PER GPU (weak scaling); also measured
                   briefly inside the default run and reported under `extra_configs`.

One "step" = one evaluation step of the batch-sharded path (adafortitran_b200.distributed.ShardedEvaluator.step,
the multi-GPU form of the reference's ModelEvaluator loop body, src/main/trainer.py:328-347): forward of the local
shard with the all-gather of the estimates FUSED into the kernel that writes them (stores into every rank's gather
buffer over NVLink), on-device error sums, NCCL all-reduce of the sums.  `value` times it with the inputs resident in
HBM (CUDA events on the launch stream, one pair per step, L2 flushed between steps, max over ranks); `e2e` runs the same
step from pinned HOST inputs to pinned host estimates (H2D / D2H inside the timed region).  Prints ONE JSON line (rank 0).

--dump-outputs DIR (our arm): after the timed steps, rank 0 writes what the last timed step returned, so that two builds
can be compared output for output on identical seeded inputs:
  estimates.npy      float32 [n, 120, 14, 2]  all-gathered estimates (re, im) of n rows: all of them, or a fixed seeded
                                              sample of DUMP_ROWS rows when the global batch is larger (64 MB at most)
  estimate_rows.npy  float64 [n]              the global row index of each dumped estimate
  error_sums.npy     float64 [2]              the reduced [sum |est - truth|^2, sum |truth|^2]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_EST = {"forti": 1_428_241_920, "ada": 1_429_387_932}   # algorithmic FLOPs / complex estimate (SURVEY.md 8d)
F_ENC_EST = 1_362_493_440                                 # of which encoder GEMM + attention (the encoder kernel)
BYTES_IN = {"forti": 192, "ada": 204}
BYTES_OUT = 13_440
SYS = dict(ofdm=dict(num_scs=120, num_symbols=14), pilot=dict(num_scs=12, num_symbols=2))
FORTI = dict(model_type="fortitran", patch_size=(3, 2), num_layers=6, model_dim=128, num_head=4, activation="gelu",
             dropout=0.1, max_seq_len=512, pos_encoding_type="learnable")
ADA = dict(FORTI, model_type="adafortitran", channel_adaptivity_hidden_sizes=[7, 42, 560], adaptive_token_length=6)
ENCODER_SOURCES = ("tc_encoder.cu", "tc_ptx.cuh", "tc_layout.cuh", "tc_encoder.cuh", "tc_math.cuh")
DUMP_ROWS = 4096                                          # 4096 x 120 x 14 x 2 float32 = 55 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
    ap.add_argument("--workload", choices=("ada", "forti"), default="ada")
    ap.add_argument("--global-batch", type=int, default=65536, help="ada: global batch, sharded over the GPUs")
    ap.add_argument("--batch-per-gpu", type=int, default=16384, help="forti: batch per GPU")
    ap.add_argument("--precision", choices=("bf16", "fp32"), default="bf16")
    ap.add_argument("--gather", choices=("peer", "nccl"), default="peer", help="all-gather of the estimates: fused peer stores / NCCL")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--cpu-batch", type=int, default=64, help="reference arm: estimates per step (BASELINE configs[0])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs / collectives comparison legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/*.npy (our arm)")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), hbm=p["hbm_gbs"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def encoder_source_sha():
    """Identity of the encoder kernel's sources: ncu captures under profiles/ are stamped with it."""
    h = hashlib.sha256()
    for name in ENCODER_SOURCES:
        with open(os.path.join(ROOT, "adafortitran_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic():
    """dram bytes per encoder launch from the committed ncu capture -- only if it was taken on the current sources."""
    path = os.path.join(ROOT, "profiles", "encoder_traffic.json")
    if not os.path.exists(path):
        return None, "no ncu capture committed"
    with open(path) as f:
        t = json.load(f)
    if t.get("encoder_src_sha") != encoder_source_sha():
        return None, f"stale ncu capture (taken at sources {t.get('encoder_src_sha')}, now {encoder_source_sha()})"
    return t.get("dram_bytes_per_launch"), f"ncu --set full, {t.get('captured', 'n/a')}"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(self.rows)}


def workload_config(args, world):
    ada = args.workload == "ada"
    name = "AdaFortiTran" if ada else "FortiTran"
    per = args.global_batch // world if ada else args.batch_per_gpu
    gb = per * world
    cfg = {"workload": f"{name} default config (120x14 grid, 12x2 pilots, patch 3x2, 6 layers, d=128, 4 heads), "
                       f"{args.precision} inference, " + (f"global batch {gb} sharded over {world} GPU(s) (BASELINE configs[2])" if ada
                                                          else f"batch {per} per GPU (BASELINE configs[1])") +
                       ", random-init weights (seed 0), synthetic CN(0,1) pilots" + (" + SNR/DS/Doppler metadata" if ada else ""),
           "batch_per_gpu": per, "global_batch": gb,
           "parallelism": f"dp{world}: one replica per GPU, batch-sharded; estimates all-gathered by fused peer stores over "
                          f"NVLink inside the forward ({args.gather}), error sums all-reduced (NCCL)" if world > 1 else
                          "dp1: one replica",
           "l2": "L2 flushed between timed steps (256 MiB device write); per-step intermediate stream (GBs) exceeds the 126 MB L2"}
    return cfg, per, gb


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference (baseline/_ref, installed by baseline/install_ref.py) on the host cores
# ------------------------------------------------------------------------------------------------------------------
def load_reference_model(kind):
    """Returns (callable(pilots, meta) -> estimates, kind_string).  Uses the reference's own package, config loader and
    YAML files; falls back to the oracle port only if baseline/_ref is absent."""
    import torch
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "src", "models")):
        # the reference is a script tree that expects its root on sys.path; this repository's own `src` shim must not win
        sys.path[:] = [ref] + [p for p in sys.path if os.path.abspath(p or ".") != ROOT]
        for m in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[m]
        from src.config import load_config                         # reference src/config/config_loader.py:75
        from src.models import AdaFortiTranEstimator, FortiTranEstimator   # reference src/models/__init__.py:1-3
        import src.models as ref_models
        assert os.path.abspath(ref_models.__file__).startswith(ref), ref_models.__file__
        system_config, model_config = load_config(os.path.join(ref, "config", "system_config.yaml"),
                                                  os.path.join(ref, "config", "adafortitran.yaml" if kind == "ada" else "fortitran.yaml"))
        torch.manual_seed(0)
        model = (AdaFortiTranEstimator if kind == "ada" else FortiTranEstimator)(system_config, model_config).eval()   # device='cpu'
        return model, "reference"
    from oracle.torch_port import TorchPort
    from adafortitran_b200 import AdaFortiTranEstimator, FortiTranEstimator, ModelConfig, SystemConfig
    torch.manual_seed(0)
    cls, cfg = (AdaFortiTranEstimator, ADA) if kind == "ada" else (FortiTranEstimator, FORTI)
    sd = {k: v.numpy() for k, v in cls(SystemConfig(**SYS), ModelConfig(**cfg)).state_dict().items()}
    port = TorchPort(sd, adaptive=(kind == "ada"))
    return (lambda p, meta: port(p, *(meta[1:4] if meta is not None else ()))), "port"


def cpu_reference_rate(kind, seconds, warmup=1, steps=None, batch=64):
    """Reference forward on the host cores: `steps` timed forwards of `batch` estimates (or as many as fit in `seconds`)."""
    import torch
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    model, how = load_reference_model(kind)
    g = torch.Generator().manual_seed(1)
    pilots = torch.view_as_complex(torch.randn(batch, 12, 2, 2, generator=g) * (0.5 ** 0.5))
    pick = lambda grid: torch.tensor(grid, dtype=torch.float32)[torch.randint(0, 7, (batch,), generator=g)].reshape(batch, 1)
    meta = None
    if kind == "ada":
        meta = (torch.zeros(batch, 1), pick(list(range(0, 31, 5))), pick(list(range(50, 351, 50))), pick(list(range(200, 1401, 200))),
                torch.zeros(batch, 1), [("syn",) * batch])
    call = (lambda: model(pilots, meta)) if kind == "ada" else (lambda: model(pilots) if how == "reference" else model(pilots, None))
    with torch.no_grad():
        for _ in range(max(1, warmup)):
            out = call()
        assert tuple(out.shape) == (batch, 120, 14) and out.is_complex()
        times = []
        t_end = time.perf_counter() + seconds
        while (steps and len(times) < steps) or (not steps and (len(times) < 3 or time.perf_counter() < t_end) and len(times) < 400):
            t0 = time.perf_counter()
            call()
            times.append(time.perf_counter() - t0)
    total = sum(times)
    src = "unmodified reference (baseline/_ref: src.models via its own load_config, device='cpu')" if how == "reference" \
        else "oracle/torch_port.py (baseline/_ref absent)"
    return {"value": batch * len(times) / total, "unit": "estimates/s", "cores": cores, "kind": how,
            "sample": f"{len(times)} forward passes of batch {batch} ({kind} default config, fp32, {src}, torch {torch.__version__} "
                      f"CPU, {torch.get_num_threads()} threads on {cores} cores), {total:.1f} s",
            "ms_per_step": 1e3 * total / len(times), "steps": len(times)}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    world = args.gpus
    r = cpu_reference_rate(args.workload, args.cpu_seconds, warmup=max(1, args.warmup), steps=args.steps, batch=args.cpu_batch)
    cfg, per, gb = workload_config(args, world)
    cfg["note"] = (f"reference arm: the reference's own CPU forward (its only supported device path); each step is a bounded sample of "
                   f"{args.cpu_batch} estimates of the same workload on the host cores")
    line = {
        "impl": "reference", "metric": "channel_estimates_per_sec", "value": r["value"], "unit": "estimates/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": max(1, args.warmup), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong" if args.workload == "ada" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "estimates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args):
    """The cpu_baseline leg of our arm: the reference arm in a fresh interpreter (the reference's `src` package and this
    repository's `src` shim cannot live in one process)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--steps", "0",
           "--warmup", "1", "--cpu-seconds", str(args.cpu_seconds), "--cpu-batch", str(args.cpu_batch)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        return json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as e:   # noqa: BLE001 -- reported, never fatal for the GPU line
        return {"value": None, "unit": "estimates/s", "cores": len(os.sched_getaffinity(0)), "kind": "unavailable", "sample": f"failed: {e}"}


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def make_inputs(kind, B, seed, dev):
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    pilots_h = torch.view_as_complex(torch.randn(B, 12, 2, 2, generator=g) * (0.5 ** 0.5)).contiguous().pin_memory()
    meta_h = None
    if kind == "ada":
        pick = lambda grid: torch.tensor(grid, dtype=torch.float32)[torch.randint(0, 7, (B,), generator=g)].reshape(B, 1).pin_memory()
        meta_h = (torch.zeros(B, 1), pick(list(range(0, 31, 5))), pick(list(range(50, 351, 50))), pick(list(range(200, 1401, 200))),
                  torch.zeros(B, 1), None)
    pilots_d = pilots_h.to(dev)
    meta_d = None if meta_h is None else tuple(t.to(dev) if torch.is_tensor(t) else t for t in meta_h)
    return pilots_h, meta_h, pilots_d, meta_d


def timed_steps(ev, pilots, meta, truth, steps, flush, barrier, world, dev):
    """K steps, one CUDA-event pair per step on the launch stream, L2 flushed (untimed) in between; max over ranks."""
    import torch
    import torch.distributed as dist
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    barrier()
    wall0 = time.perf_counter()
    for i in range(steps):
        flush.zero_()
        starts[i].record()
        gathered, sums = ev.step(pilots, meta, truth)
        stops[i].record()
    barrier()
    wall = time.perf_counter() - wall0
    total_ms = torch.tensor([sum(s.elapsed_time(e) for s, e in zip(starts, stops))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    return float(total_ms.item()), wall, gathered, sums


def dump_outputs(out_dir, gathered, sums):
    """Writes the step's outputs as described in the module docstring (--dump-outputs)."""
    import numpy as np
    import torch
    n = gathered.shape[0]
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    est = torch.view_as_real(gathered[torch.from_numpy(rows).to(gathered.device)]).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "estimates.npy"), est.astype(np.float32, copy=False))
    np.save(os.path.join(out_dir, "estimate_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "error_sums.npy"), sums.cpu().numpy().astype(np.float64, copy=False))


def run_ours(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from adafortitran_b200 import AdaFortiTranEstimator, FortiTranEstimator, ModelConfig, SystemConfig, _capi
    from adafortitran_b200 import distributed as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if args.steps < 1:
        raise SystemExit(f"--steps {args.steps}: at least one timed step is needed")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    kind = args.workload
    cfg, B, GB = workload_config(args, world)
    if kind == "ada" and args.global_batch % world:
        raise SystemExit(f"--global-batch {args.global_batch} must be divisible by the {world} GPUs")
    lib = _capi.lib()

    def build(k):
        torch.manual_seed(0)   # identical random-init weights on every replica
        cls, mc = (AdaFortiTranEstimator, ADA) if k == "ada" else (FortiTranEstimator, FORTI)
        m = cls(SystemConfig(**SYS), ModelConfig(**dict(mc, device=f"cuda:{local}"))).eval()
        m.precision = args.precision
        return m

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model = build(kind)
    pilots_h, meta_h, pilots_d, meta_d = make_inputs(kind, B, 1234 + rank, dev)
    tg = torch.Generator(device=dev).manual_seed(99 + rank)
    truth = torch.view_as_complex(torch.randn(B, 120, 14, 2, generator=tg, device=dev) * (0.5 ** 0.5))   # synthetic unit-power truth
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    mode = args.gather
    try:
        ev = D.ShardedEvaluator(model, B, mode=mode)
    except Exception as e:   # noqa: BLE001 -- peer memory cannot be mapped here: say so and use NCCL
        if mode != "peer":
            raise
        mode = f"nccl (peer mapping failed: {str(e)[:120]})"
        ev = D.ShardedEvaluator(model, B, mode="nccl")

    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            ev.step(pilots_d, meta_d, truth)
        barrier()
        lib.aft_profile_enable(model._handle, 1)
        launches0 = lib.aft_launch_count()
        sampler = ClockSampler(local)
        sampler.start()
        total_ms, wall, gathered, sums = timed_steps(ev, pilots_d, meta_d, truth, args.steps, flush, barrier, world, dev)
        clocks = sampler.summary()
        launches = lib.aft_launch_count() - launches0
        ms = (C.c_double * 3)()
        nl = (C.c_int64 * 3)()
        _capi.check(lib.aft_profile_read(model._handle, ms, nl))
        lib.aft_profile_enable(model._handle, 0)
        value = GB * args.steps / (total_ms / 1e3)
        sums_host = sums.cpu()
        nmse_db = float(10.0 * torch.log10(sums_host[0] / sums_host[1]))
        if args.dump_outputs:                   # before the e2e steps below overwrite the gather buffer and the sums
            if rank == 0:
                dump_outputs(args.dump_outputs, gathered, sums)
            barrier()                           # no rank's e2e step stores into rank 0's gather buffer while it is read
        reference_out = gathered[rank * B:(rank + 1) * B].clone() if gathered is not None else None

        # ---- end to end: pinned host inputs -> (H2D, forward + fused gather, error sums, all-reduce) -> pinned host estimates
        out_h = torch.empty((B, 120, 14), dtype=torch.complex64).pin_memory()
        ev.step(pilots_h, meta_h, truth, host_out=out_h)
        sums.cpu()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, s = ev.step(pilots_h, meta_h, truth, host_out=out_h)
            s_host = s.cpu()          # the step's result (metric) read back: also drains the stream
        torch.cuda.synchronize()
        e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = GB * args.e2e_steps / float(e2e_s.item()) if args.e2e_steps else None
        same = bool(torch.equal(out_h.to(dev), reference_out)) if (reference_out is not None and args.e2e_steps) else None

        # ---- the collectives of the path: fused peer stores vs the serial NCCL all-gather, same step otherwise
        coll = None
        extra = {}
        if world > 1 and not args.no_extra:
            coll = {"mode": mode, "all_gather_bytes_per_rank": B * BYTES_OUT, "step_ms": total_ms / args.steps}
            ev2 = D.ShardedEvaluator(model, B, mode="nccl" if mode == "peer" else "peer") if mode in ("peer", "nccl") else None
            if ev2 is not None:
                for _ in range(2):
                    ev2.step(pilots_d, meta_d, truth)
                t_ms, _, g2, _ = timed_steps(ev2, pilots_d, meta_d, truth, 3, flush, barrier, world, dev)
                coll["step_ms_other_mode"] = {"mode": ev2.mode, "ms": t_ms / 3}
                coll["gathered_equal_across_modes"] = bool(torch.equal(g2, gathered))
                ev2.close()
            # the NCCL all-gather + all-reduce alone (what the fused path removes from the critical path)
            loc = gathered[rank * B:(rank + 1) * B].clone()
            D.gather_estimates(loc)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            D.gather_estimates(loc)
            D.reduce_error_sums(sums.clone())
            e1.record()
            torch.cuda.synchronize()
            coll["nccl_all_gather_plus_all_reduce_ms"] = e0.elapsed_time(e1)
        ev.close()
        del gathered, reference_out
        torch.cuda.empty_cache()

        # ---- extra config: the other BASELINE workload, briefly (weak-scaling FortiTran configs[1] / sharded Ada configs[2])
        if not args.no_extra:
            other = "forti" if kind == "ada" else "ada"
            B2 = args.batch_per_gpu if other == "forti" else args.global_batch // world
            m2 = build(other)
            _, _, p2, md2 = make_inputs(other, B2, 4321 + rank, dev)
            ev3 = D.ShardedEvaluator(m2, B2, mode="peer" if mode == "peer" else "nccl")
            t2 = torch.zeros((B2, 120, 14), dtype=torch.complex64, device=dev)
            for _ in range(3):
                ev3.step(p2, md2, t2)
            t_ms, _, _, _ = timed_steps(ev3, p2, md2, t2, 3, flush, barrier, world, dev)
            ev3.close()
            name = "forti_b16384_per_gpu_weak (BASELINE configs[1])" if other == "forti" else "ada_global_b65536_strong (BASELINE configs[2])"
            extra[name] = {"value": B2 * world * 3 / (t_ms / 1e3), "unit": "estimates/s", "ms_per_step": t_ms / 3, "batch_per_gpu": B2,
                           "steps": 3}

    pk = peaks()
    enc_ms = ms[1]
    n_est = B * args.steps
    roof = None
    if enc_ms > 0 and args.precision == "bf16":
        ach = n_est * F_ENC_EST / (enc_ms / 1e3) / 1e12
        traffic, traffic_note = measured_traffic()
        roof = {"bound": "tensor", "kernel": "encoder3_kernel" if os.environ.get("AFT_ENCODER", "")[:1] == "3" else "encoder_kernel", "achieved": ach, "peak": pk["sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["sustained"], "frac_of_burst_peak": ach / pk["burst"], "traffic": traffic, "traffic_source": traffic_note,
                "peak_source": pk["source"] + ", sustained figure (kernel timed inside a long step)",
                "launches": int(nl[1]), "avg_launch_ms": enc_ms / max(1, int(nl[1])),
                "algorithmic_flops_per_launch": n_est * F_ENC_EST / max(1, int(nl[1])), "encoder_src_sha": encoder_source_sha()}
    line = {
        "metric": "channel_estimates_per_sec", "value": value, "unit": "estimates/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if kind == "ada" else "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": cfg, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "estimates/s", "h2d_bytes_per_step": B * BYTES_IN[kind],
                "d2h_bytes_per_step": B * BYTES_OUT + 16, "steps": args.e2e_steps, "matches_device_path": same,
                "what": "ShardedEvaluator.step from pinned host pilots/meta to pinned host estimates of the local shard + the "
                        "reduced error sums; per-rank bytes; includes the fused all-gather and the all-reduce"},
        "gpu_launches": int(launches),
        "roofline": roof,
        "step_tensor_frac": value / world * F_EST[kind] / 1e12 / pk["sustained"],
        "stages_ms_per_step": {"frontend": ms[0] / args.steps, "encoder": ms[1] / args.steps, "head": ms[2] / args.steps},
        "wall_s_timed_region": wall, "nmse_db_vs_synthetic_truth": nmse_db, "collectives": coll, "extra_configs": extra,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_subprocess(args)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        if a.dump_outputs:
            raise SystemExit("--dump-outputs applies to --impl ours")
        run_reference(a)
    else:
        run_ours(a)
