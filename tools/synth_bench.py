"""Synthetic-channel generation on the GPU (``aft_synthetic_channels``, ``data.SyntheticChannels``).

Measures, in one run on one card:
  * the generation rate (samples/s) and bytes written per second at batch 65536 on the reference grid (120 x 14,
    pilots 12 x 2; 890 MB written per call, past the 126 MB L2) and at batch 256 on the config-5 grid (3276 x 14, pilots
    1638 x 2; 94 MB per call), conditions drawn per sample;
  * the write-only HBM bandwidth in the same run, as tools/write_bw.py measures it (fill of a 2 GiB buffer);
  * a per-condition sweep step at batch 65536 -- generate with a fixed condition, bf16 AdaFortiTran forward,
    aft_error_sums -- against the forward alone;
  * the card's name, power limit and maximum SM clock.

  python tools/synth_bench.py --out profiles/r06_synthetic.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from adafortitran_b200 import _capi  # noqa: E402
from adafortitran_b200.data import SyntheticChannels  # noqa: E402
from tests import util  # noqa: E402


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


def write_bw_gbs(min_s):
    y = torch.empty(1 << 29, device="cuda")
    ms = timed_ms(lambda: y.fill_(1.0), min_s)
    del y
    return 4 * (1 << 29) / ms / 1e6


def generation_row(geom, batch, min_s):
    scs, sym, ps, pt = geom
    sysc = dict(ofdm=dict(num_scs=scs, num_symbols=sym), pilot=dict(num_scs=ps, num_symbols=pt))
    gen = SyntheticChannels(sysc, 12345)
    cfg = gen._cfg
    pilots = torch.empty((batch, ps, pt), dtype=torch.complex64, device="cuda")
    truth = torch.empty((batch, scs, sym), dtype=torch.complex64, device="cuda")
    cond = torch.empty((3, batch), dtype=torch.float32, device="cuda")
    lib = _capi.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    state = {"s0": 0}

    def call():       # the kernel alone: the C-ABI on preallocated buffers, a new range of samples every call
        _capi.check(lib.aft_synthetic_channels(C.byref(cfg), 12345, state["s0"], batch, C.c_void_p(cond[0].data_ptr()),
                                               C.c_void_p(cond[1].data_ptr()), C.c_void_p(cond[2].data_ptr()), 1,
                                               C.c_void_p(pilots.data_ptr()), C.c_void_p(truth.data_ptr()), st))
        state["s0"] += batch

    ms = timed_ms(call, min_s)
    nbytes = batch * (8 * (scs * sym + ps * pt) + 12)
    return {"grid": f"{scs}x{sym}", "pilots": f"{ps}x{pt}", "batch": batch, "bytes_per_call": nbytes, "ms": ms,
            "samples_per_s": batch / ms * 1e3, "gbs_written": nbytes / ms / 1e6}


def sweep_rows(batch, min_s):
    sysc = dict(ofdm=dict(num_scs=120, num_symbols=14), pilot=dict(num_scs=12, num_symbols=2))
    gen = SyntheticChannels(sysc, 777, conditions=(15.0, 200.0, 800.0))
    model = util.make_model("ada", precision="bf16", weights=util.ada_weights())
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    lib = _capi.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pilots, meta, truth = gen.batch(0, batch)
    state = {"s0": 0}

    def step():
        p, m, t = gen.batch(state["s0"], batch)
        state["s0"] += batch
        est = model(p, m)
        _capi.check(lib.aft_error_sums(C.c_void_p(est.data_ptr()), C.c_void_p(t.data_ptr()), t.numel(),
                                       C.c_void_p(sums.data_ptr()), st))

    def forward():
        model(pilots, meta)

    def generate():
        gen.batch(state["s0"], batch)
        state["s0"] += batch

    with torch.no_grad():
        fwd = timed_ms(forward, min_s)
        full = timed_ms(step, min_s)
        g = timed_ms(generate, min_s)
        fwd2 = timed_ms(forward, min_s)
    return {"batch": batch, "condition": [15.0, 200.0, 800.0], "forward_ms": [fwd, fwd2], "step_ms": full,
            "generate_ms": g, "generate_share_of_step": g / full,
            "step_over_forward": full / (0.5 * (fwd + fwd2))}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_synthetic.json"))
    ap.add_argument("--min-s", type=float, default=2.0, help="seconds of work per timed window")
    a = ap.parse_args(argv)
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"card": card(), "write_bw_gbs": write_bw_gbs(a.min_s)}
    res["generation"] = [generation_row((120, 14, 12, 2), 65536, a.min_s), generation_row((3276, 14, 1638, 2), 256, a.min_s)]
    res["write_bw_gbs_after"] = write_bw_gbs(a.min_s)
    bw = 0.5 * (res["write_bw_gbs"] + res["write_bw_gbs_after"])
    for r in res["generation"]:
        r["share_of_write_bw"] = r["gbs_written"] / bw
    res["sweep"] = sweep_rows(65536, a.min_s)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
