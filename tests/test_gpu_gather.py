"""GPU: the fused all-gather evaluation step (``aft_forward_gather``, ``aft_forward_host_gather``, ``PeerGather``,
``ShardedEvaluator``), the step ``bench.py`` times, against the plain forward and the fp64 oracle.

Local sample ``i`` of a call lands at row ``rank * rows_per_rank + row0 + i`` of every gather buffer.  The paths:

* fused (AFT_BF16 on the reference grid): the head stores each sample with one bulk copy per destination, up to nine
  (the caller's ``out`` and eight gather buffers), internal chunks of 8192 samples;
* staged (AFT_FP32, and both precisions on other grids): the forward writes ``out``, ``scatter_rows_kernel`` copies it to
  the gather buffers; internal chunks of 1024 (fp32), 1024 (S65) and 683 (S1025 bf16) samples;
* host entry: host chunks of up to 2048 samples on two lanes, tapered towards the end on the reference grid, each chunk a
  forward with ``row0`` advanced by the chunk's first sample.

A. One process, straight through the C-ABI: the library does not care whether a gather buffer is peer memory, so the
   plans point at ``world`` local buffers filled with a NaN pattern no kernel writes.  The rows a call owns equal the
   plain forward bit for bit in every buffer (and in ``out`` / the host ``out``), every other row keeps the pattern, and
   the first row, the rows either side of every chunk boundary and the last row pass the fp64 oracle.  S65 (grid 65 x 1,
   odd ``pix``) at odd row offsets needs the 8-byte path of the scatter kernel.  Bad plans are refused with
   AFT_ERR_INVALID before anything is launched.
B. ``ShardedEvaluator(model, B, "peer")`` without ``torch.distributed``: a ``PeerGather`` with one rank, at the bench's
   workload (Ada bf16, B = 65536) and at B = 5000 (host chunks tapered) in both precisions.
C. Several processes: two gloo ranks sharing one GPU (CUDA IPC between processes on one device) and, with two or more
   GPUs, one NCCL rank per GPU.  Unequal ``shard_range`` shards of a ``2 world + 1`` batch.

The error sums are formed per element in fp32 and added in fp64, so each non-negative term is off by at most
4 * 2^-24 and the sums are gated at 3e-7 relative against fp64 sums of the same fp32 tensors.
"""
import ctypes as C
import datetime
import os
import socket
import time
import traceback

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from adafortitran_b200 import _capi
from adafortitran_b200 import distributed as D
from oracle import aft_oracle as O
from tests import util
from tests.test_gpu_generic_edges import GEOMS

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FBADBAD          # a NaN bit pattern no kernel produces
SUMS_RTOL = 3e-7
# fp64-oracle gates of the suite: reference grid over the checked rows, generic grids per sample
FP32_REF_GATE, FP32_GENERIC_GATE = 1e-4, 1e-5
BF16_REF_DB = {"forti": -45.0, "ada": -38.0}
BF16_GENERIC_DB = {"forti": -40.0, "ada": -34.0}
CODES = {"fp32": _capi.AFT_FP32, "bf16": _capi.AFT_BF16}


@pytest.fixture(scope="module", autouse=True)
def report():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    print(f"\n{__name__}: wall time {time.perf_counter() - t0:.1f} s, peak torch allocation "
          f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB ({torch.cuda.get_device_name()})")


class Net:
    """A model with its fp64 oracle: "ada" / "forti" on the reference grid, or a geometry of ``GEOMS``."""

    def __init__(self, name, device="cuda"):
        self.name, self.generic = name, name in GEOMS
        if self.generic:
            from adafortitran_b200 import AdaFortiTranEstimator, FortiTranEstimator, ModelConfig, SystemConfig
            kind, layers, act, pos, grid, pilots, patch = GEOMS[name]
            S = (grid[0] // patch[0]) * (grid[1] // patch[1])
            ada = kind == "ada"
            extra = dict(channel_adaptivity_hidden_sizes=[7, 42, 2 * S], adaptive_token_length=6) if ada else {}
            torch.manual_seed(list(GEOMS).index(name))
            cls = AdaFortiTranEstimator if ada else FortiTranEstimator
            self.model = cls(SystemConfig(ofdm=dict(num_scs=grid[0], num_symbols=grid[1]),
                                          pilot=dict(num_scs=pilots[0], num_symbols=pilots[1])),
                             ModelConfig(model_type="adafortitran" if ada else "fortitran", patch_size=patch,
                                         num_layers=layers, model_dim=128, num_head=4, activation=act,
                                         max_seq_len=max(S, 8), pos_encoding_type=pos, device=device, **extra)).eval()
            self.sd = {k: v.detach().cpu().numpy() for k, v in self.model.state_dict().items()}
            self.cfg = O.OracleConfig(num_scs=grid[0], num_symbols=grid[1], pilot_scs=pilots[0],
                                      pilot_symbols=pilots[1], patch=patch, num_layers=layers, activation=act,
                                      adaptive=ada)
            self.kind, self.grid, self.pilots = kind, grid, pilots
        else:
            sd = util.ada_weights()
            self.kind = name
            self.sd = sd if name == "ada" else util.forti_weights(sd)
            self.model = util.make_model(name, device=device, weights=self.sd)
            self.cfg = util.oracle_cfg(name)
            self.grid, self.pilots = (120, 14), (12, 2)
        self.ada = self.kind == "ada"

    def inputs(self, n, seed):
        rng = np.random.default_rng(seed)
        shape = (n, *self.pilots)
        x = ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)).astype(np.complex64)
        if not self.ada:
            return x, None
        cond = (rng.choice(O.SNR_GRID, n), rng.choice(O.DS_GRID[:4], n), rng.choice(O.DOP_GRID[:3], n))
        return x, tuple(a.astype(np.float32) for a in cond)

    def plain(self, prec, x, cond):
        """model(x) on the device: the reference the gathered rows must equal bit for bit."""
        self.model.precision = prec
        with torch.no_grad():
            return self.model(torch.from_numpy(x), util.meta(*cond) if cond is not None else None)

    def oracle_gate(self, prec, y, x, cond, idx, what):
        """Rows ``idx`` of the estimates ``y`` (numpy, the call's samples) against the fp64 oracle."""
        ref = O.forward(self.cfg, self.sd, x[idx], *((a[idx] for a in cond) if cond is not None else ()))
        got = y[idx]
        if self.generic:
            errs = [O.normwise_err(got[i], ref[i]) if prec == "fp32" else O.rel_err_db(got[i], ref[i])
                    for i in range(len(idx))]
            gate = FP32_GENERIC_GATE if prec == "fp32" else BF16_GENERIC_DB[self.kind]
        else:
            errs = [O.normwise_err(got, ref) if prec == "fp32" else O.rel_err_db(got, ref)]
            gate = FP32_REF_GATE if prec == "fp32" else BF16_REF_DB[self.kind]
        assert max(errs) <= gate, (what, idx, errs)


_NETS = {}


def net(name):
    if name not in _NETS:
        _NETS[name] = Net(name)
    return _NETS[name]


@pytest.fixture(scope="module", autouse=True)
def _release_nets():
    yield
    for n in _NETS.values():
        n.model._release()
    _NETS.clear()


def _ints(t):
    return torch.view_as_real(t).view(torch.int32)


def _buffers(world, rpr, grid):
    bufs = [torch.empty((world * rpr, *grid), dtype=torch.complex64, device="cuda") for _ in range(world)]
    for b in bufs:
        _ints(b).fill_(SENTINEL)
    return bufs


def _plan(ptrs, world, rank, rpr, row0):
    g = _capi.AftGather()
    for p, v in enumerate(ptrs[:8]):
        g.peer_out[p] = v
    g.world, g.rank, g.rows_per_rank, g.row0 = world, rank, rpr, row0
    return g


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _dev_args(x, cond):
    xd = torch.from_numpy(x).cuda().contiguous()
    cd = [torch.from_numpy(a).cuda().contiguous() for a in cond] if cond is not None else [None] * 3
    return xd, cd


def _call_dev(nt, prec, x, cond, batch, out, plan):
    """aft_forward_gather; returns the status (the refusals are checked by status)."""
    lib, m = _capi.lib(), nt.model
    m._ensure_handle()
    m._sync_weights()
    code = CODES[prec]
    xd, cd = _dev_args(x, cond)
    need = lib.aft_workspace_bytes(m._handle, max(batch, 1), code)
    ws = torch.empty(need + 256, dtype=torch.uint8, device="cuda")
    ptr = C.c_void_p((ws.data_ptr() + 255) // 256 * 256)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.aft_forward_gather(m._handle, _vp(xd), _vp(cd[0]), _vp(cd[1]), _vp(cd[2]), _vp(out), batch, code, ptr,
                                need, st, C.byref(plan))
    torch.cuda.synchronize()
    return rc


def _call_host(nt, prec, x, cond, batch, out, plan):
    """aft_forward_host_gather on host inputs (returns after its work has completed)."""
    lib, m = _capi.lib(), nt.model
    m._ensure_handle()
    m._sync_weights()
    torch.cuda.synchronize()
    xh = torch.from_numpy(x).contiguous()
    ch = [torch.from_numpy(a).contiguous() for a in cond] if cond is not None else [None] * 3
    return lib.aft_forward_host_gather(m._handle, _vp(xh), _vp(ch[0]), _vp(ch[1]), _vp(ch[2]), _vp(out), batch,
                                       CODES[prec], C.byref(plan))


def _check_rows(bufs, lo, ref):
    """Rows [lo, lo + len(ref)) of every buffer equal ``ref`` bitwise, every other row holds the sentinel."""
    r = _ints(ref)
    for p, b in enumerate(bufs):
        v = _ints(b)
        assert torch.equal(v[lo:lo + len(ref)], r), f"gather buffer {p}: rows [{lo}, {lo + len(ref)})"
        assert bool((v[:lo] == SENTINEL).all()), f"gather buffer {p}: rows before {lo} overwritten"
        assert bool((v[lo + len(ref):] == SENTINEL).all()), f"gather buffer {p}: rows after {lo + len(ref)} overwritten"


def _host_chunks(batch, generic, chunk):
    """First samples of the host chunks of aft_forward_host_gather (csrc/aft_api.cu: two lanes, tapered ends)."""
    hc = min(batch, 2048, chunk) if generic else min(batch, 2048)
    starts, c0 = [], 0
    while c0 < batch:
        starts.append(c0)
        rem = batch - c0
        bc = min(rem, hc)
        if not generic and batch > hc and hc // 4 < rem <= hc + hc // 2:
            bc = min(max((rem // 2 + 63) // 64 * 64, hc // 4), rem)
        c0 += bc
    return starts


def _edge_rows(batch, starts):
    """First and last row, and the rows either side of every chunk boundary."""
    return sorted({0, batch - 1} | {s for s in starts if s} | {s - 1 for s in starts if s})


# ---------------------------------------------------------------------------------------------------------------------
# A. straight through the C-ABI
# ---------------------------------------------------------------------------------------------------------------------
# (net, precision, world, rank, rows_per_rank, row0, batch, local out)
DEVICE_CASES = {
    # 150 sequences > 148 CTAs; eight, then nine bulk copies per sample
    "ada-bf16-8dst": ("ada", "bf16", 8, 5, 80, 3, 75, False),
    "ada-bf16-9dst": ("ada", "bf16", 8, 5, 80, 3, 75, True),
    "forti-bf16-chunk8192": ("forti", "bf16", 3, 2, 8200, 2, 8195, False),
    "ada-bf16-one-sample": ("ada", "bf16", 1, 0, 1, 0, 1, False),
    "ada-fp32-chunk1024": ("ada", "fp32", 4, 1, 1030, 1, 1027, True),
    # odd pix: rows at odd offsets are 8-byte aligned only
    "S65-fp32-rank1": ("S65", "fp32", 3, 1, 5, 1, 4, True),
    "S65-fp32-odd-row0": ("S65", "fp32", 3, 0, 5, 1, 4, True),
    "S65-fp32-chunk1024": ("S65", "fp32", 2, 1, 1061, 0, 1024 + 37, True),
    "S65-bf16-rank1": ("S65", "bf16", 3, 1, 5, 1, 4, True),
    "S65-bf16-odd-row0": ("S65", "bf16", 3, 0, 5, 1, 4, True),
    "S65-bf16-chunk1024": ("S65", "bf16", 2, 1, 1061, 0, 1024 + 37, True),
    "S1025-bf16-chunk683": ("S1025", "bf16", 2, 1, 721, 1, 683 + 37, True),
}
CHUNK = {("ada", "bf16"): 8192, ("forti", "bf16"): 8192, ("ada", "fp32"): 1024, ("S65", "fp32"): 1024,
         ("S65", "bf16"): 1024, ("S1025", "bf16"): 683}


@pytest.mark.parametrize("cid", list(DEVICE_CASES))
def test_device_gather_rows(cid):
    name, prec, world, rank, rpr, row0, batch, with_out = DEVICE_CASES[cid]
    nt = net(name)
    x, cond = nt.inputs(batch, seed=len(cid) * 31 + batch)
    ref = nt.plain(prec, x, cond)
    bufs = _buffers(world, rpr, nt.grid)
    out = None
    if with_out:
        out = torch.empty_like(ref)
        _ints(out).fill_(SENTINEL)
    plan = _plan([b.data_ptr() for b in bufs], world, rank, rpr, row0)
    _capi.check(_call_dev(nt, prec, x, cond, batch, out, plan))
    _check_rows(bufs, rank * rpr + row0, ref)
    if out is not None:
        assert torch.equal(_ints(out), _ints(ref)), "local out"
    chunk = CHUNK[(name, prec)]
    nt.oracle_gate(prec, bufs[0][rank * rpr + row0:].cpu().numpy(), x, cond,
                   _edge_rows(batch, range(0, batch, chunk)), cid)


# (net, precision, world, rank, rows_per_rank, row0, batch, host out)
HOST_CASES = {
    "ada-bf16-9dst": ("ada", "bf16", 8, 7, 2060, 3, 2057, True),
    "ada-bf16-tapered-no-out": ("ada", "bf16", 2, 1, 5000, 0, 5000, False),
    "ada-fp32": ("ada", "fp32", 2, 1, 2053, 0, 2053, True),
    "S65-bf16-odd-rows": ("S65", "bf16", 3, 1, 2085, 0, 2 * 1024 + 37, True),
}


@pytest.mark.parametrize("cid", list(HOST_CASES))
def test_host_gather_rows(cid):
    name, prec, world, rank, rpr, row0, batch, with_out = HOST_CASES[cid]
    nt = net(name)
    x, cond = nt.inputs(batch, seed=len(cid) * 17 + batch)
    ref = nt.plain(prec, x, cond)
    bufs = _buffers(world, rpr, nt.grid)
    out = None
    if with_out:
        out = torch.empty(ref.shape, dtype=torch.complex64).pin_memory()
        _ints(out).fill_(SENTINEL)
    plan = _plan([b.data_ptr() for b in bufs], world, rank, rpr, row0)
    _capi.check(_call_host(nt, prec, x, cond, batch, out, plan))
    torch.cuda.synchronize()
    _check_rows(bufs, rank * rpr + row0, ref)
    if out is not None:
        assert torch.equal(_ints(out), _ints(ref.cpu())), "host out"
    starts = _host_chunks(batch, nt.generic, CHUNK.get((name, prec), 8192))
    assert len(starts) >= 3, starts
    nt.oracle_gate(prec, bufs[1][rank * rpr + row0:].cpu().numpy(), x, cond, _edge_rows(batch, starts), cid)


@pytest.mark.parametrize("entry", ["device", "host"])
def test_batch_zero_does_nothing(entry):
    nt = net("ada")
    bufs = _buffers(2, 4, nt.grid)
    x, cond = nt.inputs(1, seed=3)
    plan = _plan([b.data_ptr() for b in bufs], 2, 1, 4, 0)
    nt.model._ensure_handle()
    nt.model._sync_weights()
    before = _capi.lib().aft_launch_count()
    call = _call_dev if entry == "device" else _call_host
    assert call(nt, "bf16", x, cond, 0, None, plan) == _capi.AFT_OK
    assert _capi.lib().aft_launch_count() == before
    torch.cuda.synchronize()
    _check_rows(bufs, 0, bufs[0][:0])


def _bad_plans(bufs):
    """(what, plan, batch): every one refused before anything is launched."""
    ok = [b.data_ptr() for b in bufs]
    return [
        ("row0 + batch > rows_per_rank", _plan(ok, 3, 1, 4, 1), 4),
        ("world 0", _plan(ok, 0, 0, 4, 0), 2),
        ("world 9", _plan(ok, 9, 0, 4, 0), 2),
        ("rank -1", _plan(ok, 3, -1, 4, 0), 2),
        ("rank == world", _plan(ok, 3, 3, 4, 0), 2),
        ("rows_per_rank < 0", _plan(ok, 3, 1, -4, 0), 2),
        ("row0 < 0", _plan(ok, 3, 1, 4, -1), 2),
        ("NULL gather buffer", _plan([ok[0], None, ok[2]], 3, 1, 4, 0), 2),
        ("base 8 bytes off", _plan([ok[0], ok[1] + 8, ok[2]], 3, 1, 4, 0), 2),
    ]


@pytest.mark.parametrize("entry", ["device", "host"])
def test_refusals_launch_nothing(entry):
    nt = net("ada")
    bufs = _buffers(3, 4, nt.grid)
    x, cond = nt.inputs(4, seed=5)
    nt.model._ensure_handle()
    nt.model._sync_weights()
    lib = _capi.lib()
    call = _call_dev if entry == "device" else _call_host
    cases = [(w, "bf16", p, b, None) for w, p, b in _bad_plans(bufs)]
    if entry == "device":      # the host entry always stages through its own device buffer
        cases.append(("non-fused path without out", "fp32", _plan([b.data_ptr() for b in bufs], 3, 1, 4, 0), 2, None))
    for what, prec, plan, batch, out in cases:
        torch.cuda.synchronize()
        before = lib.aft_launch_count()
        assert call(nt, prec, x, cond, batch, out, plan) == _capi.AFT_ERR_INVALID, what
        assert lib.aft_launch_count() == before, what
        assert lib.aft_last_error().decode(), what
        torch.cuda.synchronize()
        _check_rows(bufs, 0, bufs[0][:0])


# ---------------------------------------------------------------------------------------------------------------------
# B. the step bench.py times, one rank
# ---------------------------------------------------------------------------------------------------------------------
def _truth(n, grid, seed):
    rng = np.random.default_rng(seed)
    return ((rng.standard_normal((n, *grid)) + 1j * rng.standard_normal((n, *grid)))).astype(np.complex64)


def _sums64(est, truth):
    """[sum |est - truth|^2, sum |truth|^2] in fp64 from the fp32 tensors, on the device."""
    d = torch.view_as_real(est).double() - torch.view_as_real(truth).double()
    return torch.stack([d.square().sum(), torch.view_as_real(truth).double().square().sum()])


def _check_sums(got, ref, what):
    got, ref = got.double().cpu(), ref.double().cpu()
    assert bool(((got - ref).abs() <= SUMS_RTOL * ref).all()), (what, got.tolist(), ref.tolist())


def test_evaluator_bench_workload():
    """Ada bf16, B = 65536 (eight internal chunks): the gathered rows are model(x) bit for bit, the sums match fp64."""
    nt, B = net("ada"), 65536
    x, cond = nt.inputs(B, seed=65536)
    xd, md = torch.from_numpy(x).cuda(), tuple(t.cuda() if torch.is_tensor(t) else t for t in util.meta(*cond))
    truth = torch.from_numpy(_truth(B, nt.grid, 1)).cuda()
    nt.model.precision = "bf16"
    ev = D.ShardedEvaluator(nt.model, B, "peer")
    try:
        assert ev.world == 1 and ev.peer.world == 1
        with torch.no_grad():
            g, s = ev.step(xd, md, truth)
            ref = nt.model(xd, md)
        assert torch.equal(_ints(g), _ints(ref))
        _check_sums(s, _sums64(ref, truth), "sums")
        nt.oracle_gate("bf16", g.cpu().numpy(), x, cond, _edge_rows(B, range(0, B, 8192))[:6] + [B - 1], "B=65536")
    finally:
        ev.close()


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_evaluator_generic_grid(prec):
    """S65 (odd pix): the evaluator stages the estimates of a non-default geometry, bf16 included (the fused head serves
    the reference grid only), and gathers them at odd row counts."""
    nt, B = net("S65"), 7
    x, cond = nt.inputs(B, seed=65)
    xd, md = torch.from_numpy(x).cuda(), tuple(t.cuda() if torch.is_tensor(t) else t for t in util.meta(*cond))
    truth = torch.from_numpy(_truth(B, nt.grid, 4)).cuda()
    nt.model.precision = prec
    ev = D.ShardedEvaluator(nt.model, B, "peer")
    try:
        with torch.no_grad():
            ref = nt.model(xd, md)
            g, s = ev.step(xd, md, truth)
            assert torch.equal(_ints(g), _ints(ref))
            _check_sums(s, _sums64(ref, truth), "sums")
            _ints(ev.peer.gathered).fill_(SENTINEL)
            ev.peer.row0 = 1
            g, _ = ev.step(xd[:5], tuple(t[:5] if torch.is_tensor(t) else t for t in md), truth[:5])
            torch.cuda.synchronize()
            _check_rows([g], 1, ref[:5])
    finally:
        ev.close()


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_evaluator_host_nccl_and_partial_steps(prec):
    """B = 5000: the host-input step, mode "nccl" and a short step against the device step."""
    nt, B = net("ada"), 5000
    x, cond = nt.inputs(B, seed=5000 + len(prec))
    xd, md = torch.from_numpy(x).cuda(), tuple(t.cuda() if torch.is_tensor(t) else t for t in util.meta(*cond))
    truth = torch.from_numpy(_truth(B, nt.grid, 2)).cuda()
    nt.model.precision = prec
    ev = D.ShardedEvaluator(nt.model, B, "peer")
    try:
        with torch.no_grad():
            ref = nt.model(xd, md)
            g, s = ev.step(xd, md, truth)
            assert torch.equal(_ints(g), _ints(ref)), "device step"
            sums_ref = _sums64(ref, truth)
            _check_sums(s, sums_ref, "device step")
            _ints(ev.peer.gathered).fill_(SENTINEL)
            host_out = torch.empty((B, *nt.grid), dtype=torch.complex64).pin_memory()
            g2, s2 = ev.step(torch.from_numpy(x).pin_memory(), util.meta(*cond), truth, host_out=host_out)
            assert torch.equal(_ints(host_out), _ints(ref.cpu())), "host_out"
            assert torch.equal(_ints(g2), _ints(ref)), "gathered after the host step"
            _check_sums(s2, sums_ref, "host step")
            nccl = D.ShardedEvaluator(nt.model, B, "nccl")
            g3, s3 = nccl.step(xd, md, truth)
            assert torch.equal(_ints(g3), _ints(ref)), "nccl mode"
            _check_sums(s3, sums_ref, "nccl mode")
            # a step over fewer samples than rows_per_rank leaves the rows it does not own untouched
            n = 4000
            for host in (False, True):
                _ints(ev.peer.gathered).fill_(SENTINEL)
                inp = (torch.from_numpy(x[:n]).pin_memory(), util.meta(*(a[:n] for a in cond))) if host else \
                    (xd[:n], tuple(t[:n] if torch.is_tensor(t) else t for t in md))
                g4, s4 = ev.step(*inp, truth[:n])
                torch.cuda.synchronize()
                _check_rows([g4], 0, ref[:n])
                _check_sums(s4, _sums64(ref[:n], truth[:n]), f"short step, host {host}")
    finally:
        ev.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. several processes
# ---------------------------------------------------------------------------------------------------------------------
WORLD = min(torch.cuda.device_count(), 8) if torch.cuda.is_available() else 0
MP_CASES = [("ada", "bf16"), ("ada", "fp32"), ("S65", "bf16")]


def _mp_case(rank, world, backend, dev, name, prec):
    nt = Net(name, device=str(dev))
    nt.model.precision = prec
    B = 2 * world + 1
    rpr = -(-B // world)
    lo, hi = D.shard_range(B, rank, world)
    x, cond = nt.inputs(B, seed=77)
    truth = torch.from_numpy(_truth(B, nt.grid, 3)).to(dev)
    meta = lambda a, b: tuple(t.to(dev) if torch.is_tensor(t) else t for t in util.meta(*(c[a:b] for c in cond))) \
        if cond is not None else None
    res = dict(B=B, rpr=rpr, lo=lo, hi=hi)
    with torch.no_grad():
        full = nt.model(torch.from_numpy(x).to(dev), meta(0, B))
        res["full"] = _ints(full).cpu().numpy()
        res["sums64"] = _sums64(full, truth).cpu().numpy()
        ev = D.ShardedEvaluator(nt.model, rpr, "peer")
        try:
            def fill():
                _ints(ev.peer.gathered).fill_(SENTINEL)
                torch.cuda.synchronize(dev)
                dist.barrier()
            fill()
            g, s = ev.step(torch.from_numpy(x[lo:hi]).to(dev), meta(lo, hi), truth[lo:hi])
            # stream-ordered read right after the step: the sums' all-reduce orders it after every rank's stores
            res["gathered"], res["sums"] = _ints(g).clone().cpu().numpy(), s.clone().cpu().numpy()
            dist.barrier()
            fill()
            host_out = torch.empty((hi - lo, *nt.grid), dtype=torch.complex64).pin_memory()
            hm = util.meta(*(c[lo:hi] for c in cond)) if cond is not None else None
            g, s = ev.step(torch.from_numpy(x[lo:hi]).pin_memory(), hm, truth[lo:hi], host_out=host_out)
            res["gathered_host"], res["sums_host"] = _ints(g).clone().cpu().numpy(), s.clone().cpu().numpy()
            res["host_out"] = _ints(host_out).numpy().copy()
            dist.barrier()
        finally:
            ev.close()
        if backend == "nccl":     # the serial baseline gathers with NCCL
            ev = D.ShardedEvaluator(nt.model, rpr, "nccl")
            g, s = ev.step(torch.from_numpy(x[lo:hi]).to(dev), meta(lo, hi), truth[lo:hi])
            res["gathered_nccl"], res["sums_nccl"] = _ints(g).cpu().numpy(), s.cpu().numpy()
    nt.model._release()
    return res


def _gather_worker(rank, world, port, q, backend):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        gpu = rank if backend == "nccl" else 0
        torch.cuda.set_device(gpu)
        dev = torch.device("cuda", gpu)
        timeout = datetime.timedelta(seconds=120)
        if backend == "nccl":
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=timeout)
        else:
            dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timeout)
        try:
            out = dict(rank=rank, cases={})
            for name, prec in MP_CASES:
                out["cases"][(name, prec)] = _mp_case(rank, world, backend, dev, name, prec)
            q.put(out)
        finally:
            dist.destroy_process_group()
    except BaseException:
        q.put(dict(rank=rank, error=traceback.format_exc()))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module", params=["nccl", "gloo, 2 ranks on one GPU"])
def ranks(request):
    backend = request.param.split(",")[0]
    world = WORLD if backend == "nccl" else 2
    if backend == "nccl" and WORLD < 2:
        pytest.skip("needs two or more GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, world, port, q, backend)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        out = sorted((q.get(timeout=900) for _ in procs), key=lambda r: r["rank"])
        for p in procs:
            p.join(timeout=120)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
    errors = [f"rank {r['rank']}:\n{r['error']}" for r in out if "error" in r]
    assert not errors, "\n".join(errors)
    return backend, out


@pytest.mark.parametrize("case", MP_CASES, ids=lambda c: f"{c[0]}-{c[1]}")
def test_ranks_gather_unequal_shards(ranks, case):
    backend, out = ranks
    world = len(out)
    res = [r["cases"][case] for r in out]
    B, rpr = res[0]["B"], res[0]["rpr"]
    full = res[0]["full"]
    for r, c in enumerate(res):
        assert np.array_equal(c["full"], full), f"rank {r}: plain forward"
        lo, hi = D.shard_range(B, r, world)
        assert (c["lo"], c["hi"]) == (lo, hi)
        for key in ("gathered", "gathered_host") + (("gathered_nccl",) if backend == "nccl" else ()):
            g = c[key]
            if key == "gathered_nccl":       # gather_estimates trims the padding
                assert np.array_equal(g, full), (r, key)
                continue
            assert g.shape[0] == world * rpr, (r, key)
            for p in range(world):
                plo, phi = D.shard_range(B, p, world)
                assert np.array_equal(g[p * rpr:p * rpr + phi - plo], full[plo:phi]), (r, key, p)
                assert (g[p * rpr + phi - plo:(p + 1) * rpr] == np.int32(SENTINEL)).all(), (r, key, p, "padding")
        assert np.array_equal(c["host_out"], full[lo:hi]), (r, "host_out")
        for key in ("sums", "sums_host") + (("sums_nccl",) if backend == "nccl" else ()):
            assert np.array_equal(c[key], res[0][key]), (r, key, "differs between ranks")
            _check_sums(torch.from_numpy(c[key]), torch.from_numpy(c["sums64"]), f"rank {r} {key}")
    name, prec = case
    nt = net(name)             # the same weights and inputs as the workers'
    x, cond = nt.inputs(B, seed=77)
    nt.oracle_gate(prec, full.view(np.complex64)[..., 0], x, cond, list(range(B)), f"{backend} {case}")
