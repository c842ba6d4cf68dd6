"""GPU: synthetic channels generated on the device (``aft_synthetic_channels``, ``data.SyntheticChannels``).

1. Per sample against the fp64 restatement ``oracle/channel_ref.py``: drawn conditions bit-exact, pilots and truth
   within 1e-6 normwise (max|x - ref| / max|ref| of each sample) at 120 x 14 (pilots 12 x 2), 3276 x 14 (1638 x 2),
   65 x 12 (13 x 2) and 24 x 13 (5 x 1: an odd number of symbols, so rows straddle 16-byte boundaries and take the
   kernel's 8-byte stores, and of pilots, so the last pilot's noise is half a draw).  On the CPU,
   ``tests/test_synthetic_cpu.py`` shows this gate catches a frequency phase taken in fp32 without turn reduction.
2. Shard and chunk invariance: rows [a, b) of ``batch(0, N)`` are bit-identical to ``batch(a, b - a)`` for N past the
   grid-stride edge of the kernel (4 CTAs per SM, one sample per CTA at a time); samples 2^32 - 1 and 2^32 (the high
   counter word); the same seed gives bit-identical output, another seed does not.
3. ``SyntheticChannels`` end to end: fixed and drawn conditions, the meta tuple in the Ada model's forward, and two gloo
   ranks on one GPU that generate their own ``shard_range`` rows and take one ``ShardedTrainer.step``.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from adafortitran_b200 import distributed as D
from adafortitran_b200.data import SyntheticChannels
from oracle import aft_oracle as O
from oracle import channel_ref as R
from oracle import train_ref as T
from tests import util
from tests.test_gpu_train import _gate, _nw

pytestmark = pytest.mark.gpu
GATE = 1e-6
GEOMS = {"120x14": (120, 14, 12, 2), "3276x14": (3276, 14, 1638, 2), "65x12": (65, 12, 13, 2), "24x13": (24, 13, 5, 1)}
P_DROP = 0.1


def _sys(g):
    return dict(ofdm=dict(num_scs=g[0], num_symbols=g[1]), pilot=dict(num_scs=g[2], num_symbols=g[3]))


def _gen(g, seed, sample0, n, cond=None):
    pilots, meta, truth = SyntheticChannels(_sys(g), seed, conditions=cond).batch(sample0, n)
    torch.cuda.synchronize()
    return pilots.cpu().numpy(), [m.cpu().numpy() if torch.is_tensor(m) else m for m in meta], truth.cpu().numpy()


def _ref(g, seed, sample0, n, cond=None):
    return R.synthetic_channels(seed, sample0, n, *g, cond=cond)


def _check_vs_ref(ours, ref, what):
    pilots, meta, truth = ours
    rp, rt, (snr, ds, dop) = ref
    for got, want in zip(meta[1:4], (snr, ds, dop)):
        assert np.array_equal(got.reshape(-1), want), what
    ep = max(O.normwise_err(a, b) for a, b in zip(pilots, rp))
    et = max(O.normwise_err(a, b) for a, b in zip(truth, rt))
    print(f"{what}: worst sample, pilots {ep:.2e}, truth {et:.2e}")
    assert ep <= GATE and et <= GATE, (what, ep, et)


CASES = [("120x14", 200, None), ("120x14", 16, (30.0, 350.0, 1400.0)), ("3276x14", 12, None),
         ("3276x14", 6, (30.0, 350.0, 1400.0)), ("65x12", 50, None), ("65x12", 7, (-3.5, 17.25, 0.0)),
         ("24x13", 31, None)]


@pytest.mark.parametrize("geom,n,cond", CASES)
def test_against_fp64_restatement(geom, n, cond):
    g = GEOMS[geom]
    sample0 = 1000 + n
    _check_vs_ref(_gen(g, 0xA5A5_0123_4567_89AB, sample0, n, cond), _ref(g, 0xA5A5_0123_4567_89AB, sample0, n, cond),
                  f"{geom} n={n} cond={cond}")


def _grid_stride():
    return torch.cuda.get_device_properties(0).multi_processor_count * 4


@pytest.mark.parametrize("geom", ["120x14", "65x12", "24x13"])
def test_shard_and_chunk_invariance(geom):
    g, G = GEOMS[geom], _grid_stride()
    N = G + 37
    seed = 4242
    full = _gen(g, seed, 0, N)
    for a, b in ((0, 1), (1, G), (G - 1, G + 1), (G, N), (5, N - 3), (N - 1, N)):
        part = _gen(g, seed, a, b - a)
        assert np.array_equal(part[0].view(np.float32), full[0][a:b].view(np.float32)), (a, b)
        assert np.array_equal(part[2].view(np.float32), full[2][a:b].view(np.float32)), (a, b)
        for m, fm in zip(part[1][1:4], full[1][1:4]):
            assert np.array_equal(m, fm[a:b]), (a, b)
    again = _gen(g, seed, 0, N)
    assert all(np.array_equal(x.view(np.float32), y.view(np.float32)) for x, y in ((again[0], full[0]), (again[2], full[2])))
    other = _gen(g, seed + 1, 0, N)
    assert not np.array_equal(other[2], full[2]) and not np.array_equal(other[0], full[0])
    # the sample index is the only thing that differs between rows: each row is its own sample
    assert len({full[2][i].tobytes() for i in range(N)}) == N


def test_chunks_of_a_large_grid():
    """3276 x 14: the frequency factors are held 144 subcarriers at a time (22 full chunks and 108); a batch split
    across calls gives the same rows."""
    g = GEOMS["3276x14"]
    full = _gen(g, 9, 0, 5)
    for a, b in ((0, 2), (2, 5), (4, 5)):
        part = _gen(g, 9, a, b - a)
        assert np.array_equal(part[2].view(np.float32), full[2][a:b].view(np.float32))
        assert np.array_equal(part[0].view(np.float32), full[0][a:b].view(np.float32))


def test_high_counter_word():
    g = GEOMS["120x14"]
    first = 2 ** 32 - 2
    ours = _gen(g, 77, first, 4)
    _check_vs_ref(ours, _ref(g, 77, first, 4), "samples 2^32 - 2 .. 2^32 + 1")
    for s in (2 ** 32 - 1, 2 ** 32):
        one = _gen(g, 77, s, 1)
        assert np.array_equal(one[2].view(np.float32), ours[2][s - first:s - first + 1].view(np.float32)), s
    # 2^32 is not sample 0 with the high word dropped
    assert not np.array_equal(_gen(g, 77, 0, 1)[2], ours[2][2:3])
    top = 2 ** 63 - 4                       # the last samples of the index range: sample0 + batch <= 2^63 - 1
    _check_vs_ref(_gen(g, 77, top, 3), _ref(g, 77, top, 3), "samples 2^63 - 4 .. 2^63 - 2")


# ---------------------------------------------------------------------------------------------------------------------
# SyntheticChannels end to end
# ---------------------------------------------------------------------------------------------------------------------
def test_fixed_and_drawn_conditions_in_the_model():
    g = GEOMS["120x14"]
    gen = SyntheticChannels(_sys(g), 3, conditions=(15, 100, 600))
    pilots, meta, truth = gen.batch(40, 9)
    assert pilots.shape == (9, 12, 2) and truth.shape == (9, 120, 14) and pilots.dtype == truth.dtype == torch.complex64
    assert pilots.device.type == truth.device.type == "cuda"
    assert len(meta) == 6 and all(m.shape == (9, 1) and m.dtype == torch.float32 for m in meta[:5])
    assert meta[5] == [("synthetic",) * 9]
    assert torch.equal(meta[0].reshape(-1).cpu(), torch.arange(40, 49, dtype=torch.float32))
    assert [float(m.unique()) for m in meta[1:5]] == [15.0, 100.0, 600.0, 10.0]
    drawn = SyntheticChannels(_sys(g), 3)
    p2, m2, t2 = drawn.batch(40, 300)
    snr, ds, dop = R.conditions(3, np.arange(40, 340, dtype=np.uint64))
    for got, want in zip(m2[1:4], (snr, ds, dop)):
        assert np.array_equal(got.reshape(-1).cpu().numpy(), want)
    assert len(set(np.unique(m2[1].cpu().numpy()))) == 7
    # the same sample with its drawn condition fixed is the same sample
    s = 40 + 123
    cond = (float(m2[1][123]), float(m2[2][123]), float(m2[3][123]))
    p3, _, t3 = SyntheticChannels(_sys(g), 3, conditions=cond).batch(s, 1)
    assert torch.equal(torch.view_as_real(t3[0]), torch.view_as_real(t2[123]))
    assert torch.equal(torch.view_as_real(p3[0]), torch.view_as_real(p2[123]))
    model = util.make_model("ada", weights=util.ada_weights())
    with torch.no_grad():
        est = model(p2, m2)
    assert est.shape == (300, 120, 14) and torch.isfinite(torch.view_as_real(est)).all()
    assert gen.batch(0, 0)[2].shape == (0, 120, 14)
    with pytest.raises(ValueError):
        gen.batch(-1, 3)


def _model(device="cuda"):
    m = util.make_model("ada", device=device, overrides={"dropout": P_DROP}, weights=util.ada_weights())
    m.trainable = True
    return m.train()


def _flat_grads(model):
    named, _ = model._weight_tensors()
    return {n: t.grad.detach().cpu().numpy().copy() for n, t in named}


SEED, STEP, WORLD = 0x5EED_0000_0042, 3, 2
B = 2 * WORLD + 1


def _dp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        gen = SyntheticChannels(_sys(GEOMS["120x14"]), SEED)
        lo, hi = D.shard_range(B, rank, world)
        local = gen.batch(STEP * B + lo, hi - lo)
        full = gen.batch(STEP * B, B)
        same = torch.equal(torch.view_as_real(local[0]), torch.view_as_real(full[0][lo:hi])) and \
            torch.equal(torch.view_as_real(local[2]), torch.view_as_real(full[2][lo:hi])) and \
            all(torch.equal(a, b[lo:hi]) for a, b in zip(local[1][:5], full[1][:5])) and \
            local[1][5] == [full[1][5][0][lo:hi]]
        model = _model()
        trainer = D.ShardedTrainer(model)
        seeds = []
        model.register_forward_pre_hook(lambda m, a, kw: seeds.append(kw.get("dropout_seed")), with_kwargs=True)
        torch.manual_seed(1000 + rank)
        loss = float(trainer.step(*local, B))
        q.put(dict(rank=rank, same=same, grads=_flat_grads(model), seed=seeds[-1], loss=loss))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module")
def dp():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, WORLD, port, q)) for r in range(WORLD)]
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
    return out


def _mse_ref(model, pilots, cond, truth, masks, dtype):
    named, _ = model._weight_tensors()
    P = {n: t.detach().to("cuda", dtype).clone().requires_grad_(True) for n, t in named}
    ct = torch.complex128 if dtype == torch.float64 else torch.complex64
    c = [v.to("cuda", torch.float64).reshape(-1) for v in cond]
    mk = [[[s.to("cuda") for s in layer] for layer in part] for part in masks]
    out = T.forward(P, pilots.to(ct), c, P_DROP, None, 6, masks=mk)
    t = truth.to(ct)
    loss = torch.nn.functional.mse_loss(torch.cat([out.real, out.imag], 1), torch.cat([t.real, t.imag], 1))
    return {n: g.double().cpu().numpy() for n, g in zip(P, torch.autograd.grad(loss, list(P.values())))}


def test_two_ranks_generate_their_rows_and_train(dp):
    assert all(r["same"] for r in dp)
    assert dp[0]["seed"] == dp[1]["seed"] and dp[0]["loss"] == dp[1]["loss"]
    assert all(np.array_equal(dp[1]["grads"][n], dp[0]["grads"][n]) for n in dp[0]["grads"])
    # one GPU, the global batch in one call, the same dropout seed
    pilots, meta, truth = SyntheticChannels(_sys(GEOMS["120x14"]), SEED).batch(STEP * B, B)
    model = _model()
    model.zero_grad(set_to_none=True)
    err = model(pilots, meta, sample_offset=0, dropout_seed=dp[0]["seed"]) - truth
    (torch.cat([err.real, err.imag], 1).pow(2).sum() / (2 * B * 1680)).backward()
    one = {n: g.astype(np.float64) for n, g in _flat_grads(model).items()}
    ours = {n: g.astype(np.float64) for n, g in dp[0]["grads"].items()}
    masks = [T.masks_for(dp[0]["seed"], B, e, 6, P_DROP) for e in (0, 1)]
    ref64 = _mse_ref(model, pilots, meta[1:4], truth, masks, torch.float64)
    stock = _mse_ref(model, pilots, meta[1:4], truth, masks, torch.float32)
    cat = lambda d: np.concatenate([d[n].ravel() for n in ours])
    print(f"{WORLD} ranks vs one GPU, global batch {B}: gradients {_nw(cat(ours), cat(one)):.2e} apart")
    _gate(one, stock, ref64, f"one GPU, global batch {B}")
    _gate(ours, stock, ref64, f"{WORLD} ranks, global batch {B}")
