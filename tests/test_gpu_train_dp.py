"""GPU: dropout masks indexed by global sample (``aft_forward_train_offset``, ``forward(sample_offset=, dropout_seed=)``)
and data-parallel training over the GPUs of one node (``distributed.ShardedTrainer``).

On one GPU: the offset call at ``sample0 = 0`` is bit-identical to ``aft_forward_train``; a batch forwarded as two shards
with their offsets reproduces the one-call outputs bit for bit and, summed, its gradient within the gate of
``tests/test_gpu_train.py`` against the fp64 restatement; the counter reaches 2^32 - 1 correctly; bad offsets are refused
with nothing launched.

Over several ranks, spawned once per arm: one NCCL worker per GPU (skipped with fewer than two GPUs), and two gloo
workers sharing one GPU (runs on any GPU box: the same kernels and ShardedTrainer logic, host-staged collectives).  Unequal shards
reproduce the single-GPU outputs bit for bit whatever each rank's ``torch.manual_seed``; reduced gradients are
bit-identical across ranks and pass the gate against the global batch's fp64 restatement; five Adam steps keep the
replicas bit-identical and follow the fp64 trajectory; an empty shard takes part; ``DistributedDataParallel`` over the
same keywords agrees with ``ShardedTrainer`` to fp32 summation error."""
import ctypes as C
import hashlib
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from adafortitran_b200 import _capi
from adafortitran_b200 import distributed as D
from oracle import aft_oracle as O
from oracle import train_ref as T
from tests import util
from tests.dp_masks import masks_for
from tests.test_gpu_train import TOL, _gate, _inputs, _nw, _seed_of
from tests.test_gpu_train_scale import _away_from_kinks, _ref_on_gpu

pytestmark = pytest.mark.gpu
P_DROP = 0.1
LR = 5e-4
ADAM_STEPS = 5


@pytest.fixture(scope="module", autouse=True)
def fp32_without_tf32():
    """The stock fp32 arm of the gate must be true fp32 (cuDNN convolutions default to TF32)."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


def _model(device="cuda"):
    m = util.make_model("ada", device=device, overrides={"dropout": P_DROP}, weights=util.ada_weights())
    m.trainable = True
    return m.train()


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _raw(model, pilots, cond, g, seed, sample0=None):
    """aft_forward_train (sample0 None) or aft_forward_train_offset, then aft_backward for loss = <g, out>, straight
    through the C-ABI.  Returns (out, flat gradient) as numpy."""
    lib = _capi.lib()
    model._ensure_handle()
    model._sync_weights()
    dev, n, h = model.device, len(pilots), model._handle
    x = torch.from_numpy(pilots).to(dev, torch.complex64).contiguous()
    c = [torch.from_numpy(np.asarray(v, np.float32)).to(dev) for v in cond]
    out = torch.empty((n, 120, 14), dtype=torch.complex64, device=dev)
    need = lib.aft_train_workspace_bytes(h, n)
    ws = torch.empty(need + 256, dtype=torch.uint8, device=dev)
    ptr = C.c_void_p((ws.data_ptr() + 255) // 256 * 256)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    head = (h, _vp(x), _vp(c[0]), _vp(c[1]), _vp(c[2]), _vp(out), n)
    if sample0 is None:
        _capi.check(lib.aft_forward_train(*head, P_DROP, seed, ptr, need, st))
    else:
        _capi.check(lib.aft_forward_train_offset(*head, sample0, P_DROP, seed, ptr, need, st))
    gout = torch.view_as_real(torch.from_numpy(g).to(dev, torch.complex64)).contiguous()
    flat = torch.zeros(lib.aft_param_count(h), dtype=torch.float32, device=dev)
    _capi.check(lib.aft_backward(h, _vp(gout), n, ptr, need, _vp(flat), st))
    return out.cpu().numpy(), flat.cpu().numpy()


def _ours(model, pilots, cond, g, seed, offset):
    """One differentiable call with explicit offset and seed, loss = <g, out>: (out, {name: grad})."""
    model.zero_grad(set_to_none=True)
    out = model(torch.from_numpy(pilots), util.meta(*cond), sample_offset=offset, dropout_seed=seed)
    gt = torch.from_numpy(g).to(out.device)
    (out.real * gt.real.float() + out.imag * gt.imag.float()).sum().backward()
    named, _ = model._weight_tensors()
    return out.detach().cpu().numpy(), {n: t.grad.detach().cpu().double().numpy() for n, t in named}


def _global_masks(seed, spans):
    """[real, imaginary] masks[layer][site] of the samples of consecutive ``spans``, each drawn with first = lo."""
    parts = [[masks_for(seed, hi - lo, e, 6, P_DROP, first=lo) for lo, hi in spans] for e in (0, 1)]
    return [[[torch.cat([m[l][s] for m in part]) for s in range(4)] for l in range(6)] for part in parts]


def _gate_vs_restatement(model, pilots, cond, g, masks, ours, ours_out, what):
    ref_out, ref = _ref_on_gpu(model, pilots, cond, g, torch.float64, p=P_DROP, masks=masks)
    _, stock = _ref_on_gpu(model, pilots, cond, g, torch.float32, p=P_DROP, masks=masks)
    assert _nw(ours_out.view(np.float32), ref_out.view(np.float64)) <= TOL, what
    _gate(ours, stock, ref, what)


# ---------------------------------------------------------------------------------------------------------------------
# one GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_offset_zero_bit_identical_to_forward_train():
    model = _model()
    pilots, cond, g = _inputs(3, seed=31)
    seed = 0x1234_5678_9ABC_DEF0
    o_a, g_a = _raw(model, pilots, cond, g, seed)
    o_b, g_b = _raw(model, pilots, cond, g, seed, sample0=0)
    assert np.array_equal(o_a.view(np.float32), o_b.view(np.float32))
    assert np.array_equal(g_a, g_b)
    o_c, _ = _raw(model, pilots, cond, g, seed, sample0=1)      # the offset reaches the masks
    assert not np.array_equal(o_a, o_c)


def test_two_shards_reproduce_one_call():
    model = _model()
    pilots, cond, g = _inputs(7, seed=32)
    seed = 0x0DD5_EED5_0001
    out, grads = _ours(model, pilots, cond, g, seed, 0)
    spans = [(0, 3), (3, 7)]
    outs, acc = [], None
    for lo, hi in spans:
        o, gr = _ours(model, pilots[lo:hi], [v[lo:hi] for v in cond], g[lo:hi], seed, lo)
        outs.append(o)
        acc = gr if acc is None else {n: acc[n] + gr[n] for n in acc}
    for lo, o in zip((0, 3), outs):
        assert np.array_equal(o.view(np.float32), out[lo:lo + len(o)].view(np.float32)), lo
    masks = _global_masks(seed, spans)
    _gate_vs_restatement(model, pilots, cond, g, masks, acc, np.concatenate(outs), "two shards, summed")
    _gate_vs_restatement(model, pilots, cond, g, masks, grads, out, "one call")


def test_counter_at_top_of_32_bits():
    """sample0 = 2^31 - 2, batch 2: the imaginary sequence of the last sample is 2^32 - 1."""
    model = _model()
    pilots, cond, g = _inputs(2, seed=33)
    seed = 0xC0FF_EE00_1234
    first = 2 ** 31 - 2
    out, grads = _ours(model, pilots, cond, g, seed, first)
    masks = [masks_for(seed, 2, e, 6, P_DROP, first=first) for e in (0, 1)]
    _gate_vs_restatement(model, pilots, cond, g, masks, grads, out, "sample0 2^31 - 2")


def test_refusals_and_repeatability():
    model = _model()
    pilots, cond, g = _inputs(2, seed=34)
    lib = _capi.lib()
    model._ensure_handle()
    model._sync_weights()                      # packing launches kernels: done before counting
    for sample0 in (-1, 2 ** 31 - 1, 2 ** 40):
        before = lib.aft_launch_count()
        with pytest.raises(ValueError) as e:
            _raw(model, pilots, cond, g, 5, sample0=sample0)
        assert e.value.status == _capi.AFT_ERR_INVALID and "2^31" in str(e.value), sample0
        assert lib.aft_launch_count() == before, sample0
    with pytest.raises(ValueError, match="2\\^31"):
        model(torch.from_numpy(pilots), util.meta(*cond), sample_offset=-3)
    with torch.no_grad():
        with pytest.raises(ValueError, match="inference"):
            model(torch.from_numpy(pilots), util.meta(*cond), sample_offset=4)
        with pytest.raises(ValueError, match="inference"):
            model(torch.from_numpy(pilots), util.meta(*cond), dropout_seed=4)
    o1, g1 = _ours(model, pilots, cond, g, 99, 5)
    torch.manual_seed(1)                       # the default generator plays no part when the seed is given
    o2, g2 = _ours(model, pilots, cond, g, 99, 5)
    assert np.array_equal(o1, o2) and all(np.array_equal(g1[n], g2[n]) for n in g1)


# ---------------------------------------------------------------------------------------------------------------------
# two or more GPUs
# ---------------------------------------------------------------------------------------------------------------------
WORLD = min(torch.cuda.device_count(), 8) if torch.cuda.is_available() else 0


def _batch(n, seed):
    pilots, cond, _ = _inputs(n, seed)
    truth = O.synthetic_channel(n, 15.0, 100.0, 600.0, seed=seed + 1)[1]
    return pilots, cond, truth


def _shard(data, lo, hi, dev):
    pilots, cond, truth = data
    md = tuple(t.to(dev) if torch.is_tensor(t) else t for t in util.meta(*[v[lo:hi] for v in cond]))
    return torch.from_numpy(pilots[lo:hi]).to(dev), md, torch.from_numpy(truth[lo:hi]).to(dev)


def _flat_grads(model):
    named, _ = model._weight_tensors()
    return {n: t.grad.detach().cpu().numpy().copy() for n, t in named}


def _digest(model):
    named, _ = model._weight_tensors()
    h = hashlib.sha256()
    for _, t in named:
        h.update(t.detach().cpu().numpy().tobytes())
    return h.hexdigest()


def _dp_worker(rank, world, port, q, backend, data):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    gpu = rank if backend == "nccl" else 0
    torch.cuda.set_device(gpu)
    dev = torch.device("cuda", gpu)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = dict(rank=rank, data=data)
        model = _model(f"cuda:{gpu}")
        trainer = D.ShardedTrainer(model)
        calls, outs = [], []
        model.register_forward_pre_hook(lambda m, a, kw: calls.append((kw.get("sample_offset"), kw.get("dropout_seed"))),
                                        with_kwargs=True)
        model.register_forward_hook(lambda m, a, o: outs.append(o.detach().clone()))
        # unequal shards, a different default generator on every rank
        B = 2 * world + 1
        lo, hi = D.shard_range(B, rank, world)
        torch.manual_seed(1000 + rank)
        res["loss"] = float(trainer.step(*_shard(data, lo, hi, dev), B))
        res["grads"] = _flat_grads(model)
        res["seed"], res["offset"] = calls[-1][1], calls[-1][0]
        local = outs[-1]
        torch.manual_seed(1000)                               # a single-GPU call over the global batch, rank 0's seed
        x, md, _ = _shard(data, 0, B, dev)
        full = model(x, md).detach()
        res["rows_identical"] = torch.equal(torch.view_as_real(local), torch.view_as_real(full[lo:hi]))
        model.zero_grad(set_to_none=True)                     # the global batch's gradient on one GPU
        x, md, t = _shard(data, 0, B, dev)
        err = model(x, md, sample_offset=0, dropout_seed=res["seed"]) - t
        (torch.cat([err.real, err.imag], 1).pow(2).sum() / (2 * B * 1680)).backward()
        res["single_grads"] = _flat_grads(model)
        # global batch 1: every rank but 0 holds an empty shard
        lo1, hi1 = D.shard_range(1, rank, world)
        data1 = _batch(1, seed=43)
        trainer.step(*_shard(data1, lo1, hi1, dev), 1)
        res["empty_grads"] = _flat_grads(model)
        res["empty_local"] = hi1 - lo1
        model.zero_grad(set_to_none=True)                     # the same sample on one GPU, the same loss formula
        x, md, t = _shard(data1, 0, 1, dev)
        est = model(x, md, sample_offset=0, dropout_seed=calls[-1][1])
        err = est - t
        (torch.cat([err.real, err.imag], 1).pow(2).sum() / (2 * 1680)).backward()
        res["empty_single"] = _flat_grads(model)
        # five Adam steps from identical replicas
        model = _model(f"cuda:{gpu}")
        trainer = D.ShardedTrainer(model)
        seeds = []
        model.register_forward_pre_hook(lambda m, a, kw: seeds.append(kw.get("dropout_seed")), with_kwargs=True)
        named, _ = model._weight_tensors()
        theta0 = {n: t.detach().cpu().double().clone() for n, t in named}
        opt = torch.optim.Adam(model.parameters(), lr=LR)
        torch.manual_seed(2000 + rank)
        res["digests"] = []
        for step in range(ADAM_STEPS):
            trainer.step(*_shard(_batch(B, seed=300 + step), lo, hi, dev), B)
            opt.step()
            res["digests"].append(_digest(model))
        named, _ = model._weight_tensors()
        res["adam_delta"] = {n: (t.detach().cpu().double() - theta0[n]).numpy() for n, t in named}
        res["adam_seeds"] = seeds
        # DistributedDataParallel over the same keywords, equal shards
        from torch.nn.parallel import DistributedDataParallel as DDP
        model = _model(f"cuda:{gpu}")
        trainer = D.ShardedTrainer(model)
        Be = 2 * world
        lo2, hi2 = D.shard_range(Be, rank, world)
        data2 = _batch(Be, seed=45)
        shard = _shard(data2, lo2, hi2, dev)
        seeds2 = []
        model.register_forward_pre_hook(lambda m, a, kw: seeds2.append(kw.get("dropout_seed")), with_kwargs=True)
        trainer.step(*shard, Be)
        ours = _flat_grads(model)
        ddp = DDP(model, device_ids=[gpu], broadcast_buffers=False)
        model.zero_grad(set_to_none=True)
        est = ddp(shard[0], shard[1], sample_offset=lo2, dropout_seed=seeds2[-1])
        err = est - shard[2]
        (torch.cat([err.real, err.imag], 1).pow(2).sum() / (2 * (hi2 - lo2) * 1680)).backward()
        theirs = _flat_grads(model)
        res["ddp_err"] = {n: _nw(theirs[n], ours[n]) for n in ours}
        res["ddp_err_all"] = _nw(np.concatenate([theirs[n].ravel() for n in ours]),
                                 np.concatenate([ours[n].ravel() for n in ours]))
        del ddp
        torch.cuda.synchronize()
        q.put(res)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module", params=["nccl", "gloo, 2 ranks on one GPU"])
def dp(request):
    backend = request.param.split(",")[0]
    world = WORLD if backend == "nccl" else 2
    if backend == "nccl" and WORLD < 2:
        pytest.skip("needs two or more GPUs")
    # the unequal-shard batch, its pilots redrawn away from ReLU kinks under the masks rank 0's first draw gives
    B = 2 * world + 1
    data = _batch(B, seed=41)
    masks = [T.masks_for(_seed_of(1000), B, e, 6, P_DROP) for e in (0, 1)]
    _away_from_kinks(_model(), data[0], data[1], p=P_DROP, masks=masks)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q, backend, data)) for r in range(world)]
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


def _mse_ref(model, data, masks, dtype):
    """The global batch's MSE(cat(re, im)) through the restatement in ``dtype`` on the GPU: {name: gradient}."""
    pilots, cond, truth = data
    named, _ = model._weight_tensors()
    P = {n: t.detach().to("cuda", dtype).clone().requires_grad_(True) for n, t in named}
    ct = torch.complex128 if dtype == torch.float64 else torch.complex64
    c = [torch.from_numpy(np.asarray(v, np.float64)).to("cuda") for v in cond]
    mk = [[[s.to("cuda") for s in layer] for layer in part] for part in masks]
    out = T.forward(P, torch.from_numpy(pilots).to("cuda", ct), c, P_DROP, None, 6, masks=mk)
    t = torch.from_numpy(truth).to("cuda", ct)
    loss = torch.nn.functional.mse_loss(torch.cat([out.real, out.imag], 1), torch.cat([t.real, t.imag], 1))
    return P, loss


def test_unequal_shards_match_single_gpu_and_fp64(dp):
    assert len({r["seed"] for r in dp}) == 1
    assert [r["offset"] for r in dp] == [D.shard_range(2 * len(dp) + 1, r, len(dp))[0] for r in range(len(dp))]
    assert all(r["rows_identical"] for r in dp)
    for r in dp[1:]:
        assert all(np.array_equal(r["grads"][n], dp[0]["grads"][n]) for n in r["grads"]), r["rank"]
        assert r["loss"] == dp[0]["loss"]
    B = 2 * len(dp) + 1
    data = dp[0]["data"]
    masks = [T.masks_for(dp[0]["seed"], B, e, 6, P_DROP) for e in (0, 1)]
    model = _model()
    arms = {}
    for dt in (torch.float64, torch.float32):
        P, loss = _mse_ref(model, data, masks, dt)
        arms[dt] = {n: g.double().cpu().numpy() for n, g in zip(P, torch.autograd.grad(loss, list(P.values())))}
    ours = {n: g.astype(np.float64) for n, g in dp[0]["grads"].items()}
    one = {n: g.astype(np.float64) for n, g in dp[0]["single_grads"].items()}
    cat = lambda d: np.concatenate([d[n].ravel() for n in ours])
    print(f"{len(dp)} ranks vs one GPU, global batch {B}: gradients {_nw(cat(ours), cat(one)):.2e} apart")
    _gate(one, arms[torch.float32], arms[torch.float64], f"one GPU, global batch {B}")
    _gate(ours, arms[torch.float32], arms[torch.float64], f"{len(dp)} ranks, global batch {B}")


def test_empty_shard_takes_part(dp):
    assert [r["empty_local"] for r in dp] == [1] + [0] * (len(dp) - 1)
    for r in dp:
        assert all(np.array_equal(r["empty_grads"][n], dp[0]["empty_single"][n]) for n in r["empty_grads"]), r["rank"]


def test_adam_steps_identical_replicas_and_fp64_trajectory(dp):
    """theta_5 - theta_0 of the data-parallel run against fp64 Adam on the restatement, gated like the SGD trajectory
    of tests/test_gpu_train.py with a single-GPU ShardedTrainer run of the same global batches and seeds as the bar.
    (Stock fp32 autograd is no bar for Adam: it normalises every element, so elements whose gradient is near zero
    differ by O(1) between any two fp32 summation orders, and ours and stock sum in different orders.)"""
    for r in dp[1:]:
        assert r["digests"] == dp[0]["digests"], r["rank"]
    assert len(set(dp[0]["digests"])) == ADAM_STEPS
    B = 2 * len(dp) + 1
    single = _model()
    trainer = D.ShardedTrainer(single)             # no process group: world 1
    seeds = []
    single.register_forward_pre_hook(lambda m, a, kw: seeds.append(kw.get("dropout_seed")), with_kwargs=True)
    named, _ = single._weight_tensors()
    theta0 = {n: t.detach().double().clone() for n, t in named}
    opt = torch.optim.Adam(single.parameters(), lr=LR)
    P = {n: t.clone().requires_grad_(True) for n, t in theta0.items()}
    opt64 = torch.optim.Adam(list(P.values()), lr=LR)
    torch.manual_seed(2000)                         # rank 0's generator: the same seeds
    for step in range(ADAM_STEPS):
        pilots, cond, truth = _batch(B, seed=300 + step)
        x, md, t = _shard((pilots, cond, truth), 0, B, "cuda")
        trainer.step(x, md, t, B)
        opt.step()
        masks = [[[s.cuda() for s in layer] for layer in T.masks_for(seeds[-1], B, e, 6, P_DROP)] for e in (0, 1)]
        opt64.zero_grad()
        c = [torch.from_numpy(np.asarray(v, np.float64)).cuda() for v in cond]
        o = T.forward(P, torch.from_numpy(pilots).to("cuda", torch.complex128), c, P_DROP, None, 6, masks=masks)
        h = torch.from_numpy(truth).to("cuda", torch.complex128)
        torch.nn.functional.mse_loss(torch.cat([o.real, o.imag], 1), torch.cat([h.real, h.imag], 1)).backward()
        opt64.step()
    assert seeds == dp[0]["adam_seeds"]
    named, _ = single._weight_tensors()
    one = {n: (t.detach().double() - theta0[n]).cpu().numpy() for n, t in named}
    ref = {n: (P[n].detach() - theta0[n]).cpu().numpy() for n in theta0}
    _gate(dp[0]["adam_delta"], one, ref, f"{len(dp)} ranks, Adam theta_5 - theta_0 (bar: one GPU)")


def test_ddp_agrees_with_sharded_trainer(dp):
    for r in dp:
        worst = max(r["ddp_err"].items(), key=lambda kv: kv[1])
        print(f"rank {r['rank']}: DDP vs ShardedTrainer, all {r['ddp_err_all']:.2e}, worst {worst[0]} {worst[1]:.2e}")
        assert r["ddp_err_all"] <= 1e-6 and worst[1] <= 1e-5, (r["rank"], worst)
