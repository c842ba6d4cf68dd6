"""LinearEstimator training: ``aft_linear_backward`` and the ``trainable = True`` autograd path against fp64.

``aft_linear_backward`` computes the three products of ``y = W x + b`` as tiles of ``C[m][n] = sum_r A[r][m] B[r][n]``
(``csrc/aux.cu``, ``linear_bwd_kernel``).  A CTA owns a slab of 128 rows of C; the sum over r runs in groups of 32,
summed in fp32 within a group and in fp64 across groups.  The weight gradient (C = grad_y^T [x | 1], rows = outputs, the
last column is the bias) also splits the batch into ``nz`` contiguous ranges of whole groups (``linear_bwd_plan``):
``nz = min(ceil(592 / tiles), 64, groups)`` with ``tiles = ceil(out / 128) * ceil((in + 1) / 32)``, then the groups per
range ``per = ceil(groups / nz)`` and ``nz = ceil(groups / per)``.  With ``nz > 1`` every range writes an fp32 partial
and ``linear_bwd_reduce_kernel`` adds them in range order in fp64.  The input gradient (C = grad_y W, rows = samples)
sums over the outputs: 1680 = 52 groups + a ragged group of 16 at the reference shape.

Reference shape 24 -> 1680: 14 slabs of 128 output rows (the last holds 16), one column tile, so ``nz = min(43, groups)``.

======  ======  =====  ============  ==========================  ===============================
batch   groups  nz     range (smp)   last range (samples)        what it covers
======  ======  =====  ============  ==========================  ===============================
1       1       1      32            1                           single sample, no reduction
2       1       1      32            2
31      1       1      32            31                          one ragged group
32      1       1      32            32                          one full group
33      2       2      32            1                           first split, ragged last group
1376    43      43     32            32                          43 full ranges of one group
1377    44      22     64            33 (1 group + 1 sample)     one past: ranges of two groups
4099    129     43     96            67 (2 groups + 3)           ragged last range and group
65537   2049    43     1536          1025 (32 groups + 1)        long ranges, ragged
======  ======  =====  ============  ==========================  ===============================

The gate is that of the training path (DESIGN §10): every gradient within ``max(2e-6, 4 x the stock fp32 error)``
normwise of fp64, where stock fp32 is torch's CPU autograd of ``nn.Linear`` on the same inputs."""
import ctypes as C

import numpy as np
import pytest
import torch

from adafortitran_b200 import _capi
from tests import util

REF = (24, 1680)
REF_BATCHES = (1, 2, 31, 32, 33, 1376, 1377, 4099, 65537)
GENERIC = ((7, 33, 19), (24, 3000, 5), (100, 64, 130), (4096, 16, 3))   # (in_dim, out_dim, batch)


def _plan(batch, in_dim, out_dim):
    """``linear_bwd_plan`` restated: (nz, samples per range)."""
    tiles = -(-out_dim // 128) * -(-(in_dim + 1) // 32)
    groups = -(-batch // 32)
    nz = max(1, min(1 if tiles >= 592 else -(-592 // tiles), 64, groups))
    per = -(-groups // nz) if groups else 1
    return (-(-groups // per) if groups else 1), per * 32


def _nw(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    d = np.linalg.norm(ref)
    return float(np.linalg.norm(a - ref) / (d if d > 0 else 1.0))


def _gate(stock):
    return max(2e-6, 4 * stock)


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _fp64(x, w, gy):
    x, w, gy = (np.asarray(a, np.float64) for a in (x, w, gy))
    return gy.T @ x, gy.sum(0), gy @ w


def _stock(x, w, gy):
    """torch CPU fp32 autograd of nn.Linear: (grad_w, grad_b, grad_x)."""
    lin = torch.nn.Linear(w.shape[1], w.shape[0])
    with torch.no_grad():
        lin.weight.copy_(torch.from_numpy(w))
    xt = torch.from_numpy(x).requires_grad_(True)
    lin(xt).backward(torch.from_numpy(gy))
    return lin.weight.grad.numpy(), lin.bias.grad.numpy(), xt.grad.numpy()


def _draw(rng, batch, in_dim, out_dim):
    x = rng.standard_normal((batch, in_dim)).astype(np.float32)
    w = (rng.standard_normal((out_dim, in_dim)) / np.sqrt(in_dim)).astype(np.float32)
    gy = rng.standard_normal((batch, out_dim)).astype(np.float32)
    return x, w, gy


def _backward(w, x, gy, with_x=True):
    """aft_linear_backward on device tensors; returns (grad_w, grad_b, grad_x or None) on the device."""
    out_dim, in_dim = w.shape
    batch = x.shape[0]
    gw = torch.full((out_dim, in_dim), float("nan"), device="cuda")
    gb = torch.full((out_dim,), float("nan"), device="cuda")
    gx = torch.full((batch, in_dim), float("nan"), device="cuda") if with_x else None
    need = _capi.lib().aft_linear_backward_workspace_bytes(batch, in_dim, out_dim)
    ws = torch.full((need // 4,), float("nan"), device="cuda")
    _capi.check(_capi.lib().aft_linear_backward(_vp(w), _vp(x), _vp(gy), _vp(gw), _vp(gb), _vp(gx), batch, in_dim, out_dim,
                                                _vp(ws), need, _stream()))
    return gw, gb, gx


def _check(x, w, gy, got, what):
    want, stock = _fp64(x, w, gy), _stock(x, w, gy)
    for name, g, r, s in zip(("grad_w", "grad_b", "grad_x"), got, want, stock):
        if g is None:
            continue
        g = g.detach().cpu().numpy() if torch.is_tensor(g) else g
        err, bar = _nw(g, r), _gate(_nw(s, r))
        assert err <= bar, f"{what}: {name} {err:.3g} > gate {bar:.3g} (stock {_nw(s, r):.3g})"


def _model(dtype=torch.float32, seed=0):
    from adafortitran_b200 import LinearEstimator, ModelConfig, SystemConfig
    torch.manual_seed(seed)
    m = LinearEstimator(SystemConfig(**util.SYS), ModelConfig(**dict(util.FORTI, model_type="linear", device="cuda")))
    return m.to(dtype)


# ----------------------------------------------------------------------------------------- CPU
def test_plan_table_and_workspace():
    lib = _capi.lib()
    table = {1: (1, 32), 2: (1, 32), 31: (1, 32), 32: (1, 32), 33: (2, 32), 1376: (43, 32), 1377: (22, 64),
             4099: (43, 96), 65537: (43, 1536)}
    for batch, plan in table.items():
        assert _plan(batch, *REF) == plan, batch
        nz = plan[0]
        assert lib.aft_linear_backward_workspace_bytes(batch, *REF) == max(256, nz * 1680 * 25 * 4 if nz > 1 else 0)
    assert lib.aft_linear_backward_workspace_bytes(0, *REF) == 256
    # a large W needs no split, so no partials: 3276 -> 45864 is 359 x 103 tiles
    assert _plan(3, 3276, 45864)[0] == 1 and lib.aft_linear_backward_workspace_bytes(10 ** 6, 3276, 45864) == 256
    for bad in ((-1, 24, 1680), (1, 0, 1680), (1, 4097, 1680), (1, 24, 0), (1, -3, 5)):
        assert lib.aft_linear_backward_workspace_bytes(*bad) == 0, bad


def test_refusals_launch_nothing():
    lib = _capi.lib()
    p = C.c_void_p(256)   # never dereferenced: every call below is refused before anything is enqueued
    need = lib.aft_linear_backward_workspace_bytes(4099, *REF)
    ok = dict(weight=p, x=p, grad_y=p, grad_w=p, grad_b=p, grad_x=None, batch=4099, in_dim=24, out_dim=1680, workspace=p,
              workspace_bytes=need, stream=None)
    cases = [(dict(weight=None), _capi.AFT_ERR_INVALID), (dict(grad_w=None), _capi.AFT_ERR_INVALID),
             (dict(grad_b=None), _capi.AFT_ERR_INVALID), (dict(x=None), _capi.AFT_ERR_INVALID),
             (dict(grad_y=None), _capi.AFT_ERR_INVALID), (dict(batch=-1), _capi.AFT_ERR_INVALID),
             (dict(in_dim=-24), _capi.AFT_ERR_INVALID), (dict(out_dim=-1), _capi.AFT_ERR_INVALID),
             (dict(in_dim=0), _capi.AFT_ERR_INVALID), (dict(in_dim=4097), _capi.AFT_ERR_INVALID),
             (dict(workspace=None), _capi.AFT_ERR_WORKSPACE), (dict(workspace_bytes=need - 1), _capi.AFT_ERR_WORKSPACE),
             (dict(batch=0, weight=None), _capi.AFT_ERR_INVALID), (dict(batch=0, workspace=None), _capi.AFT_ERR_WORKSPACE)]
    before = lib.aft_launch_count()
    for change, status in cases:
        a = {**ok, **change}
        rc = lib.aft_linear_backward(a["weight"], a["x"], a["grad_y"], a["grad_w"], a["grad_b"], a["grad_x"], a["batch"],
                                     a["in_dim"], a["out_dim"], a["workspace"], a["workspace_bytes"], a["stream"])
        assert rc == status, (change, rc, lib.aft_last_error())
    assert lib.aft_launch_count() == before


def test_trainable_contract_on_cpu():
    from adafortitran_b200 import LinearEstimator, ModelConfig, SystemConfig
    assert LinearEstimator.trainable is False
    m = LinearEstimator(SystemConfig(**util.SYS), ModelConfig(**dict(util.FORTI, model_type="linear", device="cpu")))
    assert m.trainable is False
    for trainable in (False, True):
        m.trainable = trainable
        m.train()
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            m(torch.zeros(2, 12, 2))
        with pytest.raises(RuntimeError, match="complex"):
            m(torch.zeros(2, 12, 2, dtype=torch.cfloat))


# ----------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("batch", REF_BATCHES)
def test_reference_shape_against_fp64(batch):
    rng = np.random.default_rng(batch)
    x, w, gy = _draw(rng, batch, *REF)
    tx, tw, tg = (torch.from_numpy(a).cuda() for a in (x, w, gy))
    got = _backward(tw, tx, tg)
    _check(x, w, gy, got, f"batch {batch}")
    again = _backward(tw, tx, tg)
    for a, b in zip(got, again):
        assert torch.equal(a, b), "repeated backward is not bit-identical"
    no_x = _backward(tw, tx, tg, with_x=False)     # grad_x = NULL: the other two are unchanged
    assert no_x[2] is None and torch.equal(no_x[0], got[0]) and torch.equal(no_x[1], got[1])


@pytest.mark.gpu
@pytest.mark.parametrize("in_dim,out_dim,batch", GENERIC)
def test_generic_shapes_against_fp64(in_dim, out_dim, batch):
    rng = np.random.default_rng(in_dim * 7 + out_dim)
    x, w, gy = _draw(rng, batch, in_dim, out_dim)
    got = _backward(*(torch.from_numpy(a).cuda() for a in (w, x, gy)))
    _check(x, w, gy, got, f"{in_dim} -> {out_dim}, batch {batch}")


@pytest.mark.gpu
def test_config5_sized_map():
    """3276 -> 45864 (W is 600 MB) at batch 3: 359 x 103 tiles, no split; grad_x sums 45864 terms per element."""
    in_dim, out_dim, batch = 3276, 45864, 3
    rng = np.random.default_rng(5)
    x, w, gy = _draw(rng, batch, in_dim, out_dim)
    gw, gb, gx = (t.cpu().numpy() for t in _backward(*(torch.from_numpy(a).cuda() for a in (w, x, gy))))
    want_b, want_x = gy.astype(np.float64).sum(0), gy.astype(np.float64) @ w.astype(np.float64)
    stock_b, stock_x = gy.sum(0), (torch.from_numpy(gy) @ torch.from_numpy(w)).numpy()
    assert _nw(gb, want_b) <= _gate(_nw(stock_b, want_b))
    assert _nw(gx, want_x) <= _gate(_nw(stock_x, want_x))
    num = den = stock_num = 0.0   # grad_w = gy^T x row block by row block (the fp64 product is 1.2 GB)
    for o in range(0, out_dim, 4096):
        ref = gy[:, o:o + 4096].astype(np.float64).T @ x.astype(np.float64)
        stock = (torch.from_numpy(gy[:, o:o + 4096]).T @ torch.from_numpy(x)).numpy()
        num += float(((gw[o:o + 4096] - ref) ** 2).sum())
        stock_num += float(((stock - ref) ** 2).sum())
        den += float((ref ** 2).sum())
    assert np.sqrt(num / den) <= _gate(np.sqrt(stock_num / den))


@pytest.mark.gpu
def test_misaligned_views_take_the_generic_path():
    """x and grad_y 4 bytes off a 16-byte boundary: element loads instead of 16-byte loads.  The groups, the batch ranges
    and the order of every sum are those of the fast path, so the gradients are bit-identical to it."""
    batch = 4099
    rng = np.random.default_rng(11)
    x, w, gy = _draw(rng, batch, *REF)
    tw = torch.from_numpy(w).cuda()
    xb, gb_ = torch.empty(batch * 24 + 1, device="cuda"), torch.empty(batch * 1680 + 1, device="cuda")
    xv, gv = xb[1:].view(batch, 24), gb_[1:].view(batch, 1680)
    xv.copy_(torch.from_numpy(x)), gv.copy_(torch.from_numpy(gy))
    assert xv.data_ptr() % 16 and gv.data_ptr() % 16
    got = _backward(tw, xv, gv)
    _check(x, w, gy, got, "misaligned x and grad_y")
    fast = _backward(tw, torch.from_numpy(x).cuda(), torch.from_numpy(gy).cuda())
    for a, b in zip(got, fast):
        assert torch.equal(a, b)
    only_x = _backward(tw, xv, torch.from_numpy(gy).cuda())   # aligned grad_y, misaligned x: generic weight gradient only
    for a, b in zip(only_x, fast):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("x_grad", [False, True])
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_autograd(x_grad, mode):
    m = _model(seed=3)
    m.trainable = True
    m.train(mode == "train")
    batch = 4099
    rng = np.random.default_rng(17)
    x = torch.from_numpy(rng.standard_normal((batch, 12, 2)).astype(np.float32)).cuda().requires_grad_(x_grad)
    g = torch.from_numpy(rng.standard_normal((batch, 120, 14)).astype(np.float32)).cuda()
    y = m(x)
    assert y.grad_fn is not None and y.dtype == torch.float32
    with torch.no_grad():
        assert torch.equal(y, m(x)), "trainable forward differs from the no_grad forward"
    (y * g).sum().backward()
    xs, ws, gs = x.detach().reshape(batch, 24).cpu().numpy(), m.linear.weight.detach().cpu().numpy(), g.reshape(batch, 1680).cpu().numpy()
    got = (m.linear.weight.grad, m.linear.bias.grad, x.grad.reshape(batch, 24) if x_grad else None)
    assert (x.grad is not None) == x_grad
    _check(xs, ws, gs, got, f"autograd {mode}, x_grad={x_grad}")
    first = [t.clone() for t in got if t is not None]
    m.zero_grad(set_to_none=True)
    x.grad = None
    (m(x) * g).sum().backward()
    again = (m.linear.weight.grad, m.linear.bias.grad, x.grad.reshape(batch, 24) if x_grad else None)
    for a, b in zip(first, [t for t in again if t is not None]):
        assert torch.equal(a, b), "repeated backward is not bit-identical"


@pytest.mark.gpu
def test_autograd_edges():
    m = _model(seed=4)
    # untrainable: unchanged behaviour
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m(torch.zeros(2, 12, 2, device="cuda"))
    m.eval()
    assert m(torch.zeros(2, 12, 2, device="cuda")).grad_fn is None
    with pytest.raises(RuntimeError, match="complex"):
        m(torch.zeros(2, 12, 2, dtype=torch.cfloat, device="cuda"))
    m.trainable = True
    with pytest.raises(RuntimeError, match="complex"):
        m(torch.zeros(2, 12, 2, dtype=torch.cfloat, device="cuda"))
    # empty batch: zero gradients
    m.train()
    x = torch.zeros(0, 12, 2, device="cuda", requires_grad=True)
    y = m(x)
    assert tuple(y.shape) == (0, 120, 14)
    y.sum().backward()
    assert torch.equal(m.linear.weight.grad, torch.zeros_like(m.linear.weight))
    assert torch.equal(m.linear.bias.grad, torch.zeros_like(m.linear.bias)) and tuple(x.grad.shape) == (0, 12, 2)
    # float64 model and input (CPU input too): gradients in float64, on the input's device
    m64 = _model(torch.float64, seed=5)
    m64.trainable = True
    rng = np.random.default_rng(23)
    x64 = torch.from_numpy(rng.standard_normal((257, 12, 2))).requires_grad_(True)
    g = torch.from_numpy(rng.standard_normal((257, 120, 14)).astype(np.float32)).cuda()
    (m64(x64) * g).sum().backward()
    assert m64.linear.weight.grad.dtype == torch.float64 and m64.linear.bias.grad.dtype == torch.float64
    assert x64.grad.dtype == torch.float64 and x64.grad.device.type == "cpu"
    # the kernel computes on the fp32 roundings of the operands: the fp64 restatement uses the same
    xs = x64.detach().reshape(257, 24).float().numpy()
    ws = m64.linear.weight.detach().float().cpu().numpy()
    _check(xs, ws, g.reshape(257, 1680).cpu().numpy(),
           (m64.linear.weight.grad, m64.linear.bias.grad, x64.grad.reshape(257, 24)), "float64 model")


@pytest.mark.gpu
def test_sgd_trajectory():
    """Five SGD steps on fixed batches with the MSE loss: ours (fp32 kernels), the same steps in fp64, and stock fp32
    (torch CPU nn.Linear).  theta_5 - theta_0 of ours must be within the gate of the fp64 update; the loss decreases."""
    steps, batch, lr = 5, 512, 200.0   # the MSE mean over 1680 outputs scales the gradient by 2 / 1680
    rng = np.random.default_rng(29)
    w_true = rng.standard_normal((1680, 24)) / np.sqrt(24)
    data = []
    for _ in range(steps):
        x = rng.standard_normal((batch, 24)).astype(np.float32)
        t = (x @ w_true.T + 0.1 * rng.standard_normal((batch, 1680))).astype(np.float32)
        data.append((x, t))
    m = _model(seed=6)
    m.trainable = True
    m.train()
    w0, b0 = m.linear.weight.detach().cpu().numpy().copy(), m.linear.bias.detach().cpu().numpy().copy()
    opt = torch.optim.SGD(m.parameters(), lr=lr)
    losses = []
    for x, t in data:
        opt.zero_grad()
        loss = torch.nn.functional.mse_loss(m(torch.from_numpy(x).cuda().reshape(batch, 12, 2)),
                                            torch.from_numpy(t).cuda().reshape(batch, 120, 14))
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(b < a for a, b in zip(losses, losses[1:])), losses

    def run(dtype):
        lin = torch.nn.Linear(24, 1680).to(dtype)
        with torch.no_grad():
            lin.weight.copy_(torch.from_numpy(w0)), lin.bias.copy_(torch.from_numpy(b0))
        o = torch.optim.SGD(lin.parameters(), lr=lr)
        for x, t in data:
            o.zero_grad()
            torch.nn.functional.mse_loss(lin(torch.from_numpy(x).to(dtype)), torch.from_numpy(t).to(dtype)).backward()
            o.step()
        return lin.weight.detach().double().numpy(), lin.bias.detach().double().numpy()

    (w64, b64), (w32, b32) = run(torch.float64), run(torch.float32)
    ours = np.concatenate([(m.linear.weight.detach().double().cpu().numpy() - w0).ravel(),
                           (m.linear.bias.detach().double().cpu().numpy() - b0).ravel()])
    ref = np.concatenate([(w64 - w0).ravel(), (b64 - b0).ravel()])
    stock = np.concatenate([(w32 - w0).ravel(), (b32 - b0).ravel()])
    assert _nw(ours, ref) <= _gate(_nw(stock, ref)), (_nw(ours, ref), _nw(stock, ref))
