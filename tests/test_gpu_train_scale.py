"""GPU: the fp32 training path at the batch sizes where the backward's deterministic chunked sums change shape.

``train_bwd.cu`` sums every weight / bias gradient as per-chunk partials (at most ``kMaxChunks = 128``, ``train.cuh``)
added in a fixed order (``k_reduce``).  How the rows are split depends on the batch B (``nseq = 2B`` sequences,
``M = 280 * nseq`` token rows), through three formulas:

* ``Ctx::wgrad_gemm`` (the GEMM weight gradients): rows per chunk ``ceil(M / 128)`` rounded up to 16, at least 512;
* ``Ctx::wgrad_rows`` over the M token rows (biases, LayerNorm, linear_1 / linear_2): ``ceil(M / 128)`` rows per chunk;
* ``Ctx::wgrad_rows`` / ``Ctx::conv_stack`` over the sequences (positional table, adapter MLP, up-sampler, both conv
  stacks): ``ceil(nseq / 128)`` sequences per chunk.

=====  ==============================  ==============================  ===========================================
batch  wgrad_gemm rows/chunk, chunks,  wgrad_rows over M: rows/chunk,  per-sequence sums: sequences/chunk, chunks,
       last chunk                      chunks, last chunk              last chunk
=====  ==============================  ==============================  ===========================================
2-5    512, 3-6, 96-240                9-22, 120-128, 4-14             1, 4-10, 1  (tests/test_gpu_train.py)
1      512, 2, 48                      5, 112, 5                       1, 2, 1
65     512, 72, 48                     285, 128, 205                   2, 65, 2
118    528 (first above 512), 126, 80  517, 128, 421                   2, 118, 2
130    576, 127, 224                   569, 128, 537                   3, 87, 2 (ragged)
257    1136, 127, 784                  1125, 128, 1045                 5, 103, 4 (ragged)
=====  ==============================  ==============================  ===========================================

Batches 1, 65 and 257 (AdaFortiTran, trained weights) and 130 (FortiTran: no adapter, a ragged last sequence chunk)
cover chunks of more than one sequence, ragged last chunks, GEMM chunks above 512 rows and the single-sample batch.
The dropout case runs at batch 257 with the loss gradient nonzero only at samples 0, 1, 128, 129 and 256 -- sample 129's
imaginary sequence straddles a 1136-row ``wgrad_gemm`` chunk boundary, sample 256 puts the Philox ``seq`` counter at
512 and 513 -- and is compared with fp64 restatements of just those samples (the other samples contribute exactly zero).

The fp64 restatement of ``oracle/train_ref.py`` runs on the GPU, 16 samples at a time: for ``loss = <g, out>`` the
gradient is a sum over samples, accumulated over the chunks in fp64 (the reference) or in fp32 (the stock fp32 autograd
arm that sets the bar of ``_gate``).  TF32 is off for the whole module, so that arm is true fp32.

Compared samples are kept clear of ReLU kinks (``_away_from_kinks``).  Where the fp64 restatement feeds a ReLU (conv
stacks, adapter MLP) a value within about 1e-6 of its rms from zero, fp32 rounding decides relu' for any fp32
implementation, and the branch taken moves the gradients of everything upstream of that element by 1e-4 to 1e-3.  With
the unmodified draw of seed 357 at batch 257, 31 samples hold such an element, and the gate failed by chance: refiner
and encoder gradients 1.0e-4 to 2.7e-4 against the stock arm's 4e-8 to 3e-6.  The cause was sample 48 alone, whose
input to the last ReLU of the final refiner comes within 1.1e-7 of that input's rms from zero: these kernels took the
other branch than fp64 there (88 tensors off by up to 1.1e-3 with only that sample's loss gradient nonzero), the stock
arm did not.  With the near-kink samples redrawn, every tensor passes."""
import ctypes as C
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch.overrides import TorchFunctionMode

from adafortitran_b200 import _capi
from oracle import train_ref as T
from tests import util
from tests.test_gpu_train import TOL, _case_model, _check_grads, _inputs, _nw, _run_ours, _seed_of

pytestmark = pytest.mark.gpu
DEV = "cuda"
REF_CHUNK = 16   # samples per restatement call
KINK = 1e-6      # smallest |ReLU input| / rms(ReLU input) a compared sample may have in the fp64 restatement


@pytest.fixture(scope="module", autouse=True)
def fp32_without_tf32():
    """F.conv2d defaults to TF32 through cuDNN; the stock fp32 arm must not use it, or its error -- the gate's bar --
    is loose.  Also reports the module's wall time and peak device memory."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved
    print(f"\n{__name__}: wall time {time.perf_counter() - t0:.1f} s, peak device memory "
          f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB ({torch.cuda.get_device_name()})")


def _gemm_rows(batch):
    """Rows per chunk of ``Ctx::wgrad_gemm`` (train_bwd.cu) over the batch's token rows."""
    rows = -(-280 * 2 * batch // 128)
    return max(-(-rows // 16) * 16, 512)


def _ref_on_gpu(model, pilots, cond, g, dtype, p=0.0, masks=None):
    """The restatement in ``dtype`` on the GPU, REF_CHUNK samples at a time, for loss = <g, out>.  Returns the output
    (numpy complex) and {name: gradient (float64 numpy)} summed over the chunks in ``dtype``.  ``masks``: the
    ``[real, imaginary]`` pair of ``masks[layer][site]`` arrays over the same samples as ``pilots``."""
    named, _ = model._weight_tensors()
    P = {n: t.detach().to(DEV, dtype).clone().requires_grad_(True) for n, t in named}
    acc = {n: torch.zeros_like(t) for n, t in P.items()}
    ctype = torch.complex128 if dtype == torch.float64 else torch.complex64
    mc = model.model_config
    outs = []
    for s in range(0, len(pilots), REF_CHUNK):
        e = min(s + REF_CHUNK, len(pilots))
        c = None
        if model.use_channel_adaptation:
            c = [torch.from_numpy(np.asarray(v[s:e], np.float64)).to(DEV) for v in cond]
        mk = None if masks is None else [[[site[s:e].to(DEV) for site in layer] for layer in part] for part in masks]
        out = T.forward(P, torch.from_numpy(pilots[s:e]).to(DEV, ctype), c, p, None, mc.num_layers, mc.activation,
                        masks=mk)
        gt = torch.from_numpy(g[s:e]).to(DEV, ctype)
        grads = torch.autograd.grad((out.real * gt.real + out.imag * gt.imag).sum(), list(P.values()))
        for a, gr in zip(acc.values(), grads):
            a += gr
        outs.append(out.detach().cpu().numpy())
    return np.concatenate(outs), {n: a.double().cpu().numpy() for n, a in acc.items()}


class _ReluMargins(TorchFunctionMode):
    """Per sample, the smallest |x| / rms(x) over the inputs x of every F.relu the restatement calls."""

    def __init__(self, n):
        super().__init__()
        self.margin = torch.full((n,), float("inf"), dtype=torch.float64, device=DEV)

    def __torch_function__(self, func, types, args=(), kwargs=None):
        if func is F.relu:
            x = args[0].detach()
            r = (x.abs() / x.pow(2).mean().sqrt()).reshape(x.shape[0], -1).amin(1)
            self.margin = torch.minimum(self.margin, r)
        return func(*args, **(kwargs or {}))


def _away_from_kinks(model, pilots, cond, p=0.0, masks=None):
    """Redraws, in place, the pilots of every sample whose fp64 restatement feeds a ReLU a value within KINK (relative
    to the rms of that ReLU's input) of zero, until none does; returns how many were redrawn.

    At such an element relu' is decided by fp32 rounding: the stock fp32 arm deviates from fp64 by up to ~1e-6 of the
    rms there, so either fp32 implementation may take the other branch, and one flipped element moves the gradients
    of everything upstream of it by 1e-4 to 1e-3.  Which implementation flips is chance, so the gate against the stock
    arm is only meaningful on samples that stay clear of the kinks."""
    named, _ = model._weight_tensors()
    P = {k: t.detach().to(DEV, torch.float64) for k, t in named}
    mc = model.model_config
    c = [torch.from_numpy(np.asarray(v, np.float64)).to(DEV) for v in cond] if model.use_channel_adaptation else None
    mk = None if masks is None else [[[site.to(DEV) for site in layer] for layer in part] for part in masks]
    rng = np.random.default_rng(len(pilots))
    redrawn = 0
    for _ in range(20):
        with torch.no_grad(), _ReluMargins(len(pilots)) as rec:
            T.forward(P, torch.from_numpy(pilots).to(DEV, torch.complex128), c, p, None, mc.num_layers, mc.activation,
                      masks=mk)
        bad = np.nonzero(rec.margin.cpu().numpy() < KINK)[0]
        if not len(bad):
            return redrawn
        shape = (len(bad),) + pilots.shape[1:]
        pilots[bad] = ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)).astype(pilots.dtype)
        redrawn += len(bad)
    raise AssertionError(f"samples {bad} still within {KINK} of a ReLU kink after 20 redraws")


def _clear_inputs(model, n, seed):
    """_inputs(n, seed) with the pilots near ReLU kinks redrawn (see _away_from_kinks)."""
    pilots, cond, g = _inputs(n, seed=seed)
    redrawn = _away_from_kinks(model, pilots, cond)
    print(f"batch {n}: {redrawn} pilot draws replaced to keep clear of ReLU kinks")
    return pilots, cond, g


@pytest.fixture(scope="module")
def ada_ref():
    """ada_trained inputs and the fp64 / stock fp32 restatements of <g, out> at batch n, computed once per n."""
    cache = {}

    def get(n):
        if n not in cache:
            model, _ = _case_model("ada_trained")
            pilots, cond, g = _clear_inputs(model, n, seed=100 + n)
            cache[n] = (pilots, cond, g, _ref_on_gpu(model, pilots, cond, g, torch.float64),
                        _ref_on_gpu(model, pilots, cond, g, torch.float32)[1])
        return cache[n]
    return get


@pytest.mark.parametrize("n", [1, 65, 257])
def test_dense_gradients_across_chunk_plans(n, ada_ref):
    pilots, cond, g, (ref_out, ref), stock = ada_ref(n)
    model, _ = _case_model("ada_trained")
    out, ours = _run_ours(model, pilots, cond, g=g)
    e = _nw(out.view(np.float32), ref_out.view(np.float64))
    print(f"batch {n}: output {e:.2e}")
    assert e <= TOL
    _check_grads(ours, ref, stock, f"ada_trained batch {n} <g, out>")


def test_fortitran_ragged_sequence_chunk():
    """Batch 130: three sequences per chunk of the per-sequence sums and a last chunk of two; FortiTran has no adapter
    (in_dim 6)."""
    model, _ = _case_model("forti_seed0")
    pilots, cond, g = _clear_inputs(model, 130, seed=230)
    out, ours = _run_ours(model, pilots, cond, g=g)
    ref_out, ref = _ref_on_gpu(model, pilots, cond, g, torch.float64)
    _, stock = _ref_on_gpu(model, pilots, cond, g, torch.float32)
    e = _nw(out.view(np.float32), ref_out.view(np.float64))
    print(f"forti batch 130: output {e:.2e}")
    assert e <= TOL
    _check_grads(ours, ref, stock, "forti_seed0 batch 130 <g, out>")


def test_dropout_at_high_sequence_indices():
    """Batch 257, p = 0.1: the loss gradient is zero except at a few samples, so the gradients are those samples'
    contributions alone, with masks at sequence indices up to 513 (forward attention, LayerNorm and activation sites,
    and the quad-shared key-row pass of attn_bwd_kernel)."""
    n, p, torch_seed = 257, 0.1, 123
    model, _ = _case_model("ada_trained")
    assert model.model_config.dropout == p
    model.train()
    rows = _gemm_rows(n)
    straddle = next(b for b in range(129, n) if (560 * b) // rows != (560 * b + 559) // rows)
    picked = [0, 1, 128, straddle, n - 1]
    pilots, cond, g = _inputs(n, seed=257)
    keep = np.zeros(n, bool)
    keep[picked] = True
    g[~keep] = 0
    seed = _seed_of(torch_seed)
    masks = [[[torch.from_numpy(np.stack([T.keep_mask(seed, 2 * b + part, l, s, T.SITE_SHAPES[s], p) for b in picked])
                                .astype(np.float64)) for s in range(4)] for l in range(6)] for part in (0, 1)]
    sub = lambda a: a[picked]
    cond_p = [sub(c) for c in cond]
    pil_p = sub(pilots)
    print(f"{_away_from_kinks(model, pil_p, cond_p, p, masks)} pilot draws replaced to keep clear of ReLU kinks")
    pilots[picked] = pil_p
    out, ours = _run_ours(model, pilots, cond, g=g, torch_seed=torch_seed)
    ref_out, ref = _ref_on_gpu(model, pil_p, cond_p, sub(g), torch.float64, p=p, masks=masks)
    _, stock = _ref_on_gpu(model, pil_p, cond_p, sub(g), torch.float32, p=p, masks=masks)
    e = _nw(sub(out).view(np.float32), ref_out.view(np.float64))
    print(f"dropout {p} at samples {picked}: output {e:.2e}")
    assert e <= TOL
    _check_grads(ours, ref, stock, f"dropout {p} batch {n}, samples {picked}")


def test_same_seed_bit_identical_at_scale():
    model, _ = _case_model("ada_trained")
    model.train()
    pilots, cond, g = _inputs(257, seed=7)
    o1, g1 = _run_ours(model, pilots, cond, g=g, torch_seed=7)
    o2, g2 = _run_ours(model, pilots, cond, g=g, torch_seed=7)
    assert np.array_equal(o1, o2)
    for n in g1:
        assert np.array_equal(g1[n], g2[n]), n
    o3, _ = _run_ours(model, pilots, cond, g=g, torch_seed=8)
    assert not np.array_equal(o1, o3)


def test_training_forward_p0_bit_identical_to_inference_at_scale():
    model, _ = _case_model("ada_trained")
    pilots, cond, _ = _inputs(257, seed=8)
    md = util.meta(*cond)
    with torch.no_grad():
        inf = model(torch.from_numpy(pilots), md).cpu().numpy()
    tr = model(torch.from_numpy(pilots), md)    # eval + grad enabled: the training forward with p = 0
    assert tr.requires_grad
    assert np.array_equal(tr.detach().cpu().numpy(), inf)


def test_microbatch_accumulation(ada_ref):
    """Batch 65 as 33 + 32 with two backward() calls and no zero_grad in between: AccumulateGrad adds the second
    call's gradients (views of its flat buffer) to the first's."""
    pilots, cond, g, (_, ref), stock = ada_ref(65)
    model, _ = _case_model("ada_trained")
    model.zero_grad(set_to_none=True)
    for s, e in ((0, 33), (33, 65)):
        out = model(torch.from_numpy(pilots[s:e]), util.meta(*(c[s:e] for c in cond)))
        gt = torch.from_numpy(g[s:e]).to(out.device)
        (out.real * gt.real.float() + out.imag * gt.imag.float()).sum().backward()
    named, _ = model._weight_tensors()
    ours = {n: t.grad.detach().cpu().numpy() for n, t in named}
    _check_grads(ours, ref, stock, "ada_trained batch 65 as 33 + 32 micro-batches")


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _filled_workspace(model, n):
    """Runs aft_forward_train (p = 0) on the model's handle at batch n; returns (workspace, aligned pointer, bytes)."""
    pilots, cond, _ = _inputs(n, seed=16)
    md = util.meta(*cond) if model.use_channel_adaptation else None
    with torch.no_grad():
        model(torch.from_numpy(pilots), md)      # creates the handle, loads the weights
    lib = _capi.lib()
    need = lib.aft_train_workspace_bytes(model._handle, n)
    ws = torch.empty(need + 256, dtype=torch.uint8, device=DEV)
    ptr = (ws.data_ptr() + 255) // 256 * 256
    pil = torch.from_numpy(pilots).to(DEV)
    cd = [torch.from_numpy(c).to(DEV) for c in cond] if model.use_channel_adaptation else [None] * 3
    out = torch.empty((n, 120, 14), dtype=torch.complex64, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _capi.check(lib.aft_forward_train(model._handle, _vp(pil), _vp(cd[0]), _vp(cd[1]), _vp(cd[2]), _vp(out), n, 0.0, 1,
                                      C.c_void_p(ptr), need, st))
    torch.cuda.synchronize()
    return ws, ptr, need


def test_backward_rejects_workspace_of_another_call():
    """aft_backward refuses, with AFT_ERR_INVALID and nothing launched: a batch other than the forward's, a workspace
    filled by an estimator with another layer count, and a workspace no forward filled."""
    lib = _capi.lib()
    six, _ = _case_model("ada_trained")
    two, _ = _case_model("layers2")
    ws6, p6, need6 = _filled_workspace(six, 2)
    ws2, p2, need2 = _filled_workspace(two, 2)
    grads = torch.zeros(lib.aft_param_count(six._handle), dtype=torch.float32, device=DEV)
    g = torch.ones((3, 120, 14, 2), dtype=torch.float32, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rejected(batch, ptr, nbytes, what):
        n0 = lib.aft_launch_count()
        rc = lib.aft_backward(six._handle, _vp(g), batch, C.c_void_p(ptr), nbytes, _vp(grads), st)
        assert rc == _capi.AFT_ERR_INVALID and what in lib.aft_last_error(), (rc, lib.aft_last_error())
        assert lib.aft_launch_count() == n0

    rejected(3, p6, need6, b"differs")
    rejected(1, p6, need6, b"differs")
    rejected(2, p2, need2, b"not filled")
    zeroed = torch.zeros(need6 + 256, dtype=torch.uint8, device=DEV)
    rejected(2, (zeroed.data_ptr() + 255) // 256 * 256, need6, b"not filled")
    assert not grads.any()
    n0 = lib.aft_launch_count()          # the workspace the rejected calls saw is still good for its own batch
    _capi.check(lib.aft_backward(six._handle, _vp(g), 2, C.c_void_p(p6), need6, _vp(grads), st))
    torch.cuda.synchronize()
    assert lib.aft_launch_count() > n0 and grads.any() and torch.isfinite(grads).all()


def test_empty_differentiable_batch():
    model, _ = _case_model("ada_trained")
    model.zero_grad(set_to_none=True)
    out = model(torch.zeros(0, 12, 2, dtype=torch.complex64), util.meta([], [], []))
    assert out.shape == (0, 120, 14) and out.requires_grad
    out.abs().pow(2).sum().backward()
    named, _ = model._weight_tensors()
    for n, t in named:
        assert t.grad is not None and t.grad.shape == t.shape and not t.grad.any(), n
