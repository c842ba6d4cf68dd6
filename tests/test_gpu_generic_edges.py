"""GPU: the shape-generic paths (grids other than the reference default 120 x 14 / pilots 12 x 2 / patch 3 x 2) at their
tile, key-tile, persistent-loop and chunk edges, against the fp64 oracle, per sample.

AFT_FP32 runs ``csrc/generic_f32.cu`` (up-sampler, conv stacks, tokens + ``linear_1``, head; ``g_attention`` with
128-query blocks over 64-key tiles) and the shape-generic GEMMs of ``gemm_f32.cu``.  AFT_BF16 runs the same front end and
head around ``csrc/tc_long.cu``: ``lin_block_kernel`` (one persistent CTA per 128-row tile, ``min(2 B T, SMs)`` CTAs)
and ``attn_long_kernel`` (64-key tiles through a 4-stage ring, padding keys masked).  ``aft_api.cu`` splits a batch
into internal chunks sized from the workspace (``generic_chunk``) and, in ``aft_forward_host``, into host chunks on two
lanes.

Per geometry: T 128-row tiles, nkt 64-key tiles, the valid keys of the last key tile, the composition batch B
(``SMs // T + 12``, so ``2 B T`` row tiles exceed twice the SM count) with its row tiles and tiles per
``lin_block_kernel`` CTA on a 148-SM B200, and the internal chunk (samples) of each precision.  The chunk figures are
computed from ``generic_floats_per_chunk``; the chunk test finds them on the device by bisection.

======  =====  ====  ===  ==============  ===  ==========  ========  ===================  ==================================
id      S      T     nkt  last-tile keys  B    row tiles   per CTA   chunk fp32 / bf16    edge
======  =====  ====  ===  ==============  ===  ==========  ========  ===================  ==================================
S1      1      1     1    1               160  320         2-3       1024 / 1024          one token, 127 padding query rows,
                                                                                          one layer (qkv-only launch, then
                                                                                          the last-layer launch)
S64     64     1     1    64              160  320         2-3       1024 / 1024          exactly one full key tile
S65     65     1     2    1               160  320         2-3       1024 / 1024          Ada; W = 1, patch 1 x 1, odd pix
S128    128    1     2    64              160  320         2-3       1024 / 1024          exact row tile
S129    129    2     3    1               86   344         2-3       1024 / 1024          sinusoidal table at odd S
S192    192    2     3    64              86   344         2-3       961 / 1024           Ada; key tile 1 = second half of
                                                                                          row tile 0
S257    257    3     5    1               61   366         2-3       643 / 1024           3 layers, ring wraps once
S258    258    3     5    2               61   366         2-3       579 / 1024           up-sampler on the tiled GEMM
                                                                                          (P pix = 1,198,152, K 774, N 1548)
P64     16     1     1    16              160  320         2-3       1024 / 1024          8 x 8 patch: linear_2 fold of 64
S1025   1025   9     17   1               28   504         3-4       180 / 683            ring wraps four times
======  =====  ====  ===  ==============  ===  ==========  ========  ===================  ==================================

The internal chunk and host-lane checks run at S65 and S1025: ``chunk + 37`` samples (two internal chunks, the second
ragged) and ``2 hc + 37`` samples through ``aft_forward_host`` with ``hc = min(2048, chunk)`` (both lanes used twice,
ragged last host chunk; the generic path does not taper).

Exactness: every kernel of both paths computes a row, tile or (sequence, head, query tile) in an order that does not
depend on where it sits in the batch, so a repeat, a permuted batch, each sample run alone and the two halves of a
chunked batch are bit-identical to the corresponding rows of the batch.  Ids S = 64 k + 1 leave one valid key in the
last key tile: a missing or shifted padding mask adds up to 63 bogus keys to 64 k + 1 real ones.

Gates apply to each sample: fp32 <= 1e-5 normwise (ten times tighter than the project's 1e-4, see ``FP32_GATE``); bf16
output-relative error power <= -40 dB (FortiTran) / -34 dB (AdaFortiTran, random init: the raw metadata dominates the
token features, DESIGN.md 5), against the oracle and against the fp32 path.  The bf16 gates cannot see a padding mask
that is off by one key at S >= 65 (the extra key moves the output by -49 to -82 dB), nor a removed mask at S65 and
S1025 (-47 / -46 dB); a removed mask is caught at S1, S129, S257, S258 and P64, an off-by-one mask at S1 and P64.
``tests/test_gpu_long_stages.py`` closes that gap: it checks each ``tc_long.cu`` kernel alone against fp64, with
constructed weights under which the padding mask, the last key, the key ring and the rescale decide the result.  The Ada rows draw their metadata from the lower part of the reference's
condition grid (SNR 0-30 dB, delay spread 50-200 ns, Doppler 200-600 Hz).
"""
import time

import numpy as np
import pytest
import torch

from adafortitran_b200 import _capi
from oracle import aft_oracle as O
from tests import util

pytestmark = pytest.mark.gpu

# id: (kind, layers, activation, positional table, grid, pilots, patch)
GEOMS = {
    "S1": ("forti", 1, "relu", "learnable", (3, 2), (1, 1), (3, 2)),
    "S64": ("forti", 2, "gelu", "learnable", (128, 4), (16, 2), (2, 4)),
    "S65": ("ada", 2, "gelu", "learnable", (65, 1), (13, 1), (1, 1)),
    "S128": ("forti", 2, "gelu", "learnable", (256, 4), (32, 2), (4, 2)),
    "S129": ("forti", 2, "gelu", "sinusoidal", (129, 2), (43, 2), (1, 2)),
    "S192": ("ada", 2, "gelu", "learnable", (96, 4), (24, 2), (1, 2)),
    "S257": ("forti", 3, "relu", "learnable", (514, 2), (257, 1), (2, 2)),
    "S258": ("forti", 2, "gelu", "learnable", (258, 6), (129, 6), (3, 2)),
    "P64": ("forti", 2, "gelu", "learnable", (64, 16), (16, 4), (8, 8)),
    "S1025": ("forti", 2, "gelu", "learnable", (205, 10), (41, 5), (1, 2)),
}
PRECS = {"fp32": _capi.AFT_FP32, "bf16": _capi.AFT_BF16}
# Tighter than the project's 1e-4: every sample here measures <= 1.5e-6 (deterministic inputs and kernels), while
# g_attention skipping the one valid key of the last key tile moves S257 / S1025 by only 5.6e-5 / 2.0e-5 (fp64
# restatement of that fault on these samples), which 1e-4 lets through.
FP32_GATE = 1e-5
BF16_GATE_DB = {"forti": -40.0, "ada": -34.0}
RESULTS = {}   # (id, precision) -> worst per-sample figures, printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def report():
    """Wall time, peak device memory (torch's allocator and, sampled after each test, the whole device) and the worst
    per-sample figures of every case."""
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    print(f"\n{__name__}: wall time {time.perf_counter() - t0:.1f} s, peak torch allocation "
          f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB, peak device memory in use {_DEVICE_PEAK[0] / 1e9:.2f} GB "
          f"({torch.cuda.get_device_name()}, {torch.cuda.get_device_properties(0).multi_processor_count} SMs)")
    for (gid, prec), r in sorted(RESULTS.items()):
        print(f"  {gid:6s} {prec}: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(r.items())))


_DEVICE_PEAK = [0]


@pytest.fixture(autouse=True)
def _sample_device_memory():
    yield
    free, total = torch.cuda.mem_get_info()
    _DEVICE_PEAK[0] = max(_DEVICE_PEAK[0], total - free)


def _record(gid, prec, key, value, worse=max):
    r = RESULTS.setdefault((gid, prec), {})
    r[key] = worse(r[key], value) if key in r else value


class Case:
    """One geometry: the model (seeded initialisation), the composition batch and the fp64 oracle on chosen samples."""

    def __init__(self, gid):
        from adafortitran_b200 import AdaFortiTranEstimator, FortiTranEstimator, ModelConfig, SystemConfig
        kind, layers, act, pos, grid, pilots, patch = GEOMS[gid]
        self.gid, self.kind, self.pilots = gid, kind, pilots
        self.S = (grid[0] // patch[0]) * (grid[1] // patch[1])
        self.T = -(-self.S // 128)
        ada = kind == "ada"
        extra = dict(channel_adaptivity_hidden_sizes=[7, 42, 2 * self.S], adaptive_token_length=6) if ada else {}
        torch.manual_seed(list(GEOMS).index(gid))
        cls = AdaFortiTranEstimator if ada else FortiTranEstimator
        self.model = cls(SystemConfig(ofdm=dict(num_scs=grid[0], num_symbols=grid[1]), pilot=dict(num_scs=pilots[0], num_symbols=pilots[1])),
                         ModelConfig(model_type="adafortitran" if ada else "fortitran", patch_size=patch, num_layers=layers, model_dim=128,
                                     num_head=4, activation=act, max_seq_len=max(self.S, 8), pos_encoding_type=pos, device="cuda",
                                     **extra)).eval()
        self.sd = {k: v.detach().cpu().numpy() for k, v in self.model.state_dict().items()}
        self.cfg = O.OracleConfig(num_scs=grid[0], num_symbols=grid[1], pilot_scs=pilots[0], pilot_symbols=pilots[1], patch=patch,
                                  num_layers=layers, activation=act, adaptive=ada)
        self.sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        # composition batch: 2 B T row tiles > 2 x SMs, so every lin_block_kernel CTA runs at least two tiles
        self.B = self.sm // self.T + 12
        self.x, self.md = self.inputs(self.B, seed=100 + list(GEOMS).index(gid))
        # a sample whose sequences lie on the CTAs' second persistent iteration (row tiles SMs .. 2 SMs - 1); the last
        # sample lies on the third
        self.second = (self.sm + self.sm // 2) // (2 * self.T)
        assert self.sm <= 2 * self.second * self.T and 2 * (self.second + 1) * self.T <= 2 * self.sm
        B = self.B
        self.idx = sorted({0, 1, B // 4, self.second, B // 2, 3 * B // 4, B - 2, B - 1}) if self.S < 1000 else [0, self.second, B // 2, B - 1]
        self.ref = self.oracle(self.idx)
        self.y32 = self.run("fp32", self.x, self.md)

    def inputs(self, n, seed):
        rng = np.random.default_rng(seed)
        shape = (n, *self.pilots)
        x = ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)).astype(np.complex64)
        if self.kind != "ada":
            return x, None
        md = (rng.choice(O.SNR_GRID, n), rng.choice(O.DS_GRID[:4], n), rng.choice(O.DOP_GRID[:3], n))
        return x, tuple(a.astype(np.float32) for a in md)

    def oracle(self, idx, x=None, md=None):
        x, md = (self.x, self.md) if x is None else (x, md)
        return O.forward(self.cfg, self.sd, x[idx], *(a[idx] for a in md or ()))

    def run(self, prec, x, md):
        self.model.precision = prec
        with torch.no_grad():
            return self.model(torch.from_numpy(x), util.meta(*md) if md is not None else None).cpu().numpy()

    def run_host(self, prec, x, md):
        self.model.precision = prec
        with torch.no_grad():
            return self.model.forward_host(torch.from_numpy(x), util.meta(*md) if md is not None else None).numpy()


@pytest.fixture(scope="module")
def case(request):
    c = Case(request.param)
    yield c
    c.model._release()


def _check_samples(c, prec, y, ref, what):
    """Per-sample gate against the fp64 oracle; returns the worst figure."""
    assert np.isfinite(y.view(np.float32)).all()
    if prec == "fp32":
        errs = [O.normwise_err(y[i], ref[i]) for i in range(len(ref))]
        worst = max(errs)
        _record(c.gid, prec, what, worst)
        assert worst <= FP32_GATE, (what, errs)
    else:
        errs = [O.rel_err_db(y[i], ref[i]) for i in range(len(ref))]
        worst = max(errs)
        _record(c.gid, prec, what, worst)
        assert worst <= BF16_GATE_DB[c.kind], (what, errs)
    return worst


@pytest.mark.parametrize("prec", list(PRECS))
@pytest.mark.parametrize("case", list(GEOMS), indirect=True)
def test_oracle_parity_per_sample(case, prec):
    """Samples 0, 1, B-2, B-1, one on the second persistent iteration and three in between, each against the fp64 oracle;
    the bf16 path also against the fp32 path, every sample of the batch."""
    c = case
    y = c.y32 if prec == "fp32" else c.run(prec, c.x, c.md)
    assert y.shape == (c.B, *GEOMS[c.gid][4])
    _check_samples(c, prec, y[c.idx], c.ref, "vs_oracle")
    if prec == "bf16":
        worst = max(O.rel_err_db(y[i], c.y32[i]) for i in range(c.B))
        _record(c.gid, prec, "vs_fp32_db", worst)
        assert worst <= BF16_GATE_DB[c.kind], worst


@pytest.mark.parametrize("prec", list(PRECS))
@pytest.mark.parametrize("case", list(GEOMS), indirect=True)
def test_batch_composition_is_exact(case, prec):
    """Bit-identity: a repeat, a permuted batch, the first / second-iteration / last sample run alone, and the real part
    of the output with the imaginary pilots shifted across samples."""
    c = case
    assert 2 * c.B * c.T > 2 * c.sm
    y = c.y32 if prec == "fp32" else c.run(prec, c.x, c.md)
    assert np.array_equal(c.run(prec, c.x, c.md), y), "repeat"
    perm = np.random.default_rng(7).permutation(c.B)
    assert np.array_equal(c.run(prec, c.x[perm], None if c.md is None else tuple(a[perm] for a in c.md)), y[perm]), "permutation"
    for i in (0, c.second, c.B - 1):
        sl = slice(i, i + 1)
        assert np.array_equal(c.run(prec, c.x[sl], None if c.md is None else tuple(a[sl] for a in c.md)), y[sl]), f"sample {i} alone"
    x2 = (c.x.real + 1j * np.roll(c.x.imag, 1, axis=0)).astype(np.complex64)
    assert np.array_equal(c.run(prec, x2, c.md).real, y.real), "re/im independence"


@pytest.mark.parametrize("prec", list(PRECS))
@pytest.mark.parametrize("case", ["S65", "S1025"], indirect=True)
def test_internal_chunk_and_host_lanes(case, prec):
    """The internal chunk, found where ``aft_workspace_bytes`` stops growing with the batch: ``chunk + 37`` samples equal
    the two parts run separately, bit for bit, and the samples either side of the boundary pass the oracle gate.
    ``aft_forward_host`` over ``2 hc + 37`` samples equals the device forward at the same batch, bit for bit."""
    c = case
    code = PRECS[prec]
    c.model._ensure_handle()
    lib = _capi.lib()
    ws = lambda b: lib.aft_workspace_bytes(c.model._handle, b, code)
    hi = 1 << 16
    top = ws(hi)
    assert top > 0
    lo = 1
    while lo < hi:                      # smallest batch whose workspace is the full chunk's
        mid = (lo + hi) // 2
        if ws(mid) == top:
            hi = mid
        else:
            lo = mid + 1
    chunk = lo
    assert 1 < chunk < 1 << 16 and ws(chunk - 1) < top
    _record(c.gid, prec, "chunk", chunk)
    n = chunk + 37
    x, md = c.inputs(n, seed=200 + code)
    part = lambda a, s: None if a is None else tuple(v[s] for v in a)
    y = c.run(prec, x, md)
    assert np.array_equal(y[:chunk], c.run(prec, x[:chunk], part(md, slice(0, chunk)))), "first chunk"
    assert np.array_equal(y[chunk:], c.run(prec, x[chunk:], part(md, slice(chunk, n)))), "ragged second chunk"
    idx = [chunk - 1, chunk]
    _check_samples(c, prec, y[idx], c.oracle(idx, x, md), "chunk_edge_vs_oracle")
    hc = min(2048, chunk)
    nh = 2 * hc + 37
    xh, mdh = c.inputs(nh, seed=300 + code)
    yd = c.run(prec, xh, mdh)
    c.model._workspace = None           # the two host lanes allocate their own chunk workspaces
    torch.cuda.empty_cache()
    assert np.array_equal(c.run_host(prec, xh, mdh), yd), "forward_host"
