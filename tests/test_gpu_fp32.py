"""GPU: the fp32 CUDA path through the C-ABI against the golden vectors and the oracle.
Gate (BASELINE.json north_star / SURVEY.md 7.3): max|y - ref| / max|ref| <= 1e-4."""
import numpy as np
import pytest
import torch

from oracle import aft_oracle as O
from tests import util

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def sd():
    return util.ada_weights()


@pytest.fixture(scope="module")
def ada(sd):
    return util.make_model("ada", weights=sd)


def run(model, pilots, snr=None, ds=None, dop=None):
    md = util.meta(snr, ds, dop) if snr is not None else None
    with torch.no_grad():
        y = model(torch.from_numpy(pilots), md)
    assert y.dtype == torch.complex64 and y.device.type == "cuda"
    return y.cpu().numpy()


def test_golden_ada(ada):
    g = util.golden("golden_ada.npz")
    y = run(ada, g["pilots"], g["snr"], g["ds"], g["dop"])
    assert y.shape == (8, 120, 14)
    assert O.normwise_err(y, g["out"]) <= TOL
    assert O.normwise_err(y, g["out64"]) <= TOL


def test_golden_fortitran(sd):
    g = util.golden("golden_forti.npz")
    m = util.make_model("forti", weights=util.forti_weights(sd))
    assert O.normwise_err(run(m, g["pilots"]), g["out"]) <= TOL
    # FortiTran ignores meta_data (reference fortitran.py:160-161)
    with torch.no_grad():
        y2 = m(torch.from_numpy(g["pilots"]), util.meta(np.zeros(8), np.zeros(8), np.zeros(8))).cpu().numpy()
    assert O.normwise_err(y2, g["out"]) <= TOL


def test_golden_variants(sd):
    g = util.golden("golden_ada.npz")
    v = util.golden("golden_variants.npz")
    args = (g["pilots"][:4], g["snr"][:4], g["ds"][:4], g["dop"][:4])
    m = util.make_model("ada", weights=sd, overrides={"activation": "relu"})
    assert O.normwise_err(run(m, *args), v["out_relu"]) <= TOL
    m = util.make_model("ada", overrides={"num_layers": 2},
                        weights={k: a for k, a in sd.items() if not any(f"layers.{i}." in k for i in range(2, 6))})
    assert O.normwise_err(run(m, *args), v["out_layers2"]) <= TOL
    m = util.make_model("ada", overrides={"pos_encoding_type": "sinusoidal"})
    s2 = {k: a for k, a in sd.items() if "position_embeddings" not in k}
    s2["transformer_encoder.positional_encoding.pe"] = m.state_dict()["transformer_encoder.positional_encoding.pe"].cpu().numpy()
    m.load_state_dict(util.to_torch(s2))
    assert O.normwise_err(run(m, *args), v["out_sinusoidal"]) <= TOL


def test_golden_sweep(ada):
    g = util.golden("golden_sweep.npz")
    pilots = g["pilots"].reshape(-1, 12, 2)
    conds = np.repeat(g["conds"], 4, axis=0)
    y = run(ada, pilots, conds[:, 0], conds[:, 1], conds[:, 2]).reshape(21, 4, 120, 14)
    for i in range(21):
        assert O.normwise_err(y[i], g["out"][i]) <= TOL, i


def test_oracle_parity_ragged_batches(ada, sd):
    """Seeded batches of awkward sizes (1, 3, 65) against the oracle on the same inputs."""
    for b, seed in ((1, 11), (3, 12), (65, 13)):
        p, snr, ds, dop = O.synthetic_batch(b, seed=seed)
        ref = O.forward(util.oracle_cfg(), sd, p, snr, ds, dop, dtype=np.float64)
        assert O.normwise_err(run(ada, p, snr, ds, dop), ref) <= TOL, b


def test_empty_batch(ada):
    with torch.no_grad():
        y = ada(torch.zeros(0, 12, 2, dtype=torch.cfloat), util.meta([], [], []))
    assert y.shape == (0, 120, 14)


def test_properties_at_scale(ada):
    """Size-independent properties at a batch that crosses the internal chunk boundary (fp32 chunk = 1024):
    batch-permutation equivariance, real/imag independence, determinism."""
    b = 1024 + 37
    p, snr, ds, dop = O.synthetic_batch(b, seed=21)
    y = run(ada, p, snr, ds, dop)
    assert np.isfinite(y.view(np.float32)).all()
    perm = np.random.default_rng(0).permutation(b)
    yp = run(ada, p[perm], snr[perm], ds[perm], dop[perm])
    assert np.array_equal(yp, y[perm])
    # f(x).real depends only on x.real (reference fortitran.py:176-177)
    p2 = (p.real + 1j * np.roll(p.imag, 1, axis=0)).astype(np.complex64)
    y2 = run(ada, p2, snr, ds, dop)
    assert np.array_equal(y2.real, y.real)
    # spot-check a few rows of the big batch against the oracle
    idx = [0, 1023, 1024, b - 1]
    ref = O.forward(util.oracle_cfg(), util.ada_weights(), p[idx], snr[idx], ds[idx], dop[idx])
    assert O.normwise_err(y[idx], ref) <= TOL


def test_weight_update_is_picked_up(sd):
    m = util.make_model("ada", weights=sd)
    p, snr, ds, dop = O.synthetic_batch(2, seed=5)
    y0 = run(m, p, snr, ds, dop)
    with torch.no_grad():
        m.transformer_encoder.linear_2.bias.add_(1.0)
    y1 = run(m, p, snr, ds, dop)
    sd2 = dict(sd)
    sd2["transformer_encoder.linear_2.bias"] = sd["transformer_encoder.linear_2.bias"] + 1.0
    ref = O.forward(util.oracle_cfg(), sd2, p, snr, ds, dop)
    assert O.normwise_err(y1, ref) <= TOL and not np.array_equal(y0, y1)


def test_host_entry_point_matches_device(ada):
    p, snr, ds, dop = O.synthetic_batch(2048 + 5, seed=8)
    y = run(ada, p, snr, ds, dop)
    yh = ada.forward_host(torch.from_numpy(p), util.meta(snr, ds, dop)).numpy()
    assert np.array_equal(y, yh)


def test_error_sums_kernel(ada):
    import ctypes as C
    from adafortitran_b200 import _capi
    rng = np.random.default_rng(3)
    a = (rng.standard_normal((5, 120, 14)) + 1j * rng.standard_normal((5, 120, 14))).astype(np.complex64)
    b = (rng.standard_normal((5, 120, 14)) + 1j * rng.standard_normal((5, 120, 14))).astype(np.complex64)
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _capi.check(_capi.lib().aft_error_sums(C.c_void_p(ta.data_ptr()), C.c_void_p(tb.data_ptr()), a.size,
                                          C.c_void_p(sums.data_ptr()), C.c_void_p(st)))
    s = sums.cpu().numpy()
    assert abs(s[0] - np.sum(np.abs(a.astype(np.complex128) - b) ** 2)) / s[0] < 1e-6
    assert abs(s[1] - np.sum(np.abs(b.astype(np.complex128)) ** 2)) / s[1] < 1e-6
    # the reference's reported metric from these sums
    assert abs(10 * np.log10(s[0] / a.size) - O.mse_db_reference(a, b)) < 1e-4
    # Grid edges of the capped grid (148 * 8 blocks of 256 threads, grid-stride): one element, a partial block, one
    # element past a block, one element past one pass (303,105), and 4096 estimates + 3.  Magnitudes 1e-3 .. 1e3, every
    # fifth element with est == truth, sums prefilled (the call accumulates).  Each term is formed in fp32 and added in
    # fp64: a non-negative term is off by at most 4 * 2^-24, so the sums are within 3e-7 of fp64 sums of the same inputs.
    lib = _capi.lib()
    for n in (1, 255, 257, 148 * 8 * 256 + 1, 4096 * 1680 + 3):
        mag = 10.0 ** rng.uniform(-3, 3, size=(2, n))
        a = (mag[0] * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
        b = (mag[1] * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
        a[3::5] = b[3::5]
        ref = np.array([np.sum(np.abs(a.astype(np.complex128) - b) ** 2), np.sum(np.abs(b.astype(np.complex128)) ** 2)])
        pre = np.array([0.375, 0.625]) * ref
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        sums = torch.from_numpy(pre.copy()).cuda()
        _capi.check(lib.aft_error_sums(C.c_void_p(ta.data_ptr()), C.c_void_p(tb.data_ptr()), n,
                                       C.c_void_p(sums.data_ptr()), C.c_void_p(st)))
        err = np.abs(sums.cpu().numpy() - (pre + ref))
        assert (err <= 3e-7 * ref).all(), (n, err / ref)
    kept, before = sums.cpu().numpy(), lib.aft_launch_count()     # count 0: nothing launched, sums untouched
    _capi.check(lib.aft_error_sums(C.c_void_p(ta.data_ptr()), C.c_void_p(tb.data_ptr()), 0, C.c_void_p(sums.data_ptr()),
                                   C.c_void_p(st)))
    assert lib.aft_launch_count() == before
    assert np.array_equal(sums.cpu().numpy(), kept)
