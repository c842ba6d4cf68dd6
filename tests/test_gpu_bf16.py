"""GPU: the bf16 tcgen05 path through the C-ABI.

Gates (BASELINE.json north_star; SURVEY.md 7.3 / 8d):
  * official : |delta NMSE| <= 0.05 dB against the reference forward on the 21-condition synthetic sweep;
  * self-imposed: output-relative error against the fp64 oracle <= -45 dB for FortiTran and <= -38 dB for AdaFortiTran.
    (AdaFortiTran feeds raw SNR/delay-spread/Doppler values (up to 1400) into the token features, so at random init the
    residual stream is dominated by metadata-driven components ~1e4 times larger than the pilot-driven ones; ANY bf16
    operand path loses those: the reference's own bf16 autocast reaches only -33.6 dB (SURVEY.md 7.3, probe P5), a numpy
    model of this kernel's rounding points predicts -37.7 dB, the kernel measures -39 .. -41 dB.)
The kernel-level building blocks are checked first (aft_selftest) so a failure localises.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from adafortitran_b200 import _capi
from oracle import aft_oracle as O
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sd():
    return util.ada_weights()


def run(model, pilots, snr=None, ds=None, dop=None):
    md = util.meta(snr, ds, dop) if snr is not None else None
    with torch.no_grad():
        return model(torch.from_numpy(pilots), md).cpu().numpy()


@pytest.mark.parametrize("which,tol", [(0, 1e-4), (1, 5e-3), (2, 5e-3), (4, 2e-2)])
def test_tcgen05_building_blocks(which, tol):
    """UMMA GEMM tile (SWIZZLE_128B K-major descriptors, TMEM loads) and attention tiles (SWIZZLE_64B Q/K, MN-major V,
    P as TMEM A operand) against a double-precision host reference inside the library."""
    torch.zeros(1, device="cuda")
    err = C.c_double(-1)
    st = torch.cuda.current_stream().cuda_stream
    _capi.check(_capi.lib().aft_selftest(which, C.byref(err), C.c_void_p(st)))
    assert 0 <= err.value <= tol, err.value


def test_fortitran_vs_oracle(sd):
    g = util.golden("golden_forti.npz")
    m = util.make_model("forti", weights=util.forti_weights(sd), precision="bf16")
    y = run(m, g["pilots"])
    assert O.rel_err_db(y, g["out"]) <= -45.0
    assert O.normwise_err(y, g["out"]) <= 2e-2


def test_adafortitran_vs_oracle(sd):
    g = util.golden("golden_ada.npz")
    m = util.make_model("ada", weights=sd, precision="bf16")
    y = run(m, g["pilots"], g["snr"], g["ds"], g["dop"])
    assert O.rel_err_db(y, g["out64"]) <= -38.0       # measured -39.1 dB (profiles/r02_gates_report.json)


def test_variants_relu_layers2_sinusoidal(sd):
    g = util.golden("golden_ada.npz")
    v = util.golden("golden_variants.npz")
    args = (g["pilots"][:4], g["snr"][:4], g["ds"][:4], g["dop"][:4])
    m = util.make_model("ada", weights=sd, precision="bf16", overrides={"activation": "relu"})
    assert O.rel_err_db(run(m, *args), v["out_relu"]) <= -38.0
    m = util.make_model("ada", precision="bf16", overrides={"num_layers": 2},
                        weights={k: a for k, a in sd.items() if not any(f"layers.{i}." in k for i in range(2, 6))})
    assert O.rel_err_db(run(m, *args), v["out_layers2"]) <= -38.0
    m = util.make_model("ada", precision="bf16", overrides={"pos_encoding_type": "sinusoidal"})
    s2 = {k: a for k, a in sd.items() if "position_embeddings" not in k}
    s2["transformer_encoder.positional_encoding.pe"] = m.state_dict()["transformer_encoder.positional_encoding.pe"].cpu().numpy()
    m.load_state_dict(util.to_torch(s2))
    assert O.rel_err_db(run(m, *args), v["out_sinusoidal"]) <= -38.0


def test_sweep_delta_nmse(sd):
    """21 conditions x 256 synthetic channels: NMSE of the bf16 path vs NMSE of the fp32 path (itself <= 1e-4 from the
    reference) -- the north_star gate is 0.05 dB; also checked against the committed reference outputs."""
    bf = util.make_model("ada", weights=sd, precision="bf16")
    fp = util.make_model("ada", weights=sd, precision="fp32")
    g = util.golden("golden_sweep.npz")
    worst = 0.0
    table = []
    for i, (s, d, f) in enumerate(g["conds"]):
        p, h = O.synthetic_channel(256, float(s), float(d), float(f), seed=9000 + i)
        md = ([s] * 256, [d] * 256, [f] * 256)
        yb, yf = run(bf, p, *md), run(fp, p, *md)
        worst = max(worst, abs(O.nmse_db(yb, h) - O.nmse_db(yf, h)))
        table.append(dict(snr=float(s), ds=float(d), dop=float(f), nmse_fp32_db=O.nmse_db(yf, h), nmse_bf16_db=O.nmse_db(yb, h),
                          mse_ref_def_fp32_db=O.mse_db_reference(yf, h), bf16_vs_fp32_rel_err_db=O.rel_err_db(yb, yf)))
        # conditioning degrades with the raw metadata magnitude (Doppler up to 1400): informational floor only
        assert O.rel_err_db(yb, yf) <= -30.0, (i, table[-1])
        # the committed reference outputs for this condition (4 samples)
        yr = run(bf, g["pilots"][i], *( [s] * 4, [d] * 4, [f] * 4))
        assert abs(O.nmse_db(yr, g["truth"][i]) - O.nmse_db(g["out"][i], g["truth"][i])) <= 0.05, i
    import json, os
    os.makedirs(os.path.join(util.ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(util.ROOT, "gpurun_out", "sweep_bf16_vs_fp32.json"), "w") as fh:
        json.dump(dict(worst_delta_nmse_db=worst, conditions=table), fh, indent=1)
    assert worst <= 0.05, worst


def test_trained_weights_sweep():
    """The accuracy gates on weights that MEAN something: a pseudo-trained AdaFortiTran (a few hundred Adam steps of the live
    reference on synthetic channels, tests/golden/make_golden_trained.py; NMSE -3 ... -13 dB per condition instead of the
    ~0 dB of a random initialisation).  Per condition of the 21-point sweep: the fp32 path reproduces the reference's
    recorded outputs (<= 1e-4 normwise), and the bf16 path keeps the reference's NMSE within the north-star's 0.05 dB and
    its output within -30 dB of output-relative error power."""
    g = util.golden("golden_trained.npz")
    sd = {k[3:]: g[k] for k in g if k.startswith("sd/")}
    m32 = util.make_model("ada", weights=sd, precision="fp32")
    mbf = util.make_model("ada", weights=sd, precision="bf16")
    n, seed0 = int(g["samples"]), int(g["seed0"])
    rows, worst_d, worst_rel, worst_32 = [], 0.0, -1e9, 0.0
    for i, (snr, ds, dop) in enumerate(g["conds"]):
        pilots, truth = O.synthetic_channel(int(g["gen_batch"]), float(snr), float(ds), float(dop), seed=seed0 + i)   # as the generator drew them
        pilots, truth = pilots[:n], truth[:n]
        args = (pilots, np.full(n, snr, np.float32), np.full(n, ds, np.float32), np.full(n, dop, np.float32))
        ref = g["out"][i]
        assert abs(O.nmse_db(ref, truth) - float(g["nmse_db"][i])) < 1e-3        # inputs regenerated exactly
        y32, ybf = run(m32, *args), run(mbf, *args)
        e32 = O.normwise_err(y32, ref)
        d = abs(O.nmse_db(ybf, truth) - O.nmse_db(ref, truth))
        rel = O.rel_err_db(ybf, ref)
        worst_d, worst_rel, worst_32 = max(worst_d, d), max(worst_rel, rel), max(worst_32, e32)
        rows.append(dict(snr=float(snr), ds=float(ds), doppler=float(dop), nmse_ref_db=O.nmse_db(ref, truth),
                         nmse_fp32_db=O.nmse_db(y32, truth), nmse_bf16_db=O.nmse_db(ybf, truth), fp32_normwise=e32, bf16_rel_err_db=rel))
    import json, os
    out = os.path.join(util.ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "trained_sweep_bf16_vs_reference.json"), "w") as f:
        json.dump(dict(worst_abs_delta_nmse_db=worst_d, worst_bf16_rel_err_db=worst_rel, worst_fp32_normwise=worst_32,
                       conditions=rows), f, indent=1)
    assert max(r["nmse_ref_db"] for r in rows) < -2.5          # the fixture is informative: every condition well below 0 dB
    assert worst_32 <= 1e-4, worst_32
    assert worst_d <= 0.05, worst_d
    assert worst_rel <= -30.0, worst_rel


def test_ragged_and_chunked_batches(sd):
    """Batch sizes that do not fill the persistent grid (1, 3, 75 = 150 sequences > 148 CTAs) and one that crosses the
    internal chunk boundary (8192 + 3); properties: determinism, permutation equivariance, re/im independence."""
    m = util.make_model("forti", weights=util.forti_weights(sd), precision="bf16")
    cfg = util.oracle_cfg("forti")
    for b, seed in ((1, 31), (3, 32), (75, 33)):
        p, *_ = O.synthetic_batch(b, seed=seed)
        ref = O.forward(cfg, util.forti_weights(sd), p)
        assert O.rel_err_db(run(m, p), ref) <= -45.0, b
    b = 8192 + 3
    p, *_ = O.synthetic_batch(b, seed=34)
    y = run(m, p)
    assert np.isfinite(y.view(np.float32)).all()
    assert np.array_equal(run(m, p), y)                     # deterministic
    perm = np.random.default_rng(1).permutation(b)
    assert np.array_equal(run(m, p[perm]), y[perm])         # sequences are independent
    p2 = (p.real + 1j * np.roll(p.imag, 1, axis=0)).astype(np.complex64)
    assert np.array_equal(run(m, p2).real, y.real)
    idx = [0, 8191, 8192, b - 1]
    assert O.rel_err_db(y[idx], O.forward(cfg, util.forti_weights(sd), p[idx])) <= -45.0


def test_full_size_batch_properties(sd):
    """BASELINE config 2 at full size (FortiTran, B = 16384, two internal chunks of 8192): determinism, independence of
    the sequences (permutation equivariance), a checksum against the fp32 path (its own kernels, <= 1e-4 from the
    reference) and oracle parity on samples taken from both chunks."""
    w = util.forti_weights(sd)
    bf = util.make_model("forti", weights=w, precision="bf16")
    fp = util.make_model("forti", weights=w, precision="fp32")
    b = 16384
    p, *_ = O.synthetic_batch(b, seed=41)
    y = run(bf, p)
    assert y.shape == (b, 120, 14) and np.isfinite(y.view(np.float32)).all()
    assert np.array_equal(run(bf, p), y)
    perm = np.random.default_rng(2).permutation(b)
    assert np.array_equal(run(bf, p[perm]), y[perm])
    assert O.rel_err_db(y, run(fp, p)) <= -45.0                       # whole-batch error power vs the fp32 path
    idx = [0, 5000, 8191, 8192, 12345, b - 1]
    assert O.rel_err_db(y[idx], O.forward(util.oracle_cfg("forti"), w, p[idx])) <= -45.0


def test_host_entry_point_bf16(sd):
    m = util.make_model("ada", weights=sd, precision="bf16")
    # 2057: one tapered tail (1088 + 512 + 457); 5000: full chunks of 2048 followed by the tapering ones (aft_api.cu)
    for b, seed in ((2048 + 9, 35), (5000, 36)):
        p, snr, ds, dop = O.synthetic_batch(b, seed=seed)
        y = run(m, p, snr, ds, dop)
        yh = m.forward_host(torch.from_numpy(p), util.meta(snr, ds, dop)).numpy()
        assert np.array_equal(y, yh), b


def test_misaligned_output_is_rejected(sd):
    """The estimates leave the head kernel as 16-byte vectors / bulk copies: `aft_forward` must refuse an output pointer
    that is not 16-byte aligned (AFT_ERR_INVALID, nothing launched) instead of faulting on the device."""
    m = util.make_model("forti", weights=util.forti_weights(sd), precision="bf16")
    p, *_ = O.synthetic_batch(2, seed=5)
    with torch.no_grad():
        m(torch.from_numpy(p))                                     # creates the handle, loads the weights
        lib = _capi.lib()
        pil = torch.from_numpy(p).cuda().contiguous()
        raw = torch.empty(2 * 120 * 14 * 8 + 64, dtype=torch.uint8, device="cuda")
        ws = m._get_workspace(2, _capi.AFT_BF16)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        n0 = lib.aft_launch_count()
        rc = lib.aft_forward(m._handle, C.c_void_p(pil.data_ptr()), None, None, None, C.c_void_p(raw.data_ptr() + 8), 2,
                             _capi.AFT_BF16, C.c_void_p(ws_ptr), ws.numel() - (ws_ptr - ws.data_ptr()), st)
        assert rc == _capi.AFT_ERR_INVALID and b"16-byte aligned" in lib.aft_last_error()
        assert lib.aft_launch_count() == n0
        torch.cuda.synchronize()
        y = m(torch.from_numpy(p))                                 # the handle is still usable
        assert torch.isfinite(torch.view_as_real(y)).all()


def test_empty_batch_and_profile_api(sd):
    m = util.make_model("forti", weights=util.forti_weights(sd), precision="bf16")
    with torch.no_grad():
        assert m(torch.zeros(0, 12, 2, dtype=torch.cfloat)).shape == (0, 120, 14)
        m(torch.zeros(4, 12, 2, dtype=torch.cfloat))
        lib = _capi.lib()
        _capi.check(lib.aft_profile_enable(m._handle, 1))
        n0 = lib.aft_launch_count()
        m(torch.zeros(4, 12, 2, dtype=torch.cfloat))
        ms, nl = (C.c_double * 3)(), (C.c_int64 * 3)()
        _capi.check(lib.aft_profile_read(m._handle, ms, nl))
        assert lib.aft_launch_count() - n0 == 3 and list(nl) == [1, 1, 1] and all(t > 0 for t in ms)
        _capi.check(lib.aft_profile_enable(m._handle, 0))


def test_protocol_under_random_delays():
    """The encoder / conv kernels are static programs of several roles that meet only through mbarriers.  The "chaos"
    build (adafortitran_b200.build variant, built by __graft_entry__.build) delays every wait by a pseudo-random time, so
    a hand-off that only works because of the usual relative timing shows up as a wrong result or a trapped wait."""
    import json, os, subprocess, sys
    from adafortitran_b200.build import build as build_lib, lib_file
    lib = lib_file("chaos")
    if not os.path.exists(lib):
        build_lib(variant="chaos")      # normally built by __graft_entry__.build(); nvcc, about a minute
    elif os.path.getmtime(lib) + 120 < os.path.getmtime(lib_file()):
        try:                            # clearly older than the product library: refresh it if a compiler is around
            build_lib(variant="chaos")
        except Exception:
            pass
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, AFT_B200_LIB=lib)
    for batch, kind, gate in (("296", "forti", -45.0), ("74", "ada", -36.0)):
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "chaos_check.py"), batch, kind], env=env,
                           capture_output=True, text=True, timeout=900)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")]
        assert line, r.stdout + r.stderr
        res = json.loads(line[-1])
        assert r.returncode == 0, res
        assert res["lib"] == "libaft_b200_chaos.so" and res["wait_timeouts"] == 0 and res["rel_db_bf16_vs_fp32"] <= gate, res
