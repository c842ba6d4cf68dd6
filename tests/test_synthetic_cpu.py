"""CPU: the synthetic-channel rule (``include/aft.h``, "Synthetic channels") and its fp64 restatement
``oracle/channel_ref.py``.

* The restatement draws from the channel model of ``aft_oracle.synthetic_channel``: mean |H|^2, frequency correlation at
  dk in {1, 8, 40}, time correlation at dl in {1, 6, 13} and pilot error power agree between the two within 5 standard
  errors at 16384 samples per arm, the time correlation matches J0(2 pi f_d dl Ts) (Jakes) and the pilot error power
  sigma^2.
* The product's condition grids are the oracle's; uniforms and grid indices cover their ranges.
* The 1e-6 gate of ``tests/test_gpu_synthetic.py`` catches a frequency phase taken in fp32 without turn reduction.
* ``aft_synthetic_channels`` refuses bad arguments with nothing launched, and ``SyntheticChannels`` checks its condition.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.special import j0

from adafortitran_b200 import _capi, data
from oracle import aft_oracle as O
from oracle import channel_ref as R

N_ARM = 16384
COND = (10.0, 300.0, 1000.0)        # SNR dB, delay spread ns, Doppler Hz
DK, DL = (1, 8, 40), (1, 6, 13)
TS = 1e-3 / 14


def _stats(pilots, truth):
    """Per-sample statistics: {name: [n] array (complex for correlations)}."""
    h = truth.astype(np.complex128)
    out = {"power": np.mean(np.abs(h) ** 2, axis=(1, 2))}
    for dk in DK:
        out[f"freq{dk}"] = np.mean(h[:, dk:, :] * np.conj(h[:, :-dk, :]), axis=(1, 2))
    for dl in DL:
        out[f"time{dl}"] = np.mean(h[:, :, dl:] * np.conj(h[:, :, :-dl]), axis=(1, 2))
    sc = np.arange(12) * 10
    err = pilots.astype(np.complex128) - h[:, sc][:, :, [2, 11]]
    out["pilot_err"] = np.mean(np.abs(err) ** 2, axis=(1, 2))
    return out


def _arm(gen, chunks):
    parts = [_stats(*gen(c)) for c in range(chunks)]
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


@pytest.fixture(scope="module")
def arms():
    oracle = _arm(lambda c: O.synthetic_channel(1024, *COND, seed=9000 + c), N_ARM // 1024)
    ref = _arm(lambda c: R.synthetic_channels(77, c * 2048, 2048, cond=COND)[:2], N_ARM // 2048)
    return oracle, ref


def _mean_se(x):
    return x.mean(), x.std(ddof=1) / np.sqrt(len(x))


@pytest.mark.parametrize("stat", ["power"] + [f"freq{d}" for d in DK] + [f"time{d}" for d in DL] + ["pilot_err"])
def test_restatement_matches_oracle_model(arms, stat):
    oracle, ref = arms
    for part in (np.real, np.imag) if np.iscomplexobj(ref[stat]) else (np.real,):
        (ma, sa), (mb, sb) = _mean_se(part(oracle[stat])), _mean_se(part(ref[stat]))
        print(f"{stat} {part.__name__}: oracle {ma:.5f} +- {sa:.5f}, restatement {mb:.5f} +- {sb:.5f}")
        assert abs(ma - mb) <= 5 * np.hypot(sa, sb), (stat, part.__name__, ma, mb, sa, sb)


@pytest.mark.parametrize("dl", DL)
def test_time_correlation_is_jakes(arms, dl):
    x = arms[1][f"time{dl}"]
    want = j0(2 * np.pi * COND[2] * dl * TS)
    m, se = _mean_se(x.real)
    mi, sei = _mean_se(x.imag)
    print(f"dl {dl}: {m:.5f} +- {se:.5f}, J0 {want:.5f}; imaginary {mi:.5f} +- {sei:.5f}")
    assert abs(m - want) <= 5 * se and abs(mi) <= 5 * sei


def test_pilot_error_power_is_sigma_squared(arms):
    m, se = _mean_se(arms[1]["pilot_err"])
    assert abs(m - 10 ** (-COND[0] / 10)) <= 5 * se, (m, se)


def test_grids_uniforms_and_indices():
    assert np.array_equal(np.asarray(data.SNR_GRID, np.float32), O.SNR_GRID)
    assert np.array_equal(np.asarray(data.DS_GRID, np.float32), O.DS_GRID)
    assert np.array_equal(np.asarray(data.DOP_GRID, np.float32), O.DOP_GRID)
    w = np.array([0, 0xFF, 0x100, 0x24924924, 0x24924A00, 0xFFFFFFFF], np.uint32)
    u = R.uniform(w)
    assert u[0] == 2.0 ** -24 and u[-1] == 1 - 2.0 ** -24 and np.all((u > 0) & (u < 1))
    assert np.array_equal(u.astype(np.float32).astype(np.float64), u)
    assert R.grid_index(w).tolist() == [0, 0, 0, 0, 1, 6]
    # every grid value is drawn, about equally often
    snr, ds, dop = R.conditions(5, np.arange(7000, dtype=np.uint64))
    for v, grid in ((snr, O.SNR_GRID), (ds, O.DS_GRID), (dop, O.DOP_GRID)):
        counts = np.array([(v == g).sum() for g in grid])
        assert counts.sum() == 7000 and counts.min() > 850, counts


def _nw_per_sample(a, b):
    """max|a - b| / max|b| of every sample (``aft_oracle.normwise_err`` per sample)."""
    return np.array([O.normwise_err(x, y) for x, y in zip(a, b)])


def test_gate_catches_unreduced_fp32_phase():
    """At 3276 x 14 (pilots 1638 x 2) k df tau reaches hundreds of turns, and an fp32 angle in radians there is off by
    up to ~1e-4 rad.  The taps of long delay carry little power, so what shows is 5e-6 .. 8e-6 of max|H| per sample at a
    350 ns delay spread: five times the GPU test's 1e-6 per-sample gate."""
    ext = dict(num_scs=3276, num_symbols=14, pilot_scs=1638, pilot_symbols=2)
    cond = (30.0, 350.0, 1400.0)
    _, ref, _ = R.synthetic_channels(11, 0, 4, cond=cond, **ext)
    _, bad, _ = R.synthetic_channels(11, 0, 4, cond=cond, phase="fp32_unreduced", **ext)
    err = _nw_per_sample(bad, ref)
    print("unreduced fp32 phase at 3276 x 14, per-sample normwise error vs fp64:", " ".join(f"{e:.2e}" for e in err))
    assert err.min() > 4e-6


# ---------------------------------------------------------------------------------------------------------------------
# refusals (no device needed: every call below is refused before anything is enqueued)
# ---------------------------------------------------------------------------------------------------------------------
P = C.c_void_p(256)


def _call(cfg=None, seed=1, sample0=0, batch=4, snr=P, ds=P, dop=P, draw=1, pilots=P, truth=P):
    cfg = cfg if cfg is not None else dict(num_scs=120, num_symbols=14, pilot_scs=12, pilot_symbols=2)
    c = None if cfg == "null" else C.byref(_capi.AftConfig(**cfg))
    return _capi.lib().aft_synthetic_channels(c, seed, sample0, batch, snr, ds, dop, draw, pilots, truth, None)


def _geom(**kw):
    g = dict(num_scs=120, num_symbols=14, pilot_scs=12, pilot_symbols=2)
    g.update(kw)
    return g


REFUSED = [
    dict(cfg="null"), dict(batch=-1), dict(sample0=-1), dict(sample0=2 ** 63 - 3, batch=4), dict(sample0=2 ** 63 - 1, batch=1),
    dict(snr=None), dict(ds=None), dict(dop=None), dict(pilots=None), dict(truth=None), dict(snr=None, draw=0),
    dict(pilots=C.c_void_p(260)), dict(truth=C.c_void_p(252)),
    dict(cfg=_geom(num_scs=0)), dict(cfg=_geom(num_symbols=-14)), dict(cfg=_geom(pilot_scs=0)),
    dict(cfg=_geom(pilot_symbols=0)), dict(cfg=_geom(pilot_scs=121)), dict(cfg=_geom(pilot_symbols=3)),
    dict(cfg=_geom(num_symbols=11)), dict(cfg=_geom(num_symbols=2, pilot_symbols=1)),
]


def test_refusals_launch_nothing():
    lib = _capi.lib()
    before = lib.aft_launch_count()
    for change in REFUSED:
        rc = _call(**change)
        assert rc == _capi.AFT_ERR_INVALID, (change, rc, lib.aft_last_error())
    assert _call(cfg=_geom(num_symbols=257)) == _capi.AFT_ERR_UNSUPPORTED
    # batch 0: nothing to do, buffers may be NULL
    assert _call(batch=0, snr=None, ds=None, dop=None, pilots=None, truth=None) == _capi.AFT_OK
    assert _call(batch=0, sample0=2 ** 63 - 1) == _capi.AFT_OK
    assert lib.aft_launch_count() == before


def test_python_checks_conditions_and_device():
    sys = dict(ofdm=dict(num_scs=120, num_symbols=14), pilot=dict(num_scs=12, num_symbols=2))
    for bad in ((float("nan"), 100, 600), (10, 0, 600), (10, -5, 600), (10, 100, -1), (10, float("inf"), 600)):
        with pytest.raises(ValueError, match="conditions"):
            data.SyntheticChannels(sys, 1, conditions=bad)
    for seed in (-1, 2 ** 64):
        with pytest.raises(ValueError, match="seed"):
            data.SyntheticChannels(sys, seed)
    with pytest.raises(RuntimeError, match="CPU fallback"):
        data.SyntheticChannels(sys, 1, device="cpu")
