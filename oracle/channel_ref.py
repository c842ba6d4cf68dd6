"""fp64 restatement of the synthetic-channel rule of ``include/aft.h`` ("Synthetic channels").

TEST INFRASTRUCTURE ONLY (same rules as ``aft_oracle.py``): imported by ``tests/`` and ``tools/``, never by the product
package.

The channel model is :func:`aft_oracle.synthetic_channel`'s (8 taps, exponential delays, uniform phases, Jakes-type
Doppler, LS pilots at subcarriers ``i * (num_scs // pilot_scs)`` and symbols ``[2, 11]``); what this file adds is the
random numbers: every draw of sample ``s`` is :func:`train_ref.philox4x32_10` with counter ``(j, s & 0xffffffff, s >> 32,
TAG)``, so a sample depends on (seed, s, condition) only.  Everything after the draws is evaluated in float64 numpy.
"""
from __future__ import annotations

import numpy as np

from oracle.aft_oracle import DOP_GRID, DS_GRID, SNR_GRID
from oracle.train_ref import philox4x32_10

TAG = 0x53594E54
TAPS = 8
DF, TS = 15e3, 1e-3 / 14
PILOT_SYMBOLS = (2, 11)


def draws(seed: int, samples: np.ndarray, j) -> list:
    """The four uint32 output words of draw ``j`` (int or array) for each global sample index in ``samples``."""
    s = np.asarray(samples, dtype=np.uint64)
    z = np.zeros_like(s)
    return philox4x32_10([z + np.uint64(j), s & np.uint64(0xFFFFFFFF), s >> np.uint64(32), z + np.uint64(TAG)],
                         (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))


def uniform(w) -> np.ndarray:
    """``((w >> 8) | 1) * 2^-24``: in (0, 1), exact in fp32 and fp64."""
    return ((np.asarray(w, np.uint32) >> np.uint32(8)) | np.uint32(1)).astype(np.float64) * 2.0 ** -24


def grid_index(w) -> np.ndarray:
    return ((np.asarray(w, np.uint32) >> np.uint32(8)).astype(np.uint64) * np.uint64(7) >> np.uint64(24)).astype(np.int64)


def conditions(seed: int, samples: np.ndarray):
    """Draw 0: (snr, ds, doppler) float32 [n] from the reference's 7 x 7 x 7 grid."""
    w = draws(seed, samples, 0)
    return SNR_GRID[grid_index(w[0])], DS_GRID[grid_index(w[1])], DOP_GRID[grid_index(w[2])]


def synthetic_channels(seed: int, sample0: int, n: int, num_scs: int = 120, num_symbols: int = 14, pilot_scs: int = 12,
                       pilot_symbols: int = 2, cond=None, phase: str = "fp64"):
    """Samples ``sample0 .. sample0 + n - 1``: (pilots c128 [n, pilot_scs, pilot_symbols], truth c128 [n, num_scs,
    num_symbols], (snr, ds, doppler) float32 [n]).  ``cond`` = (snr, ds, doppler) fixes the condition of every sample
    (scalars or [n] arrays); None draws it.

    ``phase="fp32_unreduced"`` takes the frequency phase ``2 pi k df tau`` as an fp32 angle in radians without removing
    the whole turns (and ``tau`` in fp32): what a kernel that skipped the fp64 turn count would compute.  It exists to
    show that the tests' gate catches that."""
    samples = np.arange(sample0, sample0 + n, dtype=np.uint64)
    if cond is None:
        snr, ds, dop = conditions(seed, samples)
    else:
        snr, ds, dop = (np.broadcast_to(np.asarray(v, np.float32), (n,)).copy() for v in cond)
    u = np.empty((3, n, TAPS))
    for t in range(TAPS):
        w = draws(seed, samples, 1 + t)
        for c in range(3):
            u[c, :, t] = uniform(w[c])
    u_tau, u_ph, u_dop = u
    ds64, dop64 = ds.astype(np.float64)[:, None], dop.astype(np.float64)[:, None]
    tau = -ds64 * 1e-9 * np.log(u_tau)                                  # [n, taps] seconds
    pw = np.exp(-tau / (ds64 * 1e-9))
    pw /= pw.sum(axis=1, keepdims=True)
    amp = np.sqrt(pw) * np.exp(2j * np.pi * u_ph)
    nu = dop64 * np.cos(2 * np.pi * u_dop)
    k = np.arange(num_scs, dtype=np.float64)
    l = np.arange(num_symbols, dtype=np.float64)
    if phase == "fp64":
        fre = np.exp(-2j * np.pi * k[None, None, :] * DF * tau[:, :, None])           # [n, taps, scs]
    elif phase == "fp32_unreduced":
        ang = (np.float32(2 * np.pi) * k.astype(np.float32)[None, None, :] * np.float32(DF)
               * tau.astype(np.float32)[:, :, None])
        fre = np.cos(ang).astype(np.float64) - 1j * np.sin(ang).astype(np.float64)
    else:
        raise ValueError(phase)
    dopf = amp[:, :, None] * np.exp(2j * np.pi * nu[:, :, None] * l[None, None, :] * TS)   # [n, taps, symbols]
    truth = np.einsum("ntk,ntl->nkl", fre, dopf)
    sc = np.arange(pilot_scs) * (num_scs // pilot_scs)
    sym = np.array(PILOT_SYMBOLS[:pilot_symbols])
    P = pilot_scs * pilot_symbols
    noise = np.empty((n, P), np.complex128)
    sigma = 10.0 ** (-snr.astype(np.float64) / 20)
    for q in range((P + 1) // 2):
        w = draws(seed, samples, 9 + q)
        for h in range(min(2, P - 2 * q)):
            u1, u2 = uniform(w[2 * h]), uniform(w[2 * h + 1])
            noise[:, 2 * q + h] = sigma / np.sqrt(2) * np.sqrt(-2 * np.log(u1)) * np.exp(2j * np.pi * u2)
    pilots = truth[:, sc][:, :, sym] + noise.reshape(n, pilot_scs, pilot_symbols)
    return pilots, truth, (snr, ds, dop)
