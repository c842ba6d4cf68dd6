"""Input side of the hot path (SURVEY.md §8f row N2): what ``MatDataset`` / ``extract_values`` hand to the model
(reference src/data/dataset.py:36-190, src/utils.py:68-110), with the per-file pilot extraction batched on the GPU.

* :func:`extract_values` -- file name -> the 6-tuple of metadata the reference collates into ``meta_data``.
* :func:`extract_pilots` -- batched ``_process_channel_data``: non-zero entries of the sparse LS grid, row-major
  (``aft_extract_pilots``; device tensors in, device tensors out, ``ValueError`` on a wrong pilot count).
* :class:`MatDataset` -- same ``__getitem__`` contract as the reference for ``.mat`` files holding ``H`` [scs, symbols, >=2];
  :func:`collate_on_device` stacks raw grids of a batch and extracts all pilots in one launch.
* :class:`SyntheticChannels` -- training / evaluation batches generated on the GPU (``aft_synthetic_channels``) in the
  form :func:`collate_on_device` returns; sample ``s`` of a seed is fixed by ``s`` alone, so data-parallel ranks generate
  exactly their rows of the global batch.
"""
from __future__ import annotations

import ctypes as C
import math
import re
from pathlib import Path
from typing import Callable, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _capi
from .config import PilotParams

_NAME = re.compile(r"(\d+)_SNR-(\d+)_DS-(\d+)_DOP-(\d+)_N-(\d+)_([A-Z\-]+)\.mat")


def extract_values(file_name: str):
    """``'{n}_SNR-{snr}_DS-{ds}_DOP-{dop}_N-{pilot_freq}_{channel}.mat'`` -> five float32 tensors of shape [1] and
    ``[channel]`` (reference src/utils.py:68-110, ``re.match`` semantics); ``ValueError`` otherwise."""
    m = _NAME.match(file_name)
    if not m:
        raise ValueError("Cannot extract file information.")
    vals = tuple(torch.tensor([int(m.group(i))], dtype=torch.float) for i in range(1, 6))
    return (*vals, [m.group(6)])


def extract_pilots(ls_grid: torch.Tensor, pilot_size: Tuple[int, int]) -> torch.Tensor:
    """complex64 ``[B, scs, symbols]`` sparse LS grids on a CUDA device -> complex64 ``[B, pilot_scs, pilot_symbols]``.
    Every sample must hold exactly ``pilot_scs * pilot_symbols`` non-zero entries (dataset.py:129-133)."""
    if ls_grid.dim() != 3 or not ls_grid.is_complex():
        raise ValueError(f"expected a complex [B, subcarriers, symbols] tensor, got {tuple(ls_grid.shape)} {ls_grid.dtype}")
    if ls_grid.device.type != "cuda":
        raise RuntimeError("adafortitran_b200 has no CPU fallback: extract_pilots needs a CUDA tensor")
    grid = ls_grid.to(torch.complex64).contiguous()
    batch, cells, expected = grid.shape[0], grid.shape[1] * grid.shape[2], pilot_size[0] * pilot_size[1]
    pilots = torch.zeros((batch, pilot_size[0], pilot_size[1]), dtype=torch.complex64, device=grid.device)
    counts = torch.empty((batch,), dtype=torch.int32, device=grid.device)
    with torch.cuda.device(grid.device):
        stream = torch.cuda.current_stream(grid.device).cuda_stream
        _capi.check(_capi.lib().aft_extract_pilots(C.c_void_p(grid.data_ptr()), C.c_void_p(pilots.data_ptr()),
                                                   C.c_void_p(counts.data_ptr()), batch, cells, expected, C.c_void_p(stream)))
    bad = (counts != expected).nonzero()
    if bad.numel():
        i = int(bad[0])
        raise ValueError(f"Error processing channel data: Expected {expected} pilot values, got {int(counts[i])} (sample {i})")
    return pilots


class MatDataset(torch.utils.data.Dataset):
    """Reference ``MatDataset`` contract (dataset.py:36-190): item = (LS pilots [pilot_scs, pilot_symbols] c64, ground
    truth [scs, symbols] c64, metadata 6-tuple).  ``raw=True`` returns the sparse LS grid instead of the pilots so that
    :func:`collate_on_device` can extract a whole batch on the GPU."""

    def __init__(self, data_dir: Union[str, Path], pilot_params: Union[PilotParams, Sequence[int]],
                 transform: Optional[Callable] = None, raw: bool = False) -> None:
        self.data_dir = Path(data_dir)
        if not hasattr(pilot_params, "num_scs"):   # convenience: (pilot_scs, pilot_symbols)
            pilot_params = PilotParams(num_scs=pilot_params[0], num_symbols=pilot_params[1])
        self.pilot_params = pilot_params
        self.transform = transform
        self.raw = raw
        if not self.data_dir.exists():
            raise FileNotFoundError(f"Data directory not found: {self.data_dir}")
        self.file_list: List[Path] = list(self.data_dir.glob("*.mat"))
        if not self.file_list:
            raise ValueError(f"No .mat files found in {self.data_dir}")

    def __len__(self) -> int:
        return len(self.file_list)

    def _grids(self, path: Path):
        import scipy.io as sio
        mat = sio.loadmat(path)
        if "H" not in mat or mat["H"].shape[-1] < 2:
            raise ValueError("Invalid .mat file format: missing required data")
        return (torch.tensor(mat["H"][:, :, 0], dtype=torch.cfloat), torch.tensor(mat["H"][:, :, 1], dtype=torch.cfloat))

    def __getitem__(self, idx: int):
        if not 0 <= idx < len(self):
            raise IndexError(f"Index {idx} out of range for dataset of size {len(self)}")
        path = self.file_list[idx]
        try:
            h_ideal, ls = self._grids(path)
            if self.raw:
                h_est = ls
            else:   # host form of the extraction, one file at a time (dataset.py:118-139)
                h_est = ls[ls != 0]
                expected = self.pilot_params.num_scs * self.pilot_params.num_symbols
                if h_est.numel() != expected:
                    raise ValueError(f"Expected {expected} pilot values, got {h_est.numel()}")
                h_est = h_est.view(self.pilot_params.num_scs, self.pilot_params.num_symbols)
            meta = extract_values(path.name)
            if self.transform:
                h_est, h_ideal = self.transform(h_est), self.transform(h_ideal)
            return h_est, h_ideal, meta
        except Exception as e:
            raise ValueError(f"Error processing file {path}: {e}")


def collate_on_device(batch, pilot_size: Tuple[int, int], device: Union[str, torch.device] = "cuda"):
    """Collate items of a ``MatDataset(raw=True)``: one host->device copy of the stacked sparse grids, then one
    ``aft_extract_pilots`` launch.  Returns (pilots [B, ps, pt] c64 on `device`, truth [B, scs, symbols] c64 on
    `device`, metadata collated like torch's default collate: five float32 [B, 1] tensors and [tuple of channel names])."""
    grids = torch.stack([b[0] for b in batch]).to(device, non_blocking=True)
    truth = torch.stack([b[1] for b in batch]).to(device, non_blocking=True)
    meta = [torch.stack([b[2][k] for b in batch]) for k in range(5)] + [[tuple(b[2][5][0] for b in batch)]]
    return extract_pilots(grids, pilot_size), truth, tuple(meta)


# The reference's condition grids (README.md:184-207): SNR dB, delay spread ns, maximum Doppler shift Hz.  The kernel draws
# grid indices; these are the values it maps them to.
SNR_GRID = tuple(float(v) for v in range(0, 31, 5))
DS_GRID = tuple(float(v) for v in range(50, 351, 50))
DOP_GRID = tuple(float(v) for v in range(200, 1401, 200))


class SyntheticChannels:
    """Doubly-selective channels and their noisy LS pilots, generated on the GPU (``include/aft.h``, "Synthetic
    channels": 8 exponential-delay taps, Jakes-type Doppler, 15 kHz subcarriers, 14 symbols per ms, pilots at symbols
    2 and 11).

    ``system_config``: a :class:`SystemConfig` (or its dict) giving the grid and pilot extents.  ``seed``: 64-bit
    integer naming the stream.  ``conditions``: ``None`` draws each sample's (SNR, delay spread, Doppler) from the
    reference's 7 x 7 x 7 grid; ``(snr_db, delay_spread_ns, doppler_hz)`` fixes one condition for every sample.

    :meth:`batch` ``(sample0, n)`` returns samples ``sample0 .. sample0 + n - 1`` of the stream as ``(pilots, meta,
    truth)`` on the device, ``meta`` in the form of :func:`collate_on_device`, ready for ``model(pilots, meta)``,
    ``ShardedTrainer.step`` and the evaluator.  A sample depends on the seed, its index and its condition only, so a
    data-parallel rank calls ``batch(step * global_batch + lo, hi - lo)`` with its ``shard_range`` and gets exactly its
    rows of ``batch(step * global_batch, global_batch)``."""

    def __init__(self, system_config, seed: int, conditions: Optional[Tuple[float, float, float]] = None,
                 device: Union[str, torch.device] = "cuda") -> None:
        from .config import SystemConfig
        if not isinstance(system_config, SystemConfig):
            system_config = SystemConfig(**system_config)
        self.system_config = system_config
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError(f"seed must be in [0, 2^64), got {seed}")
        self.seed = seed
        if conditions is not None:
            snr, ds, dop = (float(v) for v in conditions)
            if not all(math.isfinite(v) for v in (snr, ds, dop)) or ds <= 0 or dop < 0:
                raise ValueError(f"conditions must be finite with delay spread > 0 and Doppler >= 0, got {conditions}")
            conditions = (snr, ds, dop)
        self.conditions = conditions
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("adafortitran_b200 has no CPU fallback: SyntheticChannels generates on a CUDA device")
        o, p = system_config.ofdm, system_config.pilot
        self._cfg = _capi.AftConfig(num_scs=o.num_scs, num_symbols=o.num_symbols, pilot_scs=p.num_scs,
                                    pilot_symbols=p.num_symbols)

    def batch(self, sample0: int, n: int):
        """``(pilots c64 [n, pilot_scs, pilot_symbols], meta, truth c64 [n, num_scs, num_symbols])`` on the device.
        ``meta`` = (sample index, snr, delay spread, Doppler, pilot spacing: five float32 ``[n, 1]`` tensors,
        ``[("synthetic",) * n]``)."""
        sample0, n = int(sample0), int(n)
        o, p = self.system_config.ofdm, self.system_config.pilot
        dev = self.device
        pilots = torch.empty((n, p.num_scs, p.num_symbols), dtype=torch.complex64, device=dev)
        truth = torch.empty((n, o.num_scs, o.num_symbols), dtype=torch.complex64, device=dev)
        if self.conditions is None:
            cond = torch.empty((3, n), dtype=torch.float32, device=dev)
        else:
            cond = torch.tensor(self.conditions, dtype=torch.float32, device=dev)[:, None].repeat(1, n)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t.numel() else None
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _capi.check(_capi.lib().aft_synthetic_channels(
                C.byref(self._cfg), self.seed, sample0, n, ptr(cond[0]), ptr(cond[1]), ptr(cond[2]),
                int(self.conditions is None), ptr(pilots), ptr(truth), C.c_void_p(stream)))
        index = torch.arange(sample0, sample0 + n, dtype=torch.int64, device=dev).to(torch.float32)
        spacing = torch.full((n,), float(o.num_scs // p.num_scs), dtype=torch.float32, device=dev)
        meta = tuple(t.reshape(n, 1) for t in (index, cond[0], cond[1], cond[2], spacing)) + ([("synthetic",) * n],)
        return pilots, meta, truth
