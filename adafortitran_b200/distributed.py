"""Multi-GPU plumbing: batch-sharded evaluation (:class:`ShardedEvaluator`) and data-parallel training
(:class:`ShardedTrainer`) over the GPUs of one node.

The forward pass has no cross-sample arithmetic (reference ``src/models/fortitran.py:184-233``), so the only
collectives of the path are the ones that follow it in the evaluator (SURVEY.md 8e): an all-gather of the
complex64 estimates and a SUM all-reduce of the error / power accumulators
(reference ``src/main/trainer.py:338-345``).  One process per GPU (``torchrun``).

Two implementations of the all-gather:

* :class:`PeerGather` (GPUs of one NVLink / NVSwitch node) -- **fused into the forward**: every rank owns a gather buffer
  in peer-visible device memory (``aft_peer_alloc`` -> CUDA IPC handle -> ``aft_peer_open`` on the other ranks), and the
  kernel that produces the estimates stores each 16-byte vector into all of them while it computes the next samples.
  Nothing is left to do after the forward except the cross-rank synchronisation the error-sum all-reduce provides.
* :func:`gather_estimates` -- plain ``all_gather_into_tensor`` (NCCL on GPUs, gloo in the CPU tests): the serial baseline
  the fused path is measured against, and the fallback when peer memory cannot be mapped.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(batch: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced shard ``[lo, hi)`` of ``batch`` samples for ``rank`` (first ``batch % world`` ranks get one more)."""
    if batch < 0 or world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad shard request batch={batch} rank={rank} world={world}")
    base, extra = divmod(batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def gather_estimates(local: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather complex64 shards ``[b_r, scs, sym]`` into ``[sum b_r, scs, sym]`` (rank order).

    Equal shards use one ``all_gather_into_tensor``; unequal shards (``shard_range`` with ``batch % world != 0``) are
    padded to the largest shard for the collective and trimmed afterwards."""
    if not torch.is_complex(local):
        raise TypeError("estimates must be complex")
    world = dist.get_world_size(group)
    local = local.contiguous()
    sizes = [torch.zeros(1, dtype=torch.int64, device=local.device) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device), group=group)
    sizes = [int(s.item()) for s in sizes]
    if len(set(sizes)) == 1:
        out = torch.empty((world * local.shape[0], *local.shape[1:]), dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(torch.view_as_real(out), torch.view_as_real(local), group=group)
        return out
    big = max(sizes)
    padded = torch.zeros((big, *local.shape[1:]), dtype=local.dtype, device=local.device)
    padded[:local.shape[0]] = local
    out = torch.empty((world * big, *local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(torch.view_as_real(out), torch.view_as_real(padded), group=group)
    return torch.cat([out[r * big:r * big + n] for r, n in enumerate(sizes)], dim=0)


def reduce_error_sums(sums: torch.Tensor, group=None) -> torch.Tensor:
    """SUM all-reduce of ``[sum |est - truth|^2, sum |truth|^2, ...]`` accumulators (fp64), in place."""
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    return sums


def mse_db_from_sums(sums: torch.Tensor, count: int) -> float:
    """The reference's reported metric, ``to_db(2 * MSELoss(cat(re, im)))`` == 10 log10(sum|e|^2 / count)."""
    return float(10.0 * torch.log10(sums[0] / count))


class _DevArray:
    """Raw device memory exposed through ``__cuda_array_interface__`` so torch can view it without copying."""

    def __init__(self, ptr: int, nfloats: int):
        self.__cuda_array_interface__ = {"shape": (nfloats,), "typestr": "<f4", "data": (ptr, False), "version": 3,
                                         "strides": None}


class PeerGather:
    """Gather buffers of the fused all-gather: ``[world * rows_per_rank, scs, symbols]`` complex64 on every rank.

    Construction is collective over ``group`` (all ranks on one node, one GPU each).  ``forward(..., gather=pg)`` of the
    estimators then writes this rank's estimates into rows ``[rank * rows_per_rank + row0, ...)`` of every rank's buffer.
    After the forward the caller must synchronise the ranks on the stream (``reduce_error_sums`` does) before reading
    :attr:`gathered`.
    """

    def __init__(self, rows_per_rank: int, grid: Tuple[int, int], device: torch.device, group=None):
        from . import _capi
        self.group = group
        self._dist = dist.is_available() and dist.is_initialized()
        self.world, self.rank = (dist.get_world_size(group), dist.get_rank(group)) if self._dist else (1, 0)
        if not 1 <= self.world <= 8:
            raise ValueError(f"PeerGather supports 1..8 ranks of one node, got {self.world}")
        self.rows_per_rank, self.grid, self.device = int(rows_per_rank), tuple(grid), torch.device(device)
        self.row0 = 0
        self.force_staging = False
        self._lib = _capi.lib()
        pix = self.grid[0] * self.grid[1]
        nbytes = self.world * self.rows_per_rank * pix * 8
        handle = (C.c_ubyte * 64)()
        ptr = C.c_void_p()
        with torch.cuda.device(self.device):
            _capi.check(self._lib.aft_peer_alloc(max(nbytes, 16), C.byref(ptr), handle))
            self._local_ptr = ptr.value
            handles: List[Optional[bytes]] = [None] * self.world
            if self.world > 1:
                dist.all_gather_object(handles, bytes(handle), group=group)
            self._ptrs: List[int] = []
            self._opened: List[int] = []
            for r, hb in enumerate(handles):
                if r == self.rank:
                    self._ptrs.append(self._local_ptr)
                    continue
                buf = (C.c_ubyte * 64).from_buffer_copy(hb)
                p = C.c_void_p()
                _capi.check(self._lib.aft_peer_open(buf, C.byref(p)))
                self._ptrs.append(p.value)
                self._opened.append(p.value)
        flat = torch.as_tensor(_DevArray(self._local_ptr, self.world * self.rows_per_rank * pix * 2), device=self.device)
        self.gathered = torch.view_as_complex(flat.view(self.world * self.rows_per_rank, self.grid[0], self.grid[1], 2))
        if self.world > 1:
            dist.barrier(group=group)    # every rank has mapped every buffer before anybody stores into it

    def local_rows(self, batch: int) -> torch.Tensor:
        lo = self.rank * self.rows_per_rank + self.row0
        return self.gathered[lo:lo + batch]

    def check(self, model, batch: int) -> None:
        if tuple(model.ofdm_size) != self.grid:
            raise ValueError(f"gather buffers were built for a {self.grid} grid, the model produces {tuple(model.ofdm_size)}")
        if model.device != self.device:
            raise ValueError(f"gather buffers live on {self.device}, the model on {model.device}")
        if self.row0 + batch > self.rows_per_rank:
            raise ValueError(f"rows [{self.row0}, {self.row0 + batch}) exceed rows_per_rank {self.rows_per_rank}")

    def plan(self):
        from . import _capi
        g = _capi.AftGather()
        for r in range(self.world):
            g.peer_out[r] = self._ptrs[r]
        g.world, g.rank, g.rows_per_rank, g.row0 = self.world, self.rank, self.rows_per_rank, self.row0
        return g

    def close(self) -> None:
        if getattr(self, "_local_ptr", None) is None:
            return
        torch.cuda.synchronize(self.device)
        if self.world > 1 and dist.is_initialized():
            dist.barrier(group=self.group)     # nobody is still storing into a buffer that is about to go away
        for p in self._opened:
            self._lib.aft_peer_close(C.c_void_p(p))
        self.gathered = None
        self._lib.aft_peer_free(C.c_void_p(self._local_ptr))
        self._local_ptr, self._opened = None, []


class ShardedEvaluator:
    """Batch-sharded evaluation step over the ranks of one node (the multi-GPU form of the reference's
    ``ModelEvaluator._evaluate_dataloader`` body, ``src/main/trainer.py:328-347``): forward of the local shard, estimates
    of all ranks gathered on every rank, error / power sums reduced over the ranks.

    ``mode="peer"``: fused all-gather (:class:`PeerGather`; also used with a single rank, where the gather buffer is just
    the output buffer), ``mode="nccl"``: forward, then ``all_gather_into_tensor`` (the serial baseline).
    """

    def __init__(self, model, rows_per_rank: int, mode: str = "peer", group=None):
        if mode not in ("peer", "nccl"):
            raise ValueError("mode must be 'peer' or 'nccl'")
        self.model, self.rows_per_rank, self.mode, self.group = model, int(rows_per_rank), mode, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.peer = PeerGather(rows_per_rank, model.ofdm_size, model.device, group) if mode == "peer" else None
        self.sums = torch.zeros(2, dtype=torch.float64, device=model.device)

    def step(self, pilots, meta_data, truth_local: Optional[torch.Tensor] = None, host_out: Optional[torch.Tensor] = None):
        """One evaluation step on this rank's shard.  ``pilots`` / ``meta_data`` live on the device or on the host; host
        inputs go through ``forward_host`` (chunked copies overlapped with compute), which also delivers the local
        estimates to ``host_out`` (pinned CPU complex64).  Returns ``(gathered, sums)``: the estimates of all ranks
        ``[world * rows_per_rank, scs, sym]`` on the device -- valid for stream-ordered consumers once the all-reduce has
        run -- and the reduced ``[sum|est-truth|^2, sum|truth|^2]`` (fp64, device)."""
        from . import _capi
        model = self.model
        batch = pilots.shape[0]
        on_host = pilots.device.type == "cpu"
        if self.peer is not None:
            if on_host:
                model.forward_host(pilots, meta_data, out=host_out, gather=self.peer)
            else:
                model(pilots, meta_data, gather=self.peer)
                if host_out is not None:
                    host_out.copy_(self.peer.local_rows(batch), non_blocking=True)
            local, gathered = self.peer.local_rows(batch), self.peer.gathered
        else:
            if on_host:
                pilots = pilots.to(model.device, non_blocking=True)
                if meta_data is not None:
                    meta_data = tuple(t.to(model.device, non_blocking=True) if torch.is_tensor(t) else t for t in meta_data)
            local = model(pilots, meta_data)
            if host_out is not None:
                host_out.copy_(local, non_blocking=True)
            gathered = gather_estimates(local, self.group) if self.world > 1 else local
        self.sums.zero_()
        if truth_local is not None and batch > 0:
            st = torch.cuda.current_stream(model.device).cuda_stream
            _capi.check(_capi.lib().aft_error_sums(C.c_void_p(local.data_ptr()), C.c_void_p(truth_local.data_ptr()),
                                                  local.numel(), C.c_void_p(self.sums.data_ptr()), C.c_void_p(st)))
        if self.world > 1:
            reduce_error_sums(self.sums, self.group)     # also the cross-rank ordering point of the fused gather
        return gathered, self.sums

    def close(self) -> None:
        if self.peer is not None:
            self.peer.close()
            self.peer = None


class ShardedTrainer:
    """Data-parallel training step over the ranks of ``group`` (one process and one GPU each): the training counterpart
    of :class:`ShardedEvaluator`.

    Each rank holds a replica of ``model`` (``trainable = True``, ``precision = "fp32"``) and the shard
    ``shard_range(global_batch, rank, world)`` of every global batch.  :meth:`step` makes the ranks compute, together,
    exactly what one call over the global batch computes:

    * dropout: one seed per step, drawn on rank 0 from its default generator (as a single-GPU call draws it) and
      broadcast; every rank forwards with ``sample_offset`` = its first global sample, so each sample gets the masks it
      gets in a single call over the global batch, whatever ``torch.manual_seed`` each rank ran;
    * loss: the reference's ``MSELoss`` over ``cat(re, im)`` of the global batch.  Each rank normalises its sum of
      squared errors by the global batch, so unequal shards weigh every sample the same;
    * gradients: one SUM all-reduce of one flat buffer holding every parameter gradient (and the loss).

    Construction is collective: it broadcasts the parameters and buffers of rank 0, so the replicas start identical.
    The caller keeps the optimizer: identical gradients on identical parameters give identical updates on every rank.
    """

    def __init__(self, model, group=None):
        if not getattr(model, "trainable", False):
            raise ValueError("ShardedTrainer needs a model with trainable = True")
        if getattr(model, "precision", None) != "fp32":
            raise ValueError(f"ShardedTrainer trains on the fp32 path only, the model has precision "
                             f"{getattr(model, 'precision', None)!r}")
        self.model, self.group = model, group
        self._dist = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if self._dist else 1
        self.rank = dist.get_rank(group) if self._dist else 0
        self._src = dist.get_global_rank(group, 0) if self._dist and group is not None else 0
        # NCCL moves device tensors, gloo host tensors
        self._comm_device = model.device if self._dist and dist.get_backend(group) == "nccl" else torch.device("cpu")
        self.params = [p for p in model.parameters() if p.requires_grad]
        if self.world > 1:
            with torch.no_grad():
                for t in list(model.parameters()) + list(model.buffers()):
                    buf = t.detach().to(self._comm_device, copy=True)
                    dist.broadcast(buf, src=self._src, group=group)
                    t.copy_(buf)     # in place through autograd's view: bumps the version, so packed copies refresh

    def _seed(self) -> int:
        seed = torch.randint(0, 2 ** 62, (), dtype=torch.int64) if self.rank == 0 else torch.zeros((), dtype=torch.int64)
        if self.world > 1:
            seed = seed.to(self._comm_device)
            dist.broadcast(seed, src=self._src, group=self.group)
        return int(seed.item())

    def step(self, pilots_local, meta_local, truth_local: torch.Tensor, global_batch: int) -> torch.Tensor:
        """Forward and backward of this rank's shard of a ``global_batch``-sample batch, then the gradient all-reduce.

        ``pilots_local`` / ``meta_local`` / ``truth_local`` (complex ``[b, scs, symbols]``) hold samples ``[lo, hi)`` of
        ``shard_range(global_batch, rank, world)``; a rank with an empty shard passes empty tensors and still takes part.
        Afterwards every parameter's ``.grad`` holds the gradient of the global batch's loss (earlier ``.grad`` contents
        are discarded).  Returns that loss (a 0-dim tensor, the same on every rank)."""
        model = self.model
        lo, hi = shard_range(int(global_batch), self.rank, self.world)
        if pilots_local.shape[0] != hi - lo or truth_local.shape[0] != hi - lo:
            raise ValueError(f"rank {self.rank} of {self.world} holds samples [{lo}, {hi}) of a {global_batch}-sample batch, "
                             f"got {pilots_local.shape[0]} pilots and {truth_local.shape[0]} truths")
        seed = self._seed()
        model.zero_grad(set_to_none=True)
        est = model(pilots_local, meta_local, sample_offset=lo, dropout_seed=seed)
        truth = truth_local.to(est.device)
        if tuple(truth.shape) != tuple(est.shape):
            raise ValueError(f"truth_local has shape {tuple(truth.shape)}, the estimates {tuple(est.shape)}")
        err = est - truth
        count = 2 * int(global_batch) * est.shape[1] * est.shape[2]
        loss = torch.cat([err.real, err.imag], 1).pow(2).sum() / max(count, 1)
        loss.backward()
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in self.params]
        flat = torch.cat([g.reshape(-1) for g in grads] + [loss.detach().reshape(1).to(grads[0].dtype)])
        if self.world > 1:
            wire = flat.to(self._comm_device)
            dist.all_reduce(wire, op=dist.ReduceOp.SUM, group=self.group)
            flat = wire.to(flat.device)
        off = 0
        for p in self.params:
            p.grad = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        return flat[off]
