"""CPU, world_size 2, gloo: the host-side logic of ``distributed.ShardedTrainer`` (seed broadcast, shard checks, loss
normalisation, gradient all-reduce) over a small fp64 stand-in for the estimators, and the shard masks of
``tests/dp_masks.py``."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch import nn

from adafortitran_b200 import distributed as D
from oracle import train_ref as T
from tests.dp_masks import masks_for

GLOBAL = 5          # unequal shards over 2 ranks: [0, 3) and [3, 5)


class StandIn(nn.Module):
    """fp64 complex map [b, 3, 2] -> [b, 4, 2] with the estimators' training keywords: per-(global sample, part) dropout
    drawn from ``dropout_seed`` and ``sample_offset + b``, so a wrong offset or seed changes the gradients."""

    trainable = True
    precision = "fp32"

    def __init__(self, init_seed):
        super().__init__()
        g = torch.Generator().manual_seed(init_seed)
        self.lin = nn.Linear(6, 8).double()
        with torch.no_grad():
            self.lin.weight.copy_(torch.randn(8, 6, generator=g, dtype=torch.float64))
            self.lin.bias.copy_(torch.randn(8, generator=g, dtype=torch.float64))
        self.register_buffer("scale", torch.full((1,), 1.0 + init_seed, dtype=torch.float64))
        self.device = torch.device("cpu")
        self.seeds = []

    def forward(self, pilots, meta=None, *, sample_offset=0, dropout_seed=None):
        self.seeds.append(dropout_seed)
        n = pilots.shape[0]
        masks = []
        for b in range(n):
            g = torch.Generator().manual_seed(int(dropout_seed) ^ (sample_offset + b) * 0x9E3779B1)
            masks.append((torch.rand(2, 8, generator=g) >= 0.25).double() / 0.75)
        m = torch.stack(masks) if masks else torch.zeros(0, 2, 8, dtype=torch.float64)
        re = self.lin(pilots.real.reshape(n, 6)) * m[:, 0] * self.scale
        im = self.lin(pilots.imag.reshape(n, 6)) * m[:, 1] * self.scale
        return torch.complex(re, im).reshape(n, 4, 2)


def _data():
    g = torch.Generator().manual_seed(11)
    pilots = torch.complex(torch.randn(GLOBAL, 3, 2, generator=g, dtype=torch.float64),
                           torch.randn(GLOBAL, 3, 2, generator=g, dtype=torch.float64))
    truth = torch.complex(torch.randn(GLOBAL, 4, 2, generator=g, dtype=torch.float64),
                          torch.randn(GLOBAL, 4, 2, generator=g, dtype=torch.float64))
    return pilots, truth


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        model = StandIn(init_seed=rank)                 # replicas start different: construction broadcasts rank 0's
        trainer = D.ShardedTrainer(model)
        p0 = {k: t.detach().clone() for k, t in model.state_dict().items()}
        pilots, truth = _data()
        lo, hi = D.shard_range(GLOBAL, rank, world)
        shard_error = None
        try:                                            # both ranks pass a wrong shard: nothing collective runs
            trainer.step(pilots[lo:hi - 1], None, truth[lo:hi - 1], GLOBAL)
        except ValueError as e:
            shard_error = str(e)
        torch.manual_seed(100 + rank)                   # a different default generator on every rank
        loss = trainer.step(pilots[lo:hi], None, truth[lo:hi], GLOBAL)
        grads = [p.grad.clone() for p in trainer.params]
        # the single-process reference: rank 0's replica, its seed, the whole batch, the reference's MSE
        torch.manual_seed(100)
        seed0 = int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())
        ref = StandIn(init_seed=0)
        est = ref(pilots, None, sample_offset=0, dropout_seed=seed0)
        ref_loss = nn.functional.mse_loss(torch.cat([est.real, est.imag], 1), torch.cat([truth.real, truth.imag], 1))
        ref_grads = torch.autograd.grad(ref_loss, list(ref.lin.parameters()))
        # the same, but every rank forwarding its shard at offset 0: must not reproduce the reference
        wrong = StandIn(init_seed=0)
        parts = [wrong(pilots[a:b], None, sample_offset=0, dropout_seed=seed0) for a, b in ((0, 3), (3, 5))]
        est_w = torch.cat(parts)
        wl = nn.functional.mse_loss(torch.cat([est_w.real, est_w.imag], 1), torch.cat([truth.real, truth.imag], 1))
        wrong_grads = torch.autograd.grad(wl, list(wrong.lin.parameters()))
        q.put(dict(rank=rank, shard_error=shard_error, seeds=model.seeds, seed0=seed0,
                   params={k: t.numpy() for k, t in p0.items()}, loss=float(loss), ref_loss=float(ref_loss),
                   grad_err=max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(grads, ref_grads)),
                   wrong_err=max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(wrong_grads, ref_grads))))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def results():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    try:
        [p.start() for p in procs]
        out = sorted((q.get(timeout=120) for _ in procs), key=lambda r: r["rank"])
        [p.join(timeout=60) for p in procs]
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
    return out


def test_unequal_shards_reproduce_global_batch_gradient(results):
    for r in results:
        assert r["grad_err"] <= 1e-12, r
        assert abs(r["loss"] - r["ref_loss"]) <= 1e-12 * r["ref_loss"], r
        assert r["wrong_err"] > 1e-3       # the offset matters: the check above can fail


def test_seed_broadcast_and_replicas_start_identical(results):
    # the rejected call drew no seed; the real step forwarded with rank 0's draw on both ranks
    assert [r["seeds"] for r in results] == [[results[0]["seed0"]]] * 2
    a, b = results[0]["params"], results[1]["params"]
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert a["scale"][0] == 1.0           # the buffer too: rank 0's value


def test_shard_size_mismatch_raises(results):
    for r in results:
        assert r["shard_error"] is not None and "holds samples" in r["shard_error"], r


def test_trainer_rejects_untrainable_or_bf16_model():
    m = StandIn(0)
    m.trainable = False
    with pytest.raises(ValueError, match="trainable"):
        D.ShardedTrainer(m)
    m.trainable, m.precision = True, "bf16"
    with pytest.raises(ValueError, match="fp32"):
        D.ShardedTrainer(m)


def test_shard_masks_are_rows_of_global_batch():
    seed = 0x5EED_1234_ABCD
    for part in (0, 1):
        full = T.masks_for(seed, 5, part, 2, 0.1)          # the oracle's rule for a whole batch
        head = masks_for(seed, 5, part, 2, 0.1)
        tail = masks_for(seed, 3, part, 2, 0.1, first=2)
        for l in range(2):
            for s in range(4):
                assert torch.equal(head[l][s], full[l][s]), (part, l, s)
                assert torch.equal(tail[l][s], full[l][s][2:5]), (part, l, s)
