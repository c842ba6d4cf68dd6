"""Reference for the training path: the dropout mask rule and a differentiable fp64 restatement of the forward.

TEST INFRASTRUCTURE ONLY (same rules as ``aft_oracle.py``): imported by ``tests/`` and ``tools/``, never by the
product package.

* :func:`philox4x32_10` / :func:`keep_mask` restate the dropout rule of ``include/aft.h`` in numpy.
* :func:`real_pass` / :func:`forward` restate one real-valued pass / the complex forward of the estimators over
  explicit torch ops, with the four dropout sites of ``nn.TransformerEncoderLayer`` taking explicit masks.  The
  parameters are a dict keyed like ``BaseFortiTranEstimator._weight_tensors()`` (``up_w``, ``enh_w0``, ``L0_in_w``,
  ...); :func:`params_from_state_dict` builds it from a reference ``state_dict``.  With all masks one it is pinned to
  ``TorchPort`` (forward and autograd gradients, fp64) by ``tests/test_train_cpu.py``.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
S, D, HEADS, DH, FF = 280, 128, 4, 32, 256


def philox4x32_10(ctr, key):
    """Philox4x32-10 on uint32 arrays: ``ctr`` is a sequence of four arrays (or ints), ``key`` of two."""
    c = [np.asarray(x, dtype=np.uint64) for x in ctr]
    k = [np.uint64(key[0]), np.uint64(key[1])]
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k[0]) & mask, p1 & mask, ((p0 >> np.uint64(32)) ^ c[3] ^ k[1]) & mask, p0 & mask]
        k = [(k[0] + np.uint64(W0)) & mask, (k[1] + np.uint64(W1)) & mask]
    return [x.astype(np.uint32) for x in c]


def threshold(p: float) -> int:
    return int(np.floor(np.float64(np.float32(p)) * 2.0 ** 32))


def keep_mask(seed: int, seq: int, layer: int, site: int, shape, p: float) -> np.ndarray:
    """Boolean keep mask of ``shape`` (element i = the row-major flat index) for one (sequence, layer, site)."""
    n = int(np.prod(shape))
    i4 = np.arange((n + 3) // 4, dtype=np.uint64)
    z = np.zeros_like(i4)
    w = philox4x32_10([i4, z + np.uint64(seq), z + np.uint64((layer << 8) | site), z],
                      (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    words = np.stack(w, axis=1).reshape(-1)[:n]
    return (words >= np.uint32(threshold(p)) if threshold(p) > 0 else np.ones(n, bool)).reshape(shape)


SITE_SHAPES = {0: (HEADS, S, S), 1: (S, D), 2: (S, FF), 3: (S, D)}


def masks_for(seed: int, samples: int, part: int, layers: int, p: float) -> List[List[torch.Tensor]]:
    """masks[layer][site]: float64 [samples, *SITE_SHAPES[site]] of one pass (part 0 = real, 1 = imaginary)."""
    return [[torch.from_numpy(np.stack([keep_mask(seed, 2 * b + part, l, s, SITE_SHAPES[s], p) for b in range(samples)])
                              .astype(np.float64)) for s in range(4)] for l in range(layers)]


def params_from_state_dict(sd: Dict[str, np.ndarray], adaptive: bool, num_layers: int) -> Dict[str, torch.Tensor]:
    t = lambda k: torch.as_tensor(np.asarray(sd[k]))
    P = {"up_w": t("pilot_upsampler.weight"), "up_b": t("pilot_upsampler.bias")}
    for tag, name in (("enh", "initial_enhancer"), ("ref", "final_refiner")):
        for i, idx in enumerate((0, 2, 4, 6)):
            P[f"{tag}_w{i}"], P[f"{tag}_b{i}"] = t(f"{name}.conv_block.{idx}.weight"), t(f"{name}.conv_block.{idx}.bias")
    if adaptive:
        for n in ("snr", "ds", "dop"):
            for i, idx in enumerate((0, 2, 4)):
                P[f"{n}_w{i}"] = t(f"channel_adapter.{n}_encoder.{idx}.weight")
                P[f"{n}_b{i}"] = t(f"channel_adapter.{n}_encoder.{idx}.bias")
    te = "transformer_encoder."
    pos = [k for k in sd if k.endswith("position_embeddings") or k.endswith("positional_encoding.pe")][0]
    P.update(l1_w=t(te + "linear_1.weight"), l1_b=t(te + "linear_1.bias"), pos=t(pos),
             l2_w=t(te + "linear_2.weight"), l2_b=t(te + "linear_2.bias"))
    for l in range(num_layers):
        b = f"{te}transformer.layers.{l}."
        for tag, k in (("in_w", "self_attn.in_proj_weight"), ("in_b", "self_attn.in_proj_bias"),
                       ("out_w", "self_attn.out_proj.weight"), ("out_b", "self_attn.out_proj.bias"),
                       ("l1_w", "linear1.weight"), ("l1_b", "linear1.bias"), ("l2_w", "linear2.weight"),
                       ("l2_b", "linear2.bias"), ("n1_w", "norm1.weight"), ("n1_b", "norm1.bias"),
                       ("n2_w", "norm2.weight"), ("n2_b", "norm2.bias")):
            P[f"L{l}_{tag}"] = t(b + k)
    return P


def _convs(P, tag, x):
    for i in range(4):
        x = F.conv2d(x, P[f"{tag}_w{i}"], P[f"{tag}_b{i}"], padding=1)
        if i < 3:
            x = F.relu(x)
    return x


def real_pass(P: Dict[str, torch.Tensor], x: torch.Tensor, cond: Optional[Sequence[torch.Tensor]], masks, p: float,
              num_layers: int, activation: str = "gelu", grid=(120, 14), patch=(3, 2)) -> torch.Tensor:
    """One real-valued pass.  ``x``: [n, 24]; ``cond``: three [n, 1] tensors or None; ``masks[l][site]`` as
    :func:`masks_for` gives, or None for no dropout."""
    n = x.shape[0]
    (H, W), (ph, pw) = grid, patch
    img = F.linear(x, P["up_w"], P["up_b"]).view(n, 1, H, W)
    enh = _convs(P, "enh", img).squeeze(1)
    tok = enh.reshape(n, H // ph, ph, W // pw, pw).permute(0, 1, 3, 2, 4).reshape(n, -1, ph * pw)
    if cond is not None:
        zs = []
        for name, c in zip(("snr", "ds", "dop"), cond):
            h = F.relu(F.linear(c, P[f"{name}_w0"], P[f"{name}_b0"]))
            h = F.relu(F.linear(h, P[f"{name}_w1"], P[f"{name}_b1"]))
            zs.append(F.linear(h, P[f"{name}_w2"], P[f"{name}_b2"]).reshape(n, -1, 2))
        tok = torch.cat([tok] + zs, dim=2)
    h = F.linear(tok, P["l1_w"], P["l1_b"]) + P["pos"][:, : tok.shape[1], :]
    scale = 1.0 / (1.0 - p) if p > 0 else 1.0
    drop = lambda v, l, s: v if masks is None else v * masks[l][s].to(v.dtype) * scale
    act = F.gelu if activation == "gelu" else F.relu
    for l in range(num_layers):
        g = lambda k: P[f"L{l}_{k}"]
        qkv = F.linear(h, g("in_w"), g("in_b"))
        q, k, v = (qkv[..., i * D:(i + 1) * D].reshape(n, -1, HEADS, DH).transpose(1, 2) for i in range(3))
        a = torch.softmax((q / np.sqrt(DH)) @ k.transpose(-1, -2), dim=-1)
        o = (drop(a, l, 0) @ v).transpose(1, 2).reshape(n, -1, D)
        h = F.layer_norm(h + drop(F.linear(o, g("out_w"), g("out_b")), l, 1), (D,), g("n1_w"), g("n1_b"))
        f = F.linear(drop(act(F.linear(h, g("l1_w"), g("l1_b"))), l, 2), g("l2_w"), g("l2_b"))
        h = F.layer_norm(h + drop(f, l, 3), (D,), g("n2_w"), g("n2_b"))
    r = F.linear(h, P["l2_w"], P["l2_b"])
    rec = r.reshape(n, H // ph, W // pw, ph, pw).permute(0, 1, 3, 2, 4).reshape(n, H, W)
    return _convs(P, "ref", (enh + rec).unsqueeze(1)).squeeze(1)


def forward(P, pilots: torch.Tensor, cond, p: float, seed: Optional[int], num_layers: int, activation: str = "gelu",
            masks=None):
    """Complex forward [n, 120, 14] in the dtype of ``P``; masks from the Philox rule (``seed``) unless p == 0, or the
    ``[real, imaginary]`` pair of :func:`masks_for` results given as ``masks``."""
    n = pilots.shape[0]
    dt = P["up_w"].dtype
    x = pilots.reshape(n, -1)
    if masks is None:
        masks = [None, None] if p == 0 else [masks_for(seed, n, e, num_layers, p) for e in (0, 1)]
    c = None if cond is None else [torch.as_tensor(v).to(dt).reshape(n, 1) for v in cond]
    re = real_pass(P, x.real.to(dt), c, masks[0], p, num_layers, activation)
    im = real_pass(P, x.imag.to(dt), c, masks[1], p, num_layers, activation)
    return torch.complex(re, im)
