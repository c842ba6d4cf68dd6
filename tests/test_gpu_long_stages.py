"""The long-sequence AFT_BF16 encoder (``csrc/tc_long.cu``) kernel by kernel against fp64, read back from the caller's
workspace.

Every grid other than the reference default runs AFT_BF16 through ``tc_long.cu``: ``f32_to_ximg_kernel`` turns the
front end's fp32 rows into residual tile images, ``lin_block_kernel`` (persistent, ``min(tiles, SMs)`` CTAs) runs
out_proj, LN1, the FFN, LN2 and the next layer's in_proj, and ``attn_long_kernel`` streams 64-key tiles through a
4-stage bulk-copy ring with the padding keys of the last key tile masked and the output accumulator rescaled in TMEM
only when a row maximum grows by more than 8 (log2 units).  ``tests/test_gpu_generic_edges.py`` checks the path end to
end; an off-by-one padding mask at S1025 moves a layer's attention output by -59 dB per row, below the bf16 floor of
the output, and with seed-initialised weights no row ever rescales after its first key tile.  Here each kernel is
judged alone, and constructed weights make the masked, ragged and rescaled branches decide the result.

Workspace (``forward_chunk_generic`` / ``generic_floats_per_chunk`` in ``aft_api.cu``, ``tc_long_encoder``), for the
last internal chunk of ``nseq = 2 b`` sequences, ``seq = 2 sample + part``, ``T = ceil(S / 128)`` row tiles:

* ``enh``: fp32 ``[nseq][pix]`` at offset 0;
* ``hbuf``: fp32 ``[nseq S][128]`` after ``align_up(nseq pix, 64)`` floats: the front end's h0, then the last layer's
  output;
* the tc_long region after ``align_up(nseq S 128, 64)`` more floats, its base rounded up to 1024 bytes of the absolute
  address: ``ximg``, ``aimg`` (``nseq T`` x 32,768 B: 2 K-chunks x 128 rows x 128 B, unit ``u ^ (r & 7)``), then
  ``q``, ``k``, ``v`` (``nseq T 4`` x 8,192 B, head tile ``(seq 4 + g) T + tile``: 128 rows x 64 B, unit
  ``u ^ ((r >> 1) & 3)``).  Q carries ``qscale = log2(e) / sqrt(32)``, folded into the weights and the bias in fp32
  before the bf16 rounding.

``lin_block_kernel`` stores its new residual tile to ``ximg`` only when it also runs the next layer's in_proj, so a
forward of depth ``l + 1`` leaves layer ``l``'s input ``X_l`` (bf16, ``ximg``), its Q / K / V, its attention output
(``aimg``) and its output (fp32, ``hbuf``).  Each geometry is run with the same weights truncated to depth 1 ... L, and
every stage is compared with fp64 fed with the GPU's own inputs of that stage:

===========  ====================================================  ==============================================
stage        reference                                             figure
===========  ====================================================  ==============================================
h0           ``linear_1([patchify(enh) | adapter]) + pos`` from    relative error power per row (dB); padding rows
             the GPU's ``enh`` (front end + ``f32_to_ximg``)       exactly zero; constructed weights: bit-exact
in_proj      ``X_l`` times ``bf16(W qscale)`` plus the fp32 bias   every element, padding rows included, within one
                                                                   bf16 ulp plus ``2^-16 sum |x w|`` (fp32
                                                                   accumulation of 128 products)
attention    ``softmax2(Q K^T) V`` over the S valid keys, from     relative error power per query row (dB), worst
             the decoded bf16 Q / K / V                            per head, over full row tiles and over the
                                                                   ragged last row tile
row block    out_proj + residual, LN1, FFN (erf GELU / relu),      relative error power per row of ``hbuf`` (dB)
             LN2, from the decoded ``aimg`` and ``X_l``
layout       ``X_l`` of depth l + 1 == ``bf16_rn(hbuf)`` of depth l  bit-exact on every valid row
===========  ====================================================  ==============================================

The fp64 attention is the kernel's own tile loop (``attention``): running maximum per row, rescale when any row of the
warp outgrows its reference by more than 8, so the same code counts the rows rescaled after key tile 0.

Constructed weights (FortiTran, one layer, ``linear_1 = 0``, so ``X_0`` is the positional table on valid rows and zero
on padding rows): positions carry ``t >> 6``, ``t & 63``, ``(-1)^t`` and 1, all exact in bf16; every head scores
``Q K = +-(16 t - 131072)``, the sign that of the query row.  Even query rows see scores rising by 16 per key and 1024
per key tile, so they rescale at every tile (at S = 65 too, where the last tile holds one key) and the last valid key
takes all but 2^-16 of the weight; odd rows of the same warps see falling
scores and take f = 1 inside the warp's rescale.  Padding keys (``K = b_k = 0``) score 0, above every valid key of an
even row, so one padding key let through takes all the weight.  V carries ``t & 63``, ``(-1)^t``, ``(t >> 6) / 8`` and
``g + 1``, distinct per token and head.

Cases (natural = seed-initialised, as in the generic-edges geometries; the batch ``B = SMs // T + 12`` makes every
``lin_block_kernel`` CTA run at least two tiles):

======  =====  ===  ===  ======================  ============================================================
id      S      T    nkt  weights, layers         edge
======  =====  ===  ===  ======================  ============================================================
S1      1      1    1    FortiTran relu, 1       qkv-only launch, then the last launch; 127 padding rows
S65     65     1    2    Ada, 2                  one valid key in the last key tile
S129    129    2    3    FortiTran sinusoidal 2  ragged second row tile
S257    257    3    5    FortiTran relu, 3       middle launches, the ring wraps
S1025   1025   9    17   FortiTran, 2            the ring wraps four times
C5      7644   60   120  Ada, 6 (config 5)       2 samples: 240 row tiles on 148 CTAs (persistent second pass)
K65     65     1    2    constructed, 1          mask and last key decide the result
K1025   1025   9    17   constructed, 1          ring wraps, rescale at every tile
K7644   7644   60   120  constructed, 1          ring wraps 30 times, 28 valid keys in the last tile
======  =====  ===  ===  ======================  ============================================================

Fault table (``test_fault_table``, CPU, fp64, at layer 0 of S65, S1025, K65 and K1025 with enough sequences that
row tiles lie past 148): each plausible fault is restated where the kernel could make it and must move its stage's
figure by more than the gate plus ``FAULT_MARGIN_DB`` to count as caught (layout: any row different).  Caught by the
constructed cases: padding mask off by one (0 dB) or removed, last valid key dropped (+25 dB), key tile j reading ring
slot j - 4's stale tile (K1025, -17 dB), O not rescaled (+27 / +49 dB), head g's output in head g^1's columns, the
second persistent tile of a ``lin_block_kernel`` CTA using its first tile's attention image (K1025), LayerNorm
statistics over one 64-column half.  With natural weights a removed mask, the head swap, LayerNorm halves and a stale
residual tile stored by a middle launch are caught at S65 and S1025, the dropped last key and the second-tile image at
S65; the off-by-one mask, the ring and the rescale faults are not (``INVISIBLE``).
"""
import math
import subprocess
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import aft_oracle as O
from tests import util

D, NH, DH = 128, 4, 32
KT, RING, THRESHOLD = 64, 4, 8.0            # keys per key tile, ring stages, rescale threshold (log2 units)
TILE_IMG, HEAD_TILE = 32768, 8192
QSCALE = np.float32(np.float32(1.4426950408889634) / np.sqrt(np.float32(DH)))   # host-side fp32, as tc_weights_pack
SMS_B200 = 148
ACC_ALLOW = 2.0 ** -16                      # fp32 accumulation allowance of the in_proj check, times sum |x w|

# Gates per weight family: the worst figure measured on a B200 (1000 W power limit) over every layer of every case of
# the family, plus about 3 dB.  Measured, natural: h0 -53.2 dB (C5); attention -46.1 dB (S65 layer 1; -46.5 C5 layer 0,
# -50.7 ... -54.3 elsewhere); row block -50.6 dB (C5 layer 0).  Constructed: attention -93.3 dB (the same worst row at
# all three); row block -50.1 dB (K7644).  in_proj: 0.4976 of the bound everywhere (every element correctly rounded);
# layout bit-exact, padding rows of X_0 zero.  Rows rescaled after key tile 0: natural 0, except C5 layer 0 (120,116 of
# 122,304 query rows: the raw metadata features); constructed 42,240 (K65), 114,912 (K1025), 61,152 (K7644).
GATES = {
    "natural": dict(h0_db=-50.0, att_db=-43.0, row_db=-47.5),
    "constructed": dict(h0_db=None, att_db=-90.0, row_db=-47.0),
}
FAULT_MARGIN_DB = 3.0

# id: (kind, layers, activation, positional table, grid, pilots, patch, batch or None for SMs // T + 12)
GEOMS = {
    "S1": ("forti", 1, "relu", "learnable", (3, 2), (1, 1), (3, 2), None),
    "S65": ("ada", 2, "gelu", "learnable", (65, 1), (13, 1), (1, 1), None),
    "S129": ("forti", 2, "gelu", "sinusoidal", (129, 2), (43, 2), (1, 2), None),
    "S257": ("forti", 3, "relu", "learnable", (514, 2), (257, 1), (2, 2), None),
    "S1025": ("forti", 2, "gelu", "learnable", (205, 10), (41, 5), (1, 2), None),
    "C5": ("ada", 6, "gelu", "learnable", (3276, 14), (1638, 2), (3, 2), 2),
    "K65": ("built", 1, "gelu", "learnable", (65, 1), (13, 1), (1, 1), None),
    "K1025": ("built", 1, "gelu", "learnable", (205, 10), (41, 5), (1, 2), None),
    "K7644": ("built", 1, "gelu", "learnable", (3276, 14), (1638, 2), (3, 2), 2),
}
CONSTRUCTED = ("K65", "K1025", "K7644")

RESULTS = {}   # (id, layer) -> figures, printed at the end of the module


def align_up(v, a):
    return (v + a - 1) // a * a


def geom_S(gid):
    grid, patch = GEOMS[gid][4], GEOMS[gid][6]
    return (grid[0] // patch[0]) * (grid[1] // patch[1])


# ---------------------------------------------------------------------------------------------------------------------
# workspace layout and decoders
# ---------------------------------------------------------------------------------------------------------------------

def ws_layout(nseq, S, pix, base):
    """Byte offsets (from the workspace start at absolute address ``base``) of the regions of the last internal chunk."""
    T = -(-S // 128)
    tiles = nseq * T
    hbuf = align_up(nseq * pix, 64) * 4
    img = hbuf + align_up(nseq * S * D, 64) * 4
    tc = align_up(base + img, 1024) - base
    region = tiles * TILE_IMG                   # = tiles x 4 heads x 8,192 B: every region a multiple of 1024
    return dict(T=T, tiles=tiles, hbuf=hbuf, img=img, ximg=tc, aimg=tc + region, q=tc + 2 * region,
                k=tc + 3 * region, v=tc + 4 * region, end=tc + 5 * region)


def _tile_index():
    """Element (row, col) of a residual / attention-output tile image -> index of its bf16."""
    r = np.arange(128)[:, None]
    c = np.arange(D)[None, :]
    return ((c >> 6) * 16384 + r * 128 + ((((c & 63) >> 3) ^ (r & 7)) << 4) + (c & 7) * 2) // 2


def _head_index():
    """Element (row, col) of a Q / K / V head tile -> index of its bf16."""
    r = np.arange(128)[:, None]
    c = np.arange(DH)[None, :]
    return (r * 64 + (((c >> 3) ^ ((r >> 1) & 3)) << 4) + (c & 7) * 2) // 2


TIDX, HIDX = _tile_index(), _head_index()


def _words_to_f32(w):
    return ((w.to(torch.int32) & 0xFFFF) << 16).view(torch.float32)


def decode_tiles(raw, nseq, T):
    """uint8 bytes of ``nseq T`` tile images -> float32 ``[nseq][128 T][128]``."""
    w = raw.view(torch.int16).reshape(nseq * T, TILE_IMG // 2)
    x = _words_to_f32(w[:, torch.as_tensor(TIDX, device=raw.device)])
    return x.reshape(nseq, T * 128, D)


def decode_heads(raw, nseq, T):
    """uint8 bytes of ``nseq 4 T`` head tiles -> float32 ``[nseq][4][128 T][32]``."""
    w = raw.view(torch.int16).reshape(nseq * NH * T, HEAD_TILE // 2)
    x = _words_to_f32(w[:, torch.as_tensor(HIDX, device=raw.device)])
    return x.reshape(nseq, NH, T * 128, DH)


def bf16_rn(x):
    return x.float().to(torch.bfloat16).double()


# ---------------------------------------------------------------------------------------------------------------------
# fp64 restatement (device-agnostic), with the faults of the fault table
# ---------------------------------------------------------------------------------------------------------------------

def tw(sd, device):
    return {k: torch.as_tensor(np.asarray(v, np.float64), device=device) for k, v in sd.items()}


def inproj_weights(sd, l, device):
    """The in_proj operands ``lin_block_kernel`` multiplies with: ``bf16(fl32(W_q qscale))``, ``bf16(W_k)``,
    ``bf16(W_v)`` and the fp32 bias with ``fl32(b_q qscale)`` (fp64 tensors)."""
    p = f"transformer_encoder.transformer.layers.{l}.self_attn"
    w = torch.as_tensor(np.asarray(sd[f"{p}.in_proj_weight"], np.float32), device=device)
    b = torch.as_tensor(np.asarray(sd[f"{p}.in_proj_bias"], np.float32), device=device)
    qs = torch.tensor(QSCALE, dtype=torch.float32, device=device)
    w = torch.cat([w[:D] * qs, w[D:]]).to(torch.bfloat16).double()
    b = torch.cat([b[:D] * qs, b[D:]]).double()
    return w, b


def split_heads(y):
    """``[n][R][384]`` -> q, k, v ``[n][4][R][32]``."""
    n, R = y.shape[:2]
    return tuple(y[..., i * D:(i + 1) * D].reshape(n, R, NH, DH).transpose(1, 2) for i in range(3))


def attention(q, k, v, S, fault=None):
    """``softmax2(q k^T) v`` over keys 0 .. S-1 (q already in log2 units), computed as ``attn_long_kernel`` walks it:
    64-key tiles, a running reference maximum per query row that moves only when some row of the row's warp (32
    consecutive rows) outgrows it by more than 8, the accumulator and the row sum rescaled then.  Returns the output
    ``[n][4][R][32]`` and ``rescaled`` ``[n][4][R]``: rows whose own maximum triggered a rescale after key tile 0."""
    n, h, R, _ = q.shape
    nkt = -(-S // KT)
    m_ref = torch.full((n, h, R), -math.inf, dtype=q.dtype, device=q.device)
    lsum = torch.zeros((n, h, R), dtype=q.dtype, device=q.device)
    o = torch.zeros_like(q)
    rescaled = torch.zeros((n, h, R), dtype=torch.bool, device=q.device)
    for j in range(nkt):
        src = j - RING if fault == "ring_stale" and j >= RING else j   # the slot still holds the tile of the last lap
        kj, vj = k[:, :, src * KT:(src + 1) * KT], v[:, :, src * KT:(src + 1) * KT]
        s = q @ kj.transpose(-1, -2)
        if j == nkt - 1:
            nvalid = S - j * KT + {"mask_off_by_one": 1, "mask_removed": KT, "last_key_dropped": -1}.get(fault, 0)
            s[..., max(nvalid, 0):] = -math.inf
        mt = s.amax(-1)
        grow = mt > m_ref + THRESHOLD
        warp = grow.reshape(n, h, R // 32, 32).any(-1).repeat_interleave(32, -1)
        if j > 0:
            rescaled |= grow
        mn = torch.where(warp, torch.maximum(m_ref, mt), m_ref)
        f = torch.where(warp, torch.exp2(m_ref - mn), torch.ones_like(m_ref))
        if not (fault == "no_rescale" and j > 0):
            o = o * f[..., None]
        lsum = lsum * f
        m_ref = mn
        p = torch.exp2(s - m_ref[..., None])
        lsum = lsum + p.sum(-1)
        o = o + p @ vj
    o = o / lsum[..., None]
    if fault == "head_swap":
        o = o[:, [1, 0, 3, 2]]
    return o, rescaled


def _ln(x, g, b, halves=False):
    if halves:                                   # statistics of each 64-column half alone
        return torch.cat([_ln(x[..., :64], g[:64], b[:64]), _ln(x[..., 64:], g[64:], b[64:])], -1)
    mu = x.mean(-1, keepdim=True)
    var = x.var(-1, unbiased=False, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * g + b


def row_block(W, l, x, a, act, fault=None, T=None):
    """out_proj + residual, LN1, FFN, LN2 of layer ``l`` on rows ``x`` with attention output ``a`` (``[n][R][128]``)."""
    p = f"transformer_encoder.transformer.layers.{l}"
    if fault == "second_tile_stale_aimg":        # tile ti >= SMs takes the image of the CTA's first tile ti - SMs
        n, R = a.shape[:2]
        t = a.reshape(n * T, 128, D).clone()
        t[SMS_B200:] = t[:-SMS_B200].clone()
        a = t.reshape(n, R, D)
    halves = fault == "ln_half_stats"
    h = _ln(x + F.linear(a, W[f"{p}.self_attn.out_proj.weight"], W[f"{p}.self_attn.out_proj.bias"]),
            W[f"{p}.norm1.weight"], W[f"{p}.norm1.bias"], halves)
    f = F.linear(h, W[f"{p}.linear1.weight"], W[f"{p}.linear1.bias"])
    f = F.gelu(f) if act == "gelu" else torch.relu(f)
    f = F.linear(f, W[f"{p}.linear2.weight"], W[f"{p}.linear2.bias"])
    return _ln(h + f, W[f"{p}.norm2.weight"], W[f"{p}.norm2.bias"], halves)


def long_layer(W, sd, l, x, S, act, fault=None):
    """One layer of the long path on padded rows ``x`` ``[n][128 T][128]`` (padding rows included, as the kernels run
    them), unrounded: returns the stage outputs and the residual tile the launch stores for the next layer."""
    T = x.shape[1] // 128
    w, b = inproj_weights(sd, l, x.device)
    q, k, v = split_heads(F.linear(x, w, b))
    o, rescaled = attention(q, k, v, S, fault)
    a = o.transpose(1, 2).reshape(x.shape)
    out = row_block(W, l, x, a, act, fault, T)
    stored = x if fault == "stale_residual_store" else out
    return dict(q=q, k=k, v=v, a=a, out=out, stored=stored, rescaled=rescaled)


# ---------------------------------------------------------------------------------------------------------------------
# figures
# ---------------------------------------------------------------------------------------------------------------------

def _db(num, den):
    return 10 * torch.log10(num / den)


def fig_rows(y, ref):
    """Relative error power per row (last dimension), dB."""
    return _db(((y - ref) ** 2).sum(-1) + 1e-300, (ref ** 2).sum(-1) + 1e-300)


def fig_inproj(got, x, w, b):
    """Worst ``|got - y| / (ulp_bf16(y) + 2^-16 sum |x w|)`` over every element, ``y`` the unrounded fp64 in_proj."""
    y = F.linear(x, w, b)
    allow = F.linear(x.abs(), w.abs(), b.abs()) * ACC_ALLOW
    ulp = torch.ldexp(torch.ones_like(y), torch.frexp(y)[1] - 8)
    return float(((got - y).abs() / (ulp + allow + 1e-300)).max())


def attention_figures(rows, S):
    """``rows`` ``[n][4][R]`` per-row dB -> worst over valid rows per head, over full row tiles and the last row tile."""
    v = rows[:, :, :S]
    last = (S - 1) // 128 * 128
    fig = {"att_db": float(v.max()), "att_head_db": [round(float(v[:, g].max()), 1) for g in range(NH)],
           "att_last_tile_db": float(v[:, :, last:].max())}
    if last > 0:
        fig["att_full_tiles_db"] = float(v[:, :, :last].max())
    return fig


# ---------------------------------------------------------------------------------------------------------------------
# weights
# ---------------------------------------------------------------------------------------------------------------------

def make_model(gid, num_layers, device, sd=None, seed=None):
    from adafortitran_b200 import AdaFortiTranEstimator, FortiTranEstimator, ModelConfig, SystemConfig
    kind, _, act, pos, grid, pilots, patch, _ = GEOMS[gid]
    S = geom_S(gid)
    ada = kind == "ada"
    extra = dict(channel_adaptivity_hidden_sizes=[7, 42, 2 * S], adaptive_token_length=6) if ada else {}
    if seed is not None:
        torch.manual_seed(seed)
    cls = AdaFortiTranEstimator if ada else FortiTranEstimator
    m = cls(SystemConfig(ofdm=dict(num_scs=grid[0], num_symbols=grid[1]), pilot=dict(num_scs=pilots[0], num_symbols=pilots[1])),
            ModelConfig(model_type="adafortitran" if ada else "fortitran", patch_size=patch, num_layers=num_layers, model_dim=128,
                        num_head=4, activation=act, max_seq_len=max(S, 8), pos_encoding_type=pos, device=device, **extra)).eval()
    if sd is not None:
        m.load_state_dict(util.to_torch({k: a for k, a in sd.items() if not any(f"layers.{i}." in k for i in range(num_layers, 8))}))
    return m


def constructed(sd, S):
    """Layer-0 weights whose attention is decided by the padding mask, the last key tile, the ring and the rescale."""
    sd = dict(sd)
    t = np.arange(S)
    pos = np.zeros_like(sd["transformer_encoder.positional_encoding.position_embeddings"])
    pos[0, :S, 0] = t >> 6
    pos[0, :S, 1] = t & 63
    pos[0, :S, 2] = 1 - 2 * (t & 1)
    pos[0, :S, 3] = 1
    sd["transformer_encoder.positional_encoding.position_embeddings"] = pos
    sd["transformer_encoder.linear_1.weight"] = np.zeros_like(sd["transformer_encoder.linear_1.weight"])
    sd["transformer_encoder.linear_1.bias"] = np.zeros_like(sd["transformer_encoder.linear_1.bias"])
    w = np.zeros((3 * D, D), np.float32)
    for g in range(NH):
        q0, k0, v0 = g * DH, D + g * DH, 2 * D + g * DH
        w[q0, 2] = w[q0 + 1, 2] = 128 / QSCALE         # Q = +-128 in both dimensions after the qscale fold
        w[k0, 0], w[k0, 3] = 8, -1024                  # K0 = 8 (t >> 6) - 1024
        w[k0 + 1, 1] = 1 / 8                           # K1 = (t & 63) / 8: Q K = +-128 (t / 8 - 1024)
        w[v0, 1], w[v0 + 1, 2], w[v0 + 2, 0], w[v0 + 3, 3] = 1, 1, 1 / 8, g + 1
    p = "transformer_encoder.transformer.layers.0.self_attn"
    sd[f"{p}.in_proj_weight"] = w
    sd[f"{p}.in_proj_bias"] = np.zeros(3 * D, np.float32)
    return sd


def natural_weights(gid, device):
    """Seed-initialised state dict of geometry ``gid`` (constructed geometries: FortiTran, then ``constructed``)."""
    m = make_model(gid, GEOMS[gid][1], device, seed=list(GEOMS).index(gid) if gid != "C5" else 0)
    sd = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    m._release()
    return constructed(sd, geom_S(gid)) if gid in CONSTRUCTED else sd


# ---------------------------------------------------------------------------------------------------------------------
# CPU part
# ---------------------------------------------------------------------------------------------------------------------

def test_workspace_layout_restated():
    """The layout worked by hand.  S65, b = 160 (pix 65): enh 20,800 floats (a multiple of 64), hbuf 2,662,400 floats,
    so the tc_long region would start at byte 10,732,800 = 1024 x 10,481 + 256: at a 1024-aligned workspace it moves up
    by 768 bytes, at one 256 bytes past a multiple of 1024 by 512; 320 tiles of 32,768 B per region.  C5, b = 2 (pix 45,864):
    enh 183,456 floats -> 183,488, hbuf 3,913,728 floats, start 16,388,864 = 1024 x 16,004 + 768: at a workspace 256
    bytes past 1024 (0x7f0000000100) no move, at a 1024-aligned one 256 bytes; 240 tiles of 32,768 B per region."""
    L = ws_layout(320, 65, 65, 0)
    assert (L["T"], L["tiles"], L["hbuf"], L["img"], L["ximg"]) == (1, 320, 83200, 10732800, 10733568)
    assert L["aimg"] - L["ximg"] == 10485760 and L["end"] - L["ximg"] == 5 * 10485760
    assert ws_layout(320, 65, 65, 0x7F0000000100)["ximg"] == 10733312
    base = 0x7F0000000100
    L = ws_layout(4, 7644, 45864, base)
    assert (L["T"], L["tiles"], L["hbuf"], L["img"]) == (60, 240, 183488 * 4, (183488 + 3913728) * 4)
    assert L["img"] == 16388864 and L["ximg"] == 16388864 and (base + L["ximg"]) % 1024 == 0
    assert ws_layout(4, 7644, 45864, 0)["ximg"] == 16389120
    assert [L[r] - L["ximg"] for r in ("aimg", "q", "k", "v", "end")] == [7864320 * i for i in range(1, 6)]
    for nseq, S in ((2, 1), (320, 65), (172, 129), (122, 257), (56, 1025), (4, 7644)):
        for base in (0, 256, 512, 768):
            L = ws_layout(nseq, S, 7 * S, base)
            assert (base + L["ximg"]) % 1024 == 0 and 0 <= L["ximg"] - L["img"] < 1024
            assert L["hbuf"] >= nseq * 7 * S * 4 and L["img"] - L["hbuf"] >= nseq * S * D * 4


def test_tile_decoder_against_hand_built_image():
    """Elements placed at byte offsets worked out by hand, then whole images (two tiles of a ragged S = 129 sequence)
    built unit by unit: physical unit u of row r holds logical unit u ^ (r & 7)."""
    img = np.zeros(TILE_IMG // 2, np.uint16)
    placed = {(0, 0): (0, 0x3F80, 1.0), (1, 0): (128 + 16, 0xC000, -2.0), (5, 13): (640 + 64 + 10, 0x3F00, 0.5),
              (9, 70): (16384 + 1152 + 16 + 12, 0x4040, 3.0), (127, 127): (16384 + 16256 + 14, 0xBE80, -0.25)}
    want = np.zeros((128, D), np.float32)
    for (r, c), (off, bits, val) in placed.items():
        img[off // 2] = bits
        want[r, c] = val
    got = decode_tiles(torch.from_numpy(img.view(np.uint8)), 1, 1)
    assert np.array_equal(got[0].numpy(), want)
    rng = np.random.default_rng(3)
    vals = (rng.integers(0, 1 << 16, (2 * 128, D), dtype=np.uint32) & 0xFF7F).astype(np.uint16)
    img = np.zeros((2, 2, 128, 8, 8), np.uint16)
    for r in range(256):
        for ch in range(2):
            for u in range(8):
                lu = u ^ (r & 7)
                img[r // 128, ch, r % 128, u] = vals[r, ch * 64 + lu * 8: ch * 64 + lu * 8 + 8]
    got = decode_tiles(torch.from_numpy(img.reshape(-1).view(np.uint8)), 1, 2)
    assert np.array_equal(got[0].numpy().view(np.uint32) >> 16, vals.astype(np.uint32))


def test_head_decoder_against_hand_built_image():
    """A Q / K / V head tile: rows of 64 B, unit u of row r at u ^ ((r >> 1) & 3); then the tile order
    ``(seq 4 + g) T + tile`` over 2 sequences x 4 heads x 3 tiles (S = 257: the last tile is ragged)."""
    img = np.zeros(HEAD_TILE // 2, np.uint16)
    placed = {(0, 0): (0, 0x3F80, 1.0), (2, 0): (128 + 16, 0xC000, -2.0), (3, 9): (192 + 0 + 2, 0x3F00, 0.5),
              (6, 31): (384 + 0 + 14, 0x4040, 3.0), (127, 17): (8128 + 16 + 2, 0xBE80, -0.25)}
    want = np.zeros((128, DH), np.float32)
    for (r, c), (off, bits, val) in placed.items():
        img[off // 2] = bits
        want[r, c] = val
    heads = np.zeros((NH, HEAD_TILE // 2), np.uint16)
    heads[2] = img                                 # head 2 of a one-tile sequence
    got = decode_heads(torch.from_numpy(heads.reshape(-1).view(np.uint8)), 1, 1)
    assert np.array_equal(got[0, 2].numpy(), want) and not bool(got[0, [0, 1, 3]].any())
    nseq, T = 2, 3
    rng = np.random.default_rng(4)
    vals = (rng.integers(0, 1 << 16, (nseq, NH, T * 128, DH), dtype=np.uint32) & 0xFF7F).astype(np.uint16)
    img = np.zeros((nseq, NH, T, 128, 4, 8), np.uint16)
    for r in range(T * 128):
        for u in range(4):
            img[:, :, r // 128, r % 128, u] = vals[:, :, r, (u ^ ((r >> 1) & 3)) * 8:(u ^ ((r >> 1) & 3)) * 8 + 8]
    got = decode_heads(torch.from_numpy(img.reshape(-1).view(np.uint8)), nseq, T)
    assert np.array_equal(got.numpy().view(np.uint32) >> 16, vals.astype(np.uint32))


def test_restatement_matches_oracle():
    """The restated layer (in_proj with the qscale fold, the tile-wise attention with its deferred rescale, the row
    block) against ``oracle/aft_oracle.py`` ``encoder_layer``, unrounded weights, S = 129 and 65, gelu and relu; and
    the tile-wise attention against a plain softmax, with constructed scores that rescale at every tile."""
    sd = util.forti_weights(util.ada_weights())
    sd = {k: v.astype(np.float64) for k, v in sd.items()}
    W = tw(sd, "cpu")
    rng = np.random.default_rng(9)
    for S, act in ((129, "gelu"), (65, "relu")):
        T = -(-S // 128)
        h = rng.standard_normal((3, S, D))
        x = torch.zeros(3, T * 128, D, dtype=torch.float64)
        x[:, :S] = torch.from_numpy(h)
        for l in (0, 3):
            p = f"transformer_encoder.transformer.layers.{l}.self_attn"
            y = F.linear(x, W[f"{p}.in_proj_weight"], W[f"{p}.in_proj_bias"])
            y[..., :D] *= math.log2(math.e) / math.sqrt(DH)
            q, k, v = split_heads(y)
            o, _ = attention(q, k, v, S)
            out = row_block(W, l, x, o.transpose(1, 2).reshape(x.shape), act)
            ref = O.encoder_layer(h, sd, l, NH, act)
            assert float((out[:, :S] - torch.from_numpy(ref)).abs().max()) < 1e-11 * float(np.abs(ref).max())
    # the tile loop against softmax: rising, falling and flat score rows, ragged last key tile
    S, R = 321, 384
    t = torch.arange(R, dtype=torch.float64)
    q = torch.zeros(1, 1, R, DH, dtype=torch.float64)
    q[0, 0, :, 0] = torch.where(t % 2 == 0, 1.0, -1.0) * torch.where(t % 3 == 0, 0.0, 1.0)
    k = torch.zeros(1, 1, R, DH, dtype=torch.float64)
    k[0, 0, :, 0] = 3.0 * t
    v = torch.from_numpy(rng.standard_normal((1, 1, R, DH)))
    o, rescaled = attention(q, k, v, S)
    ref = torch.softmax(math.log(2) * (q @ k[:, :, :S].transpose(-1, -2)), -1) @ v[:, :, :S]
    assert float((o - ref).abs().max()) < 1e-12
    assert bool(rescaled[0, 0, 2:S:6].all()) and bool(rescaled[0, 0, 4:S:6].all())
    assert not bool(rescaled[0, 0, 1::2].any()) and not bool(rescaled[0, 0, ::3].any())


def test_inproj_figure_and_constructed_operands():
    """The in_proj figure is below 1 for the kernel's arithmetic (bf16 of the fp32 sum) and above it one bf16 step
    off; the constructed weights give the scores the module docstring states, exactly, at S = 7644."""
    sd = util.forti_weights(util.ada_weights())
    rng = np.random.default_rng(2)
    x = bf16_rn(torch.from_numpy(rng.standard_normal((2, 128, D))))
    w, b = inproj_weights(sd, 0, "cpu")
    y32 = (F.linear(x.float(), w.float()) + b.float()).to(torch.bfloat16).double()
    assert fig_inproj(y32, x, w, b) <= 1.0
    i = int(y32.abs().argmax())
    bad = y32.clone().reshape(-1)
    bad[i] = bf16_rn(bad[i] * (1 + 3 * 2.0 ** -8))           # three bf16 steps off
    assert fig_inproj(bad.reshape(y32.shape), x, w, b) > 1.0
    S = 7644
    T = -(-S // 128)
    sdk = constructed(dict(sd, **{"transformer_encoder.positional_encoding.position_embeddings": np.zeros((1, S, D), np.float32)}), S)
    pos = torch.from_numpy(sdk["transformer_encoder.positional_encoding.position_embeddings"][0]).double()
    assert torch.equal(bf16_rn(pos), pos)
    x = torch.zeros(1, T * 128, D, dtype=torch.float64)
    x[0, :S] = pos
    w, b = inproj_weights(sdk, 0, "cpu")
    q, k, v = split_heads(bf16_rn(F.linear(x, w, b)))
    t = torch.arange(S, dtype=torch.float64)
    sign = 1 - 2 * (t % 2)
    for g in range(NH):
        assert torch.equal(q[0, g, :S, :2], (128 * sign)[:, None].expand(S, 2))
        assert torch.equal(k[0, g, :S, 0] * 128 + k[0, g, :S, 1] * 128, 16 * t - 131072)
        assert torch.equal(v[0, g, :S, :4], torch.stack([t % 64, sign, (t // 64) / 8, torch.full_like(t, g + 1)], 1))
        assert not bool(k[0, g, S:].any()) and not bool(v[0, g, S:].any())


FAULTS = {   # name: stage whose figure it moves
    "mask_off_by_one": "att", "mask_removed": "att", "last_key_dropped": "att", "ring_stale": "att",
    "no_rescale": "att", "head_swap": "att", "second_tile_stale_aimg": "row", "ln_half_stats": "row",
    "stale_residual_store": "layout",
}
# Natural-weight cases of the fault table: (id, sequences); enough sequences that some row tiles lie past 148.
TABLE_CASES = (("S65", 150), ("S1025", 18), ("K65", 150), ("K1025", 18))
# Faults these gates cannot see.  Natural weights: one extra padding key weighs too little (S65 -49.7, S1025 -59.1 dB),
# as do the dropped last key and the stale ring tile at S1025 (-85.7 / -59.2 dB) and, at S1025, the attention image of
# another row tile (-73.2 dB); no row rescales after key tile 0, so a skipped rescale changes nothing.  Faults that
# cannot occur: no ring wrap at S65 (2 key tiles), no middle launch in the one-layer constructed models, and at K65
# every sequence and so every row tile is the same.
INVISIBLE = {("S65", "mask_off_by_one"), ("S65", "ring_stale"), ("S65", "no_rescale"),
             ("S1025", "mask_off_by_one"), ("S1025", "last_key_dropped"), ("S1025", "ring_stale"), ("S1025", "no_rescale"),
             ("S1025", "second_tile_stale_aimg"),
             ("K65", "ring_stale"), ("K65", "second_tile_stale_aimg"), ("K65", "stale_residual_store"),
             ("K1025", "stale_residual_store")}


def _table_h0(gid, sd, nseq):
    """fp64 h0 of ``nseq`` sequences (the oracle's front end on seeded pilots), padded to whole row tiles."""
    kind, _, act, _, grid, pilots, patch, _ = GEOMS[gid]
    S = geom_S(gid)
    T = -(-S // 128)
    x = torch.zeros(nseq, T * 128, D, dtype=torch.float64)
    if gid in CONSTRUCTED:
        x[:, :S] = torch.from_numpy(sd["transformer_encoder.positional_encoding.position_embeddings"][0, :S]).double()
        return x
    cfg = O.OracleConfig(num_scs=grid[0], num_symbols=grid[1], pilot_scs=pilots[0], pilot_symbols=pilots[1], patch=patch,
                         num_layers=0, activation=act, adaptive=kind == "ada")
    rng = np.random.default_rng(11)
    b = nseq // 2
    p = (rng.standard_normal((b, *pilots)) + 1j * rng.standard_normal((b, *pilots))) / np.sqrt(2)
    md = (rng.choice(O.SNR_GRID, b), rng.choice(O.DS_GRID[:4], b), rng.choice(O.DOP_GRID[:3], b)) if kind == "ada" else (None,) * 3
    st = {}
    O.forward(cfg, sd, p, *md, stages=st)
    x[:, :S] = torch.from_numpy(np.stack([st["re"]["h0"], st["im"]["h0"]], 1).reshape(nseq, S, D))
    return x


def _gate_key(gid):
    return "constructed" if gid in CONSTRUCTED else "natural"


def test_fault_table():
    """Restates the plausible faults of the long path in fp64 and checks which of them the stage gates catch: each
    fault is injected at layer 0 (the stored residual at layer 0's launch), and its stage is compared with the clean
    stage fed with the same inputs."""
    lines, rescaled = [], {}
    for gid, nseq in TABLE_CASES:
        sd = natural_weights(gid, "cpu")
        W = tw(sd, "cpu")
        S, act, L = geom_S(gid), GEOMS[gid][2], GEOMS[gid][1]
        T = -(-S // 128)
        assert nseq * T > SMS_B200
        x = _table_h0(gid, sd, nseq)
        clean = long_layer(W, sd, 0, x, S, act)
        rescaled[gid] = int(clean["rescaled"][:, :, :S].sum())
        gate = GATES[_gate_key(gid)]
        for name, stage in FAULTS.items():
            f = long_layer(W, sd, 0, x, S, act, name)
            if stage == "att":
                moved = float(fig_rows(f["a"][:, :S], clean["a"][:, :S]).max())
                caught = moved > gate["att_db"] + FAULT_MARGIN_DB
                txt = f"attention {moved:7.1f} dB (gate {gate['att_db']:g})"
            elif stage == "row":
                moved = float(fig_rows(f["out"][:, :S], clean["out"][:, :S]).max())
                caught = moved > gate["row_db"] + FAULT_MARGIN_DB
                txt = f"row block {moved:7.1f} dB (gate {gate['row_db']:g})"
            else:
                rows = int((bf16_rn(f["stored"][:, :S]) != bf16_rn(clean["out"][:, :S])).any(-1).sum()) if L > 1 else 0
                caught = rows > 0
                txt = f"layout    {rows:7d} rows differ" + ("" if L > 1 else " (one layer: no middle launch)")
            lines.append(f"  {gid:6s} {name:24s} {txt}: " + ("caught" if caught else "INVISIBLE"))
            assert caught == ((gid, name) not in INVISIBLE), lines[-1]
        lines.append(f"  {gid:6s} query rows rescaled after key tile 0: {rescaled[gid]} of {nseq * NH * S}")
    print("\nfault table (fp64 restatement, layer 0):\n" + "\n".join(lines))
    assert rescaled["K65"] > 0 and rescaled["K1025"] > 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU part
# ---------------------------------------------------------------------------------------------------------------------

class Geometry:
    """One case: the state dict, the inputs of the composition batch, and the workspace read-back of each depth."""

    def __init__(self, gid):
        self.gid = gid
        kind, self.L, self.act, _, self.grid, self.pilots, self.patch, batch = GEOMS[gid]
        self.S = geom_S(gid)
        self.T = -(-self.S // 128)
        self.pix = self.grid[0] * self.grid[1]
        self.ada = kind == "ada"
        self.sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        self.B = batch or self.sm // self.T + 12
        self.nseq = 2 * self.B
        self.sd = natural_weights(gid, "cpu")
        rng = np.random.default_rng(100 + list(GEOMS).index(gid))
        shape = (self.B, *self.pilots)
        x = ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)).astype(np.complex64)
        self.x = torch.from_numpy(x).cuda()
        self.md = None
        if self.ada:
            md = (rng.choice(O.SNR_GRID, self.B), rng.choice(O.DS_GRID[:4], self.B), rng.choice(O.DOP_GRID[:3], self.B))
            self.md = tuple(torch.from_numpy(a.astype(np.float32)).cuda() for a in md)

    def run(self, depth):
        """A forward of the whole batch at ``depth`` layers into a caller-owned workspace (0xA5 first); returns the
        decoded regions (fp64 on the device) and the layout checks of the device side."""
        import ctypes as C
        from adafortitran_b200 import _capi
        m = make_model(self.gid, depth, "cuda", sd=self.sd)
        m.precision = "bf16"
        meta = (lambda s: util.meta(*(a[s].cpu().numpy() for a in self.md))) if self.ada else (lambda s: None)
        with torch.no_grad():
            m(self.x[:1].cpu(), meta(slice(0, 1)))
        lib = _capi.lib()
        ws_of = lambda b: lib.aft_workspace_bytes(m._handle, b, _capi.AFT_BF16)
        need = ws_of(self.B)
        top, lo, hi = ws_of(1 << 16), 1, 1 << 16
        while lo < hi:                           # the internal chunk: smallest batch with the full chunk's workspace
            mid = (lo + hi) // 2
            lo, hi = (lo, mid) if ws_of(mid) == top else (mid + 1, hi)
        raw = torch.full((need + 256,), 0xA5, dtype=torch.uint8, device="cuda")
        off = (-raw.data_ptr()) % 256
        ws = raw[off:off + need]
        lay = ws_layout(self.nseq, self.S, self.pix, ws.data_ptr())
        out = torch.empty((self.B, *self.grid), dtype=torch.complex64, device="cuda")
        vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        c = list(self.md) if self.ada else [None] * 3
        _capi.check(lib.aft_forward(m._handle, vp(self.x), vp(c[0]), vp(c[1]), vp(c[2]), vp(out), self.B, _capi.AFT_BF16,
                                    vp(ws), need, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        m._release()
        nseq, S, T = self.nseq, self.S, self.T
        reg = lambda name, size: ws[lay[name]:lay[name] + size]
        d = dict(chunk=lo, need=need, end=lay["end"],
                 enh=ws[:nseq * self.pix * 4].view(torch.float32).reshape(nseq, self.pix).double(),
                 hbuf=reg("hbuf", nseq * S * D * 4).view(torch.float32).reshape(nseq, S, D).double(),
                 x=decode_tiles(reg("ximg", lay["tiles"] * TILE_IMG), nseq, T).double(),
                 a=decode_tiles(reg("aimg", lay["tiles"] * TILE_IMG), nseq, T).double())
        for r in ("q", "k", "v"):
            d[r] = decode_heads(reg(r, lay["tiles"] * TILE_IMG), nseq, T).double()
        assert bool(torch.isfinite(out.view(torch.float32)).all())
        return d

    def h0(self, enh, W):
        """fp64 ``linear_1([patchify(enh) | adapter]) + pos`` of every sequence, from the GPU's ``enh``."""
        (H, Wd), (ph, pw), n = self.grid, self.patch, enh.shape[0]
        tok = enh.reshape(n, H // ph, ph, Wd // pw, pw).permute(0, 1, 3, 2, 4).reshape(n, self.S, ph * pw)
        if self.ada:
            feats = []
            for name, v in zip(("snr", "ds", "dop"), self.md):
                p = f"channel_adapter.{name}_encoder"
                z = torch.relu(F.linear(v.double().reshape(-1, 1), W[f"{p}.0.weight"], W[f"{p}.0.bias"]))
                z = torch.relu(F.linear(z, W[f"{p}.2.weight"], W[f"{p}.2.bias"]))
                feats.append(F.linear(z, W[f"{p}.4.weight"], W[f"{p}.4.bias"]).reshape(-1, self.S, 2))
            tok = torch.cat([tok, torch.cat(feats, 2).repeat_interleave(2, 0)], 2)
        pos = [W[k] for k in ("transformer_encoder.positional_encoding.position_embeddings",
                              "transformer_encoder.positional_encoding.pe") if k in W][0][0, :self.S]
        return F.linear(tok, W["transformer_encoder.linear_1.weight"], W["transformer_encoder.linear_1.bias"]) + pos


def check_layer(g, W, l, d, prev):
    """Figures of layer ``l`` from the depth-(l + 1) read-back ``d`` (``prev``: the depth-l read-back or None)."""
    S, T, nseq = g.S, g.T, g.nseq
    fig = {}
    x = d["x"]
    if l == 0:
        fig["pad_rows_nonzero"] = int((x[:, S:] != 0).any(-1).sum())
        if g.gid in CONSTRUCTED:
            pos = torch.as_tensor(g.sd["transformer_encoder.positional_encoding.position_embeddings"][0, :S], device=x.device).double()
            fig["h0_rows_not_exact"] = int((x[:, :S] != pos).any(-1).sum())
        else:
            fig["h0_db"] = float(fig_rows(x[:, :S], g.h0(d["enh"], W)).max())
    else:
        fig["layout_rows_differ"] = int((x[:, :S] != bf16_rn(prev["hbuf"])).any(-1).sum())
    w, b = inproj_weights(g.sd, l, x.device)
    nb = max(1, (1 << 16) // (T * 128))          # sequences per block of the fp64 attention
    inproj, att, rows, resc = 0.0, [], [], 0
    for s0 in range(0, nseq, nb):
        s1 = min(nseq, s0 + nb)
        xs = x[s0:s1]
        got = torch.cat([t[s0:s1].transpose(1, 2).reshape(s1 - s0, T * 128, D) for t in (d["q"], d["k"], d["v"])], -1)
        inproj = max(inproj, fig_inproj(got, xs, w, b))
        o, rescaled = attention(d["q"][s0:s1], d["k"][s0:s1], d["v"][s0:s1], S)
        got_a = d["a"][s0:s1].reshape(s1 - s0, T * 128, NH, DH).transpose(1, 2)
        att.append(fig_rows(got_a, o))
        resc += int(rescaled[:, :, :S].sum())
        ref = row_block(W, l, xs[:, :S], d["a"][s0:s1, :S], g.act)
        rows.append(fig_rows(d["hbuf"][s0:s1], ref))
    fig["inproj_ulp"] = inproj
    fig.update(attention_figures(torch.cat(att), S))
    rows = torch.cat(rows)
    fig["row_db"] = float(rows.max())
    fig["row_last_tile_db"] = float(rows[:, (S - 1) // 128 * 128:].max())
    fig["rescaled_rows"] = resc
    return fig


def check_gates(gid, fig):
    g = GATES[_gate_key(gid)]
    bad = [k for k in ("pad_rows_nonzero", "h0_rows_not_exact", "layout_rows_differ") if fig.get(k, 0) != 0]
    if "h0_db" in fig and not fig["h0_db"] <= g["h0_db"]:
        bad.append("h0_db")
    if not fig["inproj_ulp"] <= 1.0:
        bad.append("inproj_ulp")
    bad += [k for k in ("att_db", "row_db") if not fig[k] <= g[k]]
    return bad


@pytest.fixture(scope="module")
def report():
    t0 = time.perf_counter()
    yield
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = torch.cuda.get_device_name()
    print(f"\n{__name__}: wall time {time.perf_counter() - t0:.1f} s ({q}); worst figure per stage, per layer:")
    for (gid, l), fig in sorted(RESULTS.items(), key=lambda kv: (list(GEOMS).index(kv[0][0]), kv[0][1])):
        print(f"  {gid:6s} layer {l}: " + ", ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in fig.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("gid", list(GEOMS))
def test_long_stages(report, gid):
    """Every layer of the geometry, kernel by kernel (module docstring), from forwards of depth 1 ... L."""
    g = Geometry(gid)
    W = tw(g.sd, "cuda")
    prev, bad = None, {}
    for depth in range(1, g.L + 1):
        t0 = time.perf_counter()
        d = g.run(depth)
        assert g.B <= d["chunk"], (g.B, d["chunk"])               # the batch is one internal chunk
        assert d["end"] <= d["need"], (d["end"], d["need"])       # the workspace covers the restated layout
        fig = check_layer(g, W, depth - 1, d, prev)
        fig["seconds"] = time.perf_counter() - t0
        RESULTS[(gid, depth - 1)] = fig
        bad.update({depth - 1: check_gates(gid, fig)} if check_gates(gid, fig) else {})
        prev = dict(hbuf=d["hbuf"])
        del d
    if gid in CONSTRUCTED:
        assert RESULTS[(gid, 0)]["rescaled_rows"] > 0
    assert not bad, (bad, {l: RESULTS[(gid, l)] for l in bad})
