"""The reference-grid AFT_BF16 forward stage by stage against fp64, read back from the caller's workspace.

``bench.py`` times this path: ``adapter_kernel`` -> ``frontend_tc_kernel`` -> ``encoder_kernel`` -> ``head_tc_kernel``.
``tests/test_gpu_bf16.py`` checks it end to end by error power over a whole batch (-45 dB FortiTran, -38 dB AdaFortiTran at random init); a fault confined to the encoder's 24-row tail tile
can move the output by less than that and pass.  Here each kernel is judged alone.

``aft_forward`` computes into the workspace the caller passes.  ``tc_forward_chunk`` (``csrc/tc_encoder.cu``) lays
it out for a chunk of ``b`` samples (the last internal chunk of 8192) as three regions, each 1024-byte aligned:

* ``enh``: fp32 ``[2b][1680]``, the front end's conv-enhanced images, sequence ``seq = 2 sample + part``
  (part 0 real, 1 imaginary);
* the X images: ``[2b]`` x 73,728 bytes (``csrc/tc_layout.cuh``: 2 K-chunks x 288 rows x 128 B, the 16-byte units
  of row ``r`` permuted by XOR with ``r & 7``).  The front end writes ``bf16(linear_1(tokens) + pos)`` there, the
  encoder overwrites it in place with its output, the head only reads it;
* ``z``: the adapter's fp32 ``[b][3][560]`` (AdaFortiTran only).

Each stage is compared with a torch float64 restatement of the same operation (pinned to ``oracle/aft_oracle.py`` on
the CPU) fed with the GPU's output of the stage before it:

=========  ===================================================================  =======================================
stage      reference                                                            figure (worst over the batch)
=========  ===================================================================  =======================================
adapter    ``adapter(snr, ds, dop)``                                            normwise per sample
front end  ``conv_enhancer(upsample(x))``                                       error power per 128-position conv tile
                                                                                of the padded 122 x 16 grid (16 tiles,
                                                                                tile 15 ragged), relative to the
                                                                                sequence's mean square, in dB
encoder    ``encoder(h0)``, ``h0 = bf16(linear_1([patchify(enh) | z]) + pos)``  relative error power per token row, dB;
                                                                                reported per row tile 0..127,
                                                                                128..255 and the tail 256..279
head       ``linear_2``, fold, ``+ enh``, refiner on the decoded image          relative error power per sample, dB
end to end the fp64 forward from the pilots                                     relative error power per sample, dB
=========  ===================================================================  =======================================

Batches cover the grids: ``min(2b, 148)`` CTAs for the front end and the encoder, ``min(b, 148)`` for the head, all
static grid-stride with barrier phases from ``n_run & 1``; the adapter runs groups of 32 samples on
``min(groups, 148)`` CTAs.  b = 1; 74 (one sequence per CTA); 75 (CTAs 0, 1 run a second sequence); 148, 149 (the head's
second sample per CTA); 297; 4737 (the adapter's second pass, 148 x 32 + 1); 8192 (a full chunk, 110 or 111 sequences
per encoder CTA); 8195 (the workspace then holds the 3-sample second chunk on 6 CTAs; every sample of both chunks is
also compared with the fp32 path).  Every sequence is checked at every stage.  End to end against fp64: every sample up
to b = 297, otherwise every head CTA's first and second sample and the last 148 samples.

Weights: seed-0 FortiTran and the pseudo-trained AdaFortiTran of ``golden_trained.npz`` at every batch above; a
*sharpened* FortiTran (q and k rows of every ``in_proj_weight`` x 4) at 75, 297 and 8192; at b = 75 the relu, 2-layer,
1-layer (no next-layer projection hand-off) and sinusoidal FortiTran variants; seed-0 AdaFortiTran at 1, 75, 4737 and
8195.  Gates are per weight family (``GATES``).

Seed-0 AdaFortiTran has no encoder gate.  Its raw metadata (Doppler up to 1400) makes layer 0's attention logits span
about 456 per row, and rounding q and k to bf16 moves a logit by up to 8.5, so the nearly one-hot softmax picks its key
by rounding: the encoder output is -5 to -25 dB from fp64 per row (+1.5 dB with sharpened q, k).  Its encoder rows are reported only; its adapter, front end, head and end-to-end figures are gated.

Fault table (``test_fault_table``, CPU, fp64 restatement on 4 samples; FortiTran, sharpened FortiTran, trained
AdaFortiTran).  Each fault is restated where the kernel could make it; the table prints how far it moves its stage's
figure and the per-sample output.  A fault that moves its stage by more than the gate plus ``FAULT_MARGIN_DB`` is
caught.  Caught with every weight set: one head's tail P.V holding the result of the head before last (layer 5); conv
tile 15 left zero; the head using the previous sample's parked real part; a sample given its group neighbour's adapter
features (AdaFortiTran).  Caught with the FortiTran sets: padding keys left unmasked (-36.9 dB, -14.3 dB sharpened);
tail rows without the FFN2 bias (-36.3 dB); a sequence reading another sequence's X image (seq - 148, -32.6 dB).
Invisible to these gates, below the bf16 floor of the encoder output (-53 dB worst row) or the measured error: the tail
queries missing key 279 (layer 2: -85 / -79 / -110 dB at the worst row for FortiTran / sharpened / trained), one
head's tail P.V scaled by 1 % (layer 5: -58 / -58 / -63 dB) and tail rows normalised with the LayerNorm statistics of
rows 0..23 (layer 2: -73 / -74 / -90 dB); with the trained weights also the unmasked padding keys (-82.5 dB), the lost
FFN2 bias (-76 dB) and the other sequence's image (-52.7 dB against the gate of -49).  Sharpening does not expose them
in FortiTran: its encoder output is carried by the residual path.  The attention of seed-0 AdaFortiTran would show the
missing key (-25 dB when sharpened) but is too ill-conditioned to gate.
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

S, PIX, D, GRID = 280, 1680, 128, (120, 14)
SPAD, XIMG = 288, 73728           # X image: 288 rows (280 tokens + 8 zero rows) x 128 bf16, 2 K-chunks of 36,864 B
CHUNK = 8192                      # samples per internal chunk of the bf16 path (aft_api.cu kChunkBf16)
SEQ_BLOCK = 512                   # sequences per block of the fp64 restatement on the GPU

# Gates per weight family: the worst figure measured on a B200 (1000 W) over every case of the family, plus about 3 dB
# (adapter: x 6).  Measured (seed-0 AdaFortiTran / FortiTran sets / trained AdaFortiTran): adapter 1.7e-7 / - / 1.5e-7;
# front end -62.3 / -62.3 / -50.8 dB; encoder row - / -42.6 / -52.0 dB; head -49.4 / -49.8 / -35.5 dB; end to end
# -29.3 / -46.5 / -35.7 dB.  No encoder gate for seed-0 AdaFortiTran (module docstring).
GATES = {
    "ada": dict(adapter=1e-6, front_db=-59.0, enc_row_db=None, head_db=-46.0, e2e_db=-26.0),
    "forti": dict(adapter=None, front_db=-59.0, enc_row_db=-40.0, head_db=-47.0, e2e_db=-43.0),
    "trained": dict(adapter=1e-6, front_db=-48.0, enc_row_db=-49.0, head_db=-32.0, e2e_db=-33.0),
}
FAULT_MARGIN_DB = 3.0

RESULTS = {}   # (weights, batch) -> figures, printed at the end of the module


# ---------------------------------------------------------------------------------------------------------------------
# workspace layout and X-image decoder
# ---------------------------------------------------------------------------------------------------------------------

def align_up(v, a):
    return (v + a - 1) // a * a


def ws_layout(b):
    """Byte offsets of the X images and of ``z`` and the total size of ``tc_forward_chunk``'s workspace for a chunk of
    ``b`` samples (``enh`` starts at 0)."""
    nseq = 2 * b
    x0 = align_up(nseq * PIX * 4, 1024)
    z0 = x0 + align_up(nseq * XIMG, 1024)
    return x0, z0, z0 + align_up(b * 3 * 2 * S * 4, 1024)


def _ximage_index():
    """Element (row, col) of an X image -> index of its bf16 in the image (``tc_layout.cuh`` ``image_offset``)."""
    r = np.arange(SPAD)[:, None]
    c = np.arange(D)[None, :]
    byte = (c >> 6) * SPAD * 128 + r * 128 + ((((c & 63) >> 3) ^ (r & 7)) << 4) + (c & 7) * 2
    return byte // 2


XIDX = _ximage_index()


def decode_ximages(raw):
    """bf16 words of X images ``[..., 36864]`` (numpy uint16 or a torch int16 tensor) -> float32 ``[..., 288, 128]``."""
    if isinstance(raw, np.ndarray):
        return (raw[..., XIDX].astype(np.uint32) << 16).view(np.float32)
    x = raw[..., torch.as_tensor(XIDX, device=raw.device)]
    return ((x.to(torch.int32) & 0xFFFF) << 16).view(torch.float32)


# ---------------------------------------------------------------------------------------------------------------------
# torch float64 restatement (device-agnostic), with the faults of the fault table
# ---------------------------------------------------------------------------------------------------------------------

def _tile_of_pixel():
    r, c = np.meshgrid(np.arange(GRID[0]), np.arange(GRID[1]), indexing="ij")
    return ((r + 1) * 16 + (c + 1)) // 128          # conv tile of the padded 122 x 16 position grid


TILE = _tile_of_pixel()


def tw(sd, device):
    return {k: torch.as_tensor(np.asarray(v, np.float64), device=device) for k, v in sd.items()}


def r_adapter(W, snr, ds, dop):
    """ChannelAdapter -> ``[b][3][560]`` (MLP m's output j, as ``adapter_kernel`` stores it)."""
    out = []
    for name, v in (("snr", snr), ("ds", ds), ("dop", dop)):
        p = f"channel_adapter.{name}_encoder"
        z = torch.relu(F.linear(v.reshape(-1, 1), W[f"{p}.0.weight"], W[f"{p}.0.bias"]))
        z = torch.relu(F.linear(z, W[f"{p}.2.weight"], W[f"{p}.2.bias"]))
        out.append(F.linear(z, W[f"{p}.4.weight"], W[f"{p}.4.bias"]))
    return torch.stack(out, 1)


def r_enhancer(W, prefix, img, fault=None):
    y = img[:, None]
    for i, idx in enumerate((0, 2, 4, 6)):
        y = F.conv2d(y, W[f"{prefix}.conv_block.{idx}.weight"], W[f"{prefix}.conv_block.{idx}.bias"], padding=1)
        if i < 3:
            y = torch.relu(y)
        if i == 1 and fault == "conv_tile15_zero":      # conv2's epilogue leaves tile 15 at zero
            y = y * torch.as_tensor(TILE != 15, dtype=y.dtype, device=y.device)
    return y[:, 0]


def r_frontend(W, x, fault=None):
    """Per-sequence pilots ``[n][24]`` -> conv-enhanced images ``[n][120][14]``."""
    up = F.linear(x, W["pilot_upsampler.weight"], W["pilot_upsampler.bias"]).reshape(-1, *GRID)
    return r_enhancer(W, "initial_enhancer", up, fault if fault == "conv_tile15_zero" else None)


def r_tokens(enh, z):
    """``[patchify(enh) | adaptive features]`` for sequences ``[n]``; ``z`` is per sample (n / 2) or None."""
    n = enh.shape[0]
    tok = enh.reshape(n, 40, 3, 7, 2).permute(0, 1, 3, 2, 4).reshape(n, S, 6)
    if z is None:
        return tok
    ada = z.reshape(-1, 3, S, 2).permute(0, 2, 1, 3).reshape(-1, S, 6)   # token t, feature 6 + 2 m + e <- z[m][2 t + e]
    return torch.cat([tok, ada.repeat_interleave(2, 0)], 2)


def _pos(W):
    return [W[k] for k in ("transformer_encoder.positional_encoding.position_embeddings",
                           "transformer_encoder.positional_encoding.pe") if k in W][0][0, :S]


def r_h0(W, enh, z):
    return F.linear(r_tokens(enh, z), W["transformer_encoder.linear_1.weight"], W["transformer_encoder.linear_1.bias"]) + _pos(W)


def h0_image(W, enh, z):
    """The X image the encoder reads, bit for bit: ``linear1_image`` starts from ``fp32(pos + b1)`` and adds the
    features with fp32 FMAs in feature order (an fp32 FMA of fp32 operands is their fp64 product plus sum rounded to
    fp32), then rounds once to bf16.  ``bf16(fp64 linear_1)`` would round some elements the other way, and one such
    element moves a row of the random-init AdaFortiTran encoder by about -30 dB: its input is dominated by the raw
    metadata features, so the rounding of h0 alone moves its output by -14 dB."""
    tok = r_tokens(enh, z).float()
    w = W["transformer_encoder.linear_1.weight"].float()
    acc = (_pos(W).float() + W["transformer_encoder.linear_1.bias"].float()).expand(tok.shape[0], S, D)
    for k in range(tok.shape[2]):
        acc = (tok[..., k:k + 1].double() * w[:, k].double() + acc.double()).float()
    return acc.to(torch.bfloat16).double()


def _ln(x, g, b, stats=None):
    s = x if stats is None else stats
    mu = s.mean(-1, keepdim=True)
    var = s.var(-1, unbiased=False, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * g + b


def r_layer(W, h, l, cfg, fault=None):
    p = f"transformer_encoder.transformer.layers.{l}"
    n, nh, dh = h.shape[0], cfg.num_head, D // cfg.num_head
    hit = fault is not None and l == (5 if fault.startswith("tail_pv") else 2)
    qkv = F.linear(h, W[f"{p}.self_attn.in_proj_weight"], W[f"{p}.self_attn.in_proj_bias"])
    q, k, v = (qkv[..., i * D:(i + 1) * D].reshape(n, S, nh, dh).transpose(1, 2) for i in range(3))
    if hit and fault == "pad_keys_unmasked":          # rows 280..287 of the X image are zero: K, V = the biases
        bias = W[f"{p}.self_attn.in_proj_bias"]
        k = torch.cat([k, bias[D:2 * D].reshape(1, nh, 1, dh).expand(n, nh, SPAD - S, dh)], 2)
        v = torch.cat([v, bias[2 * D:].reshape(1, nh, 1, dh).expand(n, nh, SPAD - S, dh)], 2)
    sc = q @ k.transpose(-1, -2) / math.sqrt(dh)
    if hit and fault == "tail_misses_last_key":
        sc[:, :, 256:, S - 1] = -math.inf
    o = torch.softmax(sc, -1) @ v
    if hit and fault == "tail_pv_scaled":
        o[:, 3, 256:] *= 1.01
    if hit and fault == "tail_pv_stale":               # head 3's accumulator still holds head 1's tail (same TMEM columns)
        o[:, 3, 256:] = o[:, 1, 256:]
    o = F.linear(o.transpose(1, 2).reshape(n, S, D), W[f"{p}.self_attn.out_proj.weight"], W[f"{p}.self_attn.out_proj.bias"])
    x = h + o
    stats = None
    if hit and fault == "tail_ln_stats":               # tail rows take rows 0..23's mean and variance
        stats = x.clone()
        stats[:, 256:] = x[:, :S - 256]
    h = _ln(x, W[f"{p}.norm1.weight"], W[f"{p}.norm1.bias"], stats)
    f = F.linear(h, W[f"{p}.linear1.weight"], W[f"{p}.linear1.bias"])
    f = F.gelu(f) if cfg.activation == "gelu" else torch.relu(f)
    f = F.linear(f, W[f"{p}.linear2.weight"], W[f"{p}.linear2.bias"])
    if hit and fault == "tail_no_ffn2_bias":
        f[:, 256:] -= W[f"{p}.linear2.bias"]
    return _ln(h + f, W[f"{p}.norm2.weight"], W[f"{p}.norm2.bias"])


def r_encoder(W, h, cfg, fault=None):
    if fault == "reads_other_image":                   # seq reads the image of seq - 148: same part, another sample
        h = h.roll(4, 0)
    for l in range(cfg.num_layers):
        h = r_layer(W, h, l, cfg, fault)
    return h


def r_head(W, h, enh):
    """``linear_2``, fold, ``+ enh``, refiner: encoder output ``[n][280][128]`` -> real images ``[n][120][14]``."""
    n = h.shape[0]
    r = F.linear(h, W["transformer_encoder.linear_2.weight"], W["transformer_encoder.linear_2.bias"])
    rec = r.reshape(n, 40, 7, 3, 2).permute(0, 1, 3, 2, 4).reshape(n, *GRID)
    return r_enhancer(W, "final_refiner", enh + rec)


def to_complex(y):
    return torch.complex(y[0::2], y[1::2])


def seq_pilots(pilots):
    """complex ``[b][12][2]`` -> per-sequence real inputs ``[2b][24]`` (seq = 2 sample + part)."""
    return torch.stack([pilots.real, pilots.imag], 1).reshape(-1, 24).double()


def r_stages(W, cfg, pilots, cond, fault=None):
    """The whole fp64 forward of a few samples, keeping every stage's output; ``cond`` = (snr, ds, dop) or None."""
    z = r_adapter(W, *cond) if cfg.adaptive else None
    if fault == "adapter_neighbour":
        z = z[torch.arange(z.shape[0], device=z.device) ^ 1]
    enh = r_frontend(W, seq_pilots(pilots), fault)
    h = r_encoder(W, r_h0(W, enh, z), cfg, fault)
    y = r_head(W, h, enh)
    out = to_complex(y)
    if fault == "head_previous_real":                  # part 1 combines with the previous sample's parked real part
        out = torch.complex(out.real.roll(1, 0), out.imag)
    return dict(z=z, enh=enh, h=h, out=out)


# ---------------------------------------------------------------------------------------------------------------------
# figures
# ---------------------------------------------------------------------------------------------------------------------

def _db(num, den):
    return 10 * torch.log10(num / den)


def fig_adapter(z, ref):         # [b]
    return (z - ref).abs().amax((1, 2)) / ref.abs().amax((1, 2))


def fig_front(enh, ref):         # [n][16] tile error power over the sequence's mean square, dB
    tile = torch.as_tensor(TILE, device=enh.device).reshape(-1)
    d2 = ((enh - ref) ** 2).reshape(enh.shape[0], -1)
    per = torch.zeros(enh.shape[0], 16, dtype=d2.dtype, device=d2.device).index_add_(1, tile, d2)
    cnt = torch.bincount(tile, minlength=16).to(d2.dtype)
    return _db(per / cnt + 1e-300, (ref ** 2).reshape(enh.shape[0], -1).mean(1, keepdim=True))


def fig_rows(h, ref):            # [n][280]
    return _db(((h - ref) ** 2).sum(-1) + 1e-300, (ref ** 2).sum(-1))


def fig_samples(y, ref):         # complex [b][120][14] -> [b]
    return _db((y - ref).abs().square().sum((1, 2)) + 1e-300, ref.abs().square().sum((1, 2)))


TILES = {"rows_0_127": slice(0, 128), "rows_128_255": slice(128, 256), "rows_256_279": slice(256, S)}

# ---------------------------------------------------------------------------------------------------------------------
# CPU part
# ---------------------------------------------------------------------------------------------------------------------


def test_workspace_layout_restated():
    """The restated layout, worked by hand: b = 1 (enh 13,440 B -> 14,336; X 147,456; z 6,720 -> 7,168) and b = 8192
    (every region already a multiple of 1024)."""
    assert ws_layout(1) == (14336, 14336 + 147456, 14336 + 147456 + 7168)
    assert ws_layout(8192) == (110100480, 110100480 + 1207959552, 110100480 + 1207959552 + 55050240)
    for b in (1, 3, 74, 75, 149, 297, 4737, 8192):
        x0, z0, total = ws_layout(b)
        assert x0 % 1024 == 0 and z0 % 1024 == 0 and x0 >= 2 * b * PIX * 4 and z0 - x0 >= 2 * b * XIMG


def test_ximage_decoder_against_hand_built_image():
    """Elements placed at byte offsets worked out by hand from ``tc_layout.cuh``, then a whole image built unit by unit
    (physical unit u of row r holds logical unit u ^ (r & 7))."""
    img = np.zeros(XIMG // 2, np.uint16)
    placed = {   # (row, col): (byte offset, bf16 bits)
        (0, 0): (0, 0x3F80),                               # 1.0
        (1, 0): (128 + 16, 0xC000),                        # -2.0: unit 0 ^ 1 = 1
        (5, 13): (640 + 64 + 10, 0x3F00),                  # 0.5: unit 1 ^ 5 = 4, element 5
        (9, 70): (36864 + 1152 + 16 + 12, 0x4040),         # 3.0: chunk 1, unit 0 ^ 1 = 1, element 6
        (279, 127): (36864 + 35712 + 14, 0xBE80),          # -0.25: unit 7 ^ 7 = 0, element 7
        (287, 63): (36736 + 14, 0x3FC0),                   # 1.5: padding row 287, chunk 0
    }
    for (r, c), (off, bits) in placed.items():
        img[off // 2] = bits
    x = decode_ximages(img)
    want = np.zeros((SPAD, D), np.float32)
    for (r, c), v in zip(placed, (1.0, -2.0, 0.5, 3.0, -0.25, 1.5)):
        want[r, c] = v
    assert np.array_equal(x, want)

    rng = np.random.default_rng(3)
    vals = (rng.integers(0, 1 << 16, (SPAD, D), dtype=np.uint32) & 0xFF7F).astype(np.uint16)   # no NaN patterns
    img = np.zeros((2, SPAD, 8, 8), np.uint16)
    for r in range(SPAD):
        for ch in range(2):
            for u in range(8):
                lu = u ^ (r & 7)
                img[ch, r, u] = vals[r, ch * 64 + lu * 8: ch * 64 + lu * 8 + 8]
    x = decode_ximages(img.reshape(-1))
    assert np.array_equal(x.view(np.uint32) >> 16, vals.astype(np.uint32))
    t = decode_ximages(torch.from_numpy(img.reshape(1, -1).view(np.int16)))
    assert np.array_equal(t[0].numpy(), x)


@pytest.mark.parametrize("kind", ["ada", "forti"])
def test_restatement_matches_oracle(kind):
    """The torch fp64 restatement, stage by stage, against ``oracle/aft_oracle.py`` on three samples."""
    sd = util.ada_weights() if kind == "ada" else util.forti_weights(util.ada_weights())
    cfg = util.oracle_cfg(kind)
    p, snr, ds, dop = O.synthetic_batch(3, seed=5)
    st = {}
    ref = O.forward(cfg, sd, p, snr, ds, dop, stages=st)
    W = tw(sd, "cpu")
    cond = tuple(torch.from_numpy(a).double() for a in (snr, ds, dop)) if kind == "ada" else None
    r = r_stages(W, cfg, torch.from_numpy(p), cond)
    nw = lambda a, b: float(np.abs(np.asarray(a) - b).max() / np.abs(b).max())
    if kind == "ada":
        ada = O.adapter({k: v.astype(np.float64) for k, v in sd.items()}, snr.astype(np.float64), ds.astype(np.float64),
                        dop.astype(np.float64), S)
        zt = r["z"].reshape(3, 3, S, 2).permute(0, 2, 1, 3).reshape(3, S, 6)
        assert nw(zt, ada) < 1e-12
    for part, key in ((0, "re"), (1, "im")):
        assert nw(r["enh"][part::2], st[key]["conv_enhanced"]) < 1e-12
        assert nw(r["h"][part::2], st[key]["h6"]) < 1e-12
    assert nw(r["out"].numpy(), ref) < 1e-12
    h0 = r_h0(W, r["enh"], r["z"])
    assert nw(h0[0::2], st["re"]["h0"]) < 1e-12 and nw(h0[1::2], st["im"]["h0"]) < 1e-12
    # the encoder's input image, restated from fp32 stage outputs: bf16 values within half a bf16 step (plus the fp32
    # accumulation) of linear_1
    enh32, z32 = r["enh"].float().double(), None if r["z"] is None else r["z"].float().double()
    img, h = h0_image(W, enh32, z32), r_h0(W, enh32, z32)
    assert torch.equal(img, img.float().to(torch.bfloat16).double())
    assert ((img - h).abs() <= 2 ** -8 * h.abs() + 1e-6 * h.abs().max()).all()


FAULTS = {   # name: stage whose figure it moves
    "tail_misses_last_key": "enc", "pad_keys_unmasked": "enc", "tail_pv_scaled": "enc", "tail_pv_stale": "enc",
    "tail_ln_stats": "enc", "tail_no_ffn2_bias": "enc", "reads_other_image": "enc", "conv_tile15_zero": "front",
    "head_previous_real": "head", "adapter_neighbour": "adapter",
}
# faults the gates cannot see with these weights (named in the module docstring)
INVISIBLE = ({(w, f) for w in ("forti", "sharpened") for f in ("tail_misses_last_key", "tail_pv_scaled", "tail_ln_stats")}
             | {("trained", f) for f in ("tail_misses_last_key", "pad_keys_unmasked", "tail_pv_scaled", "tail_ln_stats",
                                         "tail_no_ffn2_bias", "reads_other_image")})


def _trained_weights():
    g = util.golden("golden_trained.npz")
    return {k[3:]: g[k] for k in g if k.startswith("sd/")}


def _sharpened(sd):
    """q and k rows of every ``in_proj_weight`` x 4: attention logits x 16."""
    out = dict(sd)
    for k, v in sd.items():
        if k.endswith("self_attn.in_proj_weight"):
            w = v.copy()
            w[:2 * D] *= 4
            out[k] = w
    return out


def _stage_figure(stage, f, c):
    """How far a fault moves its stage's figure (same units and sense as the gate)."""
    if stage == "adapter":
        return float(fig_adapter(f["z"], c["z"]).max())
    if stage == "front":
        return float(fig_front(f["enh"], c["enh"]).max())
    if stage == "enc":
        return float(fig_rows(f["h"], c["h"]).max())
    return float(fig_samples(f["out"], c["out"]).max())


def _gate_of(family, stage):
    return GATES[family][{"adapter": "adapter", "front": "front_db", "enc": "enc_row_db", "head": "head_db"}[stage]]


def test_fault_table():
    """Restates the plausible faults of this path in fp64 and checks which of them the stage gates catch."""
    p, snr, ds, dop = O.synthetic_batch(4, seed=5)
    assert len({(a, b, c) for a, b, c in zip(snr, ds, dop)}) == 4   # group neighbours differ in their metadata
    pil = torch.from_numpy(p)
    forti = util.forti_weights(util.ada_weights())
    lines = []
    for wname, sd, family in (("forti", forti, "forti"), ("sharpened", _sharpened(forti), "forti"),
                              ("trained", _trained_weights(), "trained")):
        cfg = util.oracle_cfg("ada" if wname == "trained" else "forti")
        cond = tuple(torch.from_numpy(a).double() for a in (snr, ds, dop)) if cfg.adaptive else None
        W = tw(sd, "cpu")
        clean = r_stages(W, cfg, pil, cond)
        for name, stage in FAULTS.items():
            if stage == "adapter" and not cfg.adaptive:
                continue
            f = r_stages(W, cfg, pil, cond, name)
            moved = _stage_figure(stage, f, clean)
            e2e = float(fig_samples(f["out"], clean["out"]).max())
            gate = _gate_of(family, stage)
            if stage == "adapter":
                caught = moved > gate * 10 ** (FAULT_MARGIN_DB / 20)
            else:
                caught = moved > gate + FAULT_MARGIN_DB
            lines.append(f"  {wname:9s} {name:22s} {stage:7s} stage {moved:9.3g} (gate {gate:g}), output {e2e:7.1f} dB: "
                         + ("caught" if caught else "INVISIBLE"))
            assert caught == ((wname, name) not in INVISIBLE), lines[-1]
    print("\nfault table (fp64 restatement, 4 samples of synthetic_batch(4, seed=5)):\n" + "\n".join(lines))


# ---------------------------------------------------------------------------------------------------------------------
# GPU part
# ---------------------------------------------------------------------------------------------------------------------

_MODELS = {}


def weight_set(name):
    """name -> (model, state dict, oracle config, gate family).  Every set but seed0 and trained is FortiTran."""
    if name in _MODELS:
        return _MODELS[name]
    sd0 = util.forti_weights(util.ada_weights())
    kind, sd, over, gate = "forti", sd0, {}, "forti"
    if name == "seed0":
        kind, sd, gate = "ada", util.ada_weights(), "ada"
    elif name == "trained":
        kind, sd, gate = "ada", _trained_weights(), "trained"
    elif name == "sharpened":
        sd = _sharpened(sd0)
    elif name == "relu":
        over = {"activation": "relu"}
    elif name in ("layers2", "layers1"):
        nl = int(name[-1])
        over = {"num_layers": nl}
        sd = {k: a for k, a in sd0.items() if not any(f"layers.{i}." in k for i in range(nl, 6))}
    elif name == "sinusoidal":
        over = {"pos_encoding_type": "sinusoidal"}
    if name == "sinusoidal":
        m = util.make_model(kind, precision="bf16", overrides=over)
        sd = {k: a for k, a in sd0.items() if "position_embeddings" not in k}
        sd["transformer_encoder.positional_encoding.pe"] = m.state_dict()["transformer_encoder.positional_encoding.pe"].cpu().numpy()
        m.load_state_dict(util.to_torch(sd))
    else:
        m = util.make_model(kind, weights=sd, precision="bf16", overrides=over)
    cfg = util.oracle_cfg(kind, num_layers=over.get("num_layers", 6), activation=over.get("activation", "gelu"))
    _MODELS[name] = (m, sd, cfg, gate)
    return _MODELS[name]


def _forward_into_workspace(model, pil, cond, b):
    """``aft_forward`` with a workspace the caller owns (256-byte aligned, filled with 0xA5 first)."""
    import ctypes as C
    from adafortitran_b200 import _capi
    with torch.no_grad():
        model(pil[:1].cpu(), util.meta(*(a[:1].cpu().numpy() for a in cond)) if cond is not None else None)
    lib = _capi.lib()
    need = lib.aft_workspace_bytes(model._handle, b, _capi.AFT_BF16)
    raw = torch.full((need + 256,), 0xA5, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 256
    ws = raw[off:off + need]
    out = torch.empty((b, *GRID), dtype=torch.complex64, device="cuda")
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    c = [a.float().contiguous() for a in cond] if cond is not None else [None] * 3
    _capi.check(lib.aft_forward(model._handle, vp(pil), vp(c[0]), vp(c[1]), vp(c[2]), vp(out), b, _capi.AFT_BF16,
                                vp(ws), need, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return out, ws


def _inputs(adaptive, b):
    p, snr, ds, dop = O.synthetic_batch(b, seed=1000 + b)
    pil = torch.from_numpy(p).cuda()
    cond = tuple(torch.from_numpy(a).cuda() for a in (snr, ds, dop)) if adaptive else None
    return pil, cond


def e2e_samples(b):
    """Samples compared end to end with fp64: all up to 297, else every head CTA's first and second sample and the last
    148 samples."""
    return list(range(b)) if b <= 297 else sorted(set(range(296)) | set(range(b - 148, b)))


def analyse(sd, cfg, pil, cond, out, ws):
    """The worst figure of every stage of a forward of ``len(pil)`` samples, from its estimates ``out`` and the
    workspace ``ws`` it computed into (uint8, as laid out by ``ws_layout`` for the last internal chunk)."""
    b, dev = pil.shape[0], out.device
    bl = b - (b - 1) // CHUNK * CHUNK            # samples of the last internal chunk: what the workspace holds
    c0 = b - bl
    x0, z0, _ = ws_layout(bl)
    nseq = 2 * bl
    W = tw(sd, dev)
    fig = {"samples_in_workspace": bl}
    enh_g = ws[:nseq * PIX * 4].view(torch.float32).reshape(nseq, *GRID).double()
    z_g = None
    if cfg.adaptive:
        z_g = ws[z0:z0 + bl * 3 * 2 * S * 4].view(torch.float32).reshape(bl, 3, 2 * S).double()
        zr = r_adapter(W, *(a[c0:].double() for a in cond))
        fig["adapter"] = float(fig_adapter(z_g, zr).max())
    front = fig_front(enh_g, r_frontend(W, seq_pilots(pil[c0:])))
    fig["front_db"] = float(front.max())
    fig["front_tile15_db"] = float(front[:, 15].max())
    ximg = ws[x0:x0 + nseq * XIMG].view(torch.int16).reshape(nseq, XIMG // 2)
    worst = {k: -1e9 for k in TILES}
    head, pad_nonzero = [], 0
    for s0 in range(0, nseq, SEQ_BLOCK):
        s1 = min(nseq, s0 + SEQ_BLOCK)
        img = decode_ximages(ximg[s0:s1])
        pad_nonzero += int((img[:, S:] != 0).any(2).any(1).sum())
        h = img[:, :S].double()
        h0 = h0_image(W, enh_g[s0:s1], z_g[s0 // 2:s1 // 2] if z_g is not None else None)
        rows = fig_rows(h, r_encoder(W, h0, cfg))
        for k, sl in TILES.items():
            worst[k] = max(worst[k], float(rows[:, sl].max()))
        yref = to_complex(r_head(W, h, enh_g[s0:s1]))
        head.append(fig_samples(out[c0 + s0 // 2:c0 + s1 // 2].to(torch.complex128), yref))
    fig.update({f"enc_{k}_db": v for k, v in worst.items()})
    fig["head_db"] = float(torch.cat(head).max())
    fig["pad_rows_nonzero_images"] = pad_nonzero
    idx = e2e_samples(b)
    e2e = []
    for i in range(0, len(idx), SEQ_BLOCK // 2):
        sel = torch.as_tensor(idx[i:i + SEQ_BLOCK // 2], device=dev)
        ref = r_stages(W, cfg, pil[sel], tuple(a[sel].double() for a in cond) if cond is not None else None)["out"]
        e2e.append(fig_samples(out[sel].to(torch.complex128), ref))
    fig["e2e_db"] = float(torch.cat(e2e).max())
    return fig


def run_case(name, b):
    """Runs one forward of ``b`` samples and returns the worst figure of every stage (no assertions)."""
    model, sd, cfg, _ = weight_set(name)
    pil, cond = _inputs(cfg.adaptive, b)
    t0 = time.perf_counter()
    out, ws = _forward_into_workspace(model, pil, cond, b)
    fig = analyse(sd, cfg, pil, cond, out, ws)
    if b > CHUNK:                                 # every sample of both chunks against the fp32 path
        model.precision = "fp32"
        try:
            with torch.no_grad():
                y32 = model(pil, util.meta(*(a.cpu().numpy() for a in cond)) if cond is not None else None)
        finally:
            model.precision = "bf16"
        fig["vs_fp32_db"] = float(fig_samples(out.to(torch.complex128), y32.to(torch.complex128)).max())
    fig["seconds"] = time.perf_counter() - t0
    return fig


def check_gates(name, fig):
    """The figures of ``fig`` above their family's gates."""
    g = GATES[weight_set(name)[3]]
    limits = dict(front_db=g["front_db"], head_db=g["head_db"], e2e_db=g["e2e_db"], vs_fp32_db=g["e2e_db"])
    if g["adapter"] is not None:
        limits["adapter"] = g["adapter"]
    if g["enc_row_db"] is not None:
        limits.update({f"enc_{t}_db": g["enc_row_db"] for t in TILES})
    return [k for k, v in limits.items() if k in fig and not fig[k] <= v]


COMPOSITIONS = (1, 74, 75, 148, 149, 297, 4737, 8192, 8195)
CASES = ([("forti", b) for b in COMPOSITIONS] + [("trained", b) for b in COMPOSITIONS]
         + [("seed0", b) for b in (1, 75, 4737, 8195)]
         + [("sharpened", b) for b in (75, 297, 8192)]
         + [(v, 75) for v in ("relu", "layers2", "layers1", "sinusoidal")])


@pytest.fixture(scope="module")
def report():
    t0 = time.perf_counter()
    yield
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = torch.cuda.get_device_name()
    print(f"\n{__name__}: wall time {time.perf_counter() - t0:.1f} s ({q}); worst figure per stage and row tile:")
    for (name, b), fig in sorted(RESULTS.items()):
        print(f"  {name:10s} b={b:5d}: " + ", ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}" for k, v in fig.items()))
    for m, *_ in _MODELS.values():
        m._release()
    _MODELS.clear()


@pytest.mark.gpu
def test_workspace_size_on_device(report):
    """``aft_workspace_bytes(h, b, AFT_BF16)`` is the restated layout up to one chunk and stops growing above it."""
    from adafortitran_b200 import _capi
    model = weight_set("seed0")[0]
    model._ensure_handle()
    ws = lambda b: _capi.lib().aft_workspace_bytes(model._handle, b, _capi.AFT_BF16)
    for b in (1, 2, 3, 74, 75, 148, 149, 297, 4737, 8191, 8192):
        assert ws(b) == ws_layout(b)[2], b
    for b in (8193, 8195, 16384, 1 << 20):
        assert ws(b) == ws_layout(CHUNK)[2], b


@pytest.mark.gpu
@pytest.mark.parametrize("name,b", CASES, ids=[f"{n}-{b}" for n, b in CASES])
def test_stages(report, name, b):
    fig = run_case(name, b)
    RESULTS[(name, b)] = fig
    assert not check_gates(name, fig), (check_gates(name, fig), fig)

