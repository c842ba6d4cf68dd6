"""Drop-in estimators: the reference's ``src/models`` class API over the B200 kernels.

``FortiTranEstimator`` / ``AdaFortiTranEstimator`` keep the reference's constructor, ``forward(pilot_symbols,
meta_data)`` contract, attributes, ``get_model_info()`` and -- key for checkpoints -- the exact ``state_dict``
keys and shapes (SURVEY.md Appendix A; reference ``src/models/fortitran.py:23-182,235-250``,
``src/models/adafortitran.py:5-22``).  The modules below are *parameter containers only*: no PyTorch
arithmetic runs in ``forward``; it hands device pointers to ``libaft_b200.so`` through the C-ABI
(``include/aft.h``).  There is no CPU or eager fallback -- calling ``forward`` without a CUDA (sm_100)
device or without the built library raises.
"""
from __future__ import annotations

import ctypes as C
import logging
import math
import operator
import os
from typing import List, Optional, Tuple

import torch
from torch import nn

from . import _capi
from .config import ModelConfig, SystemConfig

_PRECISIONS = {"fp32": _capi.AFT_FP32, "bf16": _capi.AFT_BF16}


# ----------------------------------------------------------------------------------------------
# parameter containers (names == reference state_dict keys)
# ----------------------------------------------------------------------------------------------
class _ConvStackParams(nn.Module):
    """``conv_block.{0,2,4,6}`` of the reference ConvEnhancer (enhancers.py:12-20): 1->8->32->8->1, 3x3."""

    def __init__(self) -> None:
        super().__init__()
        chans = (1, 8, 32, 8, 1)
        mods: List[nn.Module] = []
        for i in range(4):
            mods.append(nn.Conv2d(chans[i], chans[i + 1], kernel_size=3, padding=1))
            if i < 3:
                mods.append(nn.ReLU())
        self.conv_block = nn.Sequential(*mods)


class _AdapterParams(nn.Module):
    """``{snr,ds,dop}_encoder.{0,2,4}`` of the reference ChannelAdapter (channel_adaptivity.py:20-40)."""

    def __init__(self, hidden: Tuple[int, int, int]) -> None:
        super().__init__()
        for name in ("snr", "ds", "dop"):
            setattr(self, f"{name}_encoder", nn.Sequential(
                nn.Linear(1, hidden[0]), nn.ReLU(), nn.Linear(hidden[0], hidden[1]), nn.ReLU(),
                nn.Linear(hidden[1], hidden[2])))


class _LearnablePos(nn.Module):
    def __init__(self, max_len: int, d: int) -> None:  # positional_encodings.py:52-53
        super().__init__()
        self.position_embeddings = nn.Parameter(torch.zeros(1, max_len, d))
        nn.init.trunc_normal_(self.position_embeddings, std=0.02)

    def table(self) -> torch.Tensor:
        return self.position_embeddings


class _SinusoidalPos(nn.Module):
    def __init__(self, max_len: int, d: int) -> None:  # positional_encodings.py:16-26
        super().__init__()
        pos = torch.arange(0, max_len).unsqueeze(1)
        freq = torch.exp(torch.arange(0, d, 2) * (-torch.log(torch.tensor(10000.0)) / d))
        pe = torch.zeros(1, max_len, d)
        pe[0, :, 0::2] = torch.sin(pos * freq)
        pe[0, :, 1::2] = torch.cos(pos * freq)
        self.register_buffer("pe", pe)

    def table(self) -> torch.Tensor:
        return self.pe


class _AttnParams(nn.Module):
    """Parameters of ``nn.MultiheadAttention`` (same names, shapes and initialisation)."""

    def __init__(self, d: int) -> None:
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * d, d))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * d))
        self.out_proj = nn.Linear(d, d)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.zeros_(self.out_proj.bias)


class _EncoderLayerParams(nn.Module):
    """Parameters of one ``nn.TransformerEncoderLayer(d, nhead, 2d)`` (encoders.py:44-51)."""

    def __init__(self, d: int, ff: int) -> None:
        super().__init__()
        self.self_attn = _AttnParams(d)
        self.linear1 = nn.Linear(d, ff)
        self.linear2 = nn.Linear(ff, d)
        self.norm1 = nn.LayerNorm(d)
        self.norm2 = nn.LayerNorm(d)


class _EncoderStack(nn.Module):
    def __init__(self, d: int, ff: int, num_layers: int) -> None:
        super().__init__()
        self.layers = nn.ModuleList(_EncoderLayerParams(d, ff) for _ in range(num_layers))


class _EncoderParams(nn.Module):
    """``transformer_encoder.*`` (encoders.py:36-56)."""

    def __init__(self, input_dim: int, output_dim: int, cfg: ModelConfig) -> None:
        super().__init__()
        d = cfg.model_dim
        self.linear_1 = nn.Linear(input_dim, d)
        if cfg.pos_encoding_type == "learnable":
            self.positional_encoding = _LearnablePos(cfg.max_seq_len, d)
        elif cfg.pos_encoding_type == "sinusoidal":
            self.positional_encoding = _SinusoidalPos(cfg.max_seq_len, d)
        else:  # unreachable through ModelConfig; kept for parity with encoders.py:42
            raise ValueError("pos_encoding_type must be 'learnable' or 'sinusoidal'")
        self.transformer = _EncoderStack(d, 2 * d, cfg.num_layers)
        self.linear_2 = nn.Linear(d, output_dim)


class _PatchMap(nn.Module):
    """Parameter-free patchify / de-patchify index maps (patch_processors.py:6-71).  Inside the CUDA path they
    are fused into the producer / consumer kernels; these methods exist for API completeness and tests."""

    def __init__(self, grid: Tuple[int, int], patch: Tuple[int, int], inverse: bool) -> None:
        super().__init__()
        self.grid, self.patch_size, self.inverse = tuple(grid), tuple(patch), inverse

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        (h, w), (ph, pw) = self.grid, self.patch_size
        n = x.shape[0]
        if not self.inverse:
            return x.reshape(n, h // ph, ph, w // pw, pw).permute(0, 1, 3, 2, 4).reshape(n, -1, ph * pw)
        return x.reshape(n, h // ph, w // pw, ph, pw).permute(0, 1, 3, 2, 4).reshape(n, h, w)


# ----------------------------------------------------------------------------------------------
# estimators
# ----------------------------------------------------------------------------------------------
class BaseFortiTranEstimator(nn.Module):
    """Hybrid CNN-Transformer OFDM channel estimator; arithmetic in ``libaft_b200.so``.

    ``precision``: ``"fp32"`` (CUDA-core path, <= 1e-4 normwise vs the reference) or ``"bf16"`` (tcgen05
    path).  Default from ``$AFT_PRECISION``, else ``"fp32"``.

    ``trainable`` (default ``False``): with ``True``, a ``forward`` with grad enabled is differentiable with respect to
    every parameter (fp32 CUDA-core training path, reference default geometry): it applies the reference's dropout
    (``model_config.dropout``) in ``train()`` mode and none in ``eval()`` mode, and ``loss.backward()`` fills ``.grad``
    through ``aft_backward``.  Dropout masks are drawn from torch's default generator, so ``torch.manual_seed`` makes
    runs reproducible; ``forward(..., sample_offset=, dropout_seed=)`` fixes them explicitly (data-parallel training,
    :class:`adafortitran_b200.distributed.ShardedTrainer`).
    """

    trainable = False

    def __init__(self, system_config: SystemConfig, model_config: ModelConfig,
                 use_channel_adaptation: bool = False) -> None:
        super().__init__()
        self.system_config = system_config
        self.model_config = model_config
        self.use_channel_adaptation = use_channel_adaptation
        self.device = torch.device(model_config.device)
        self.logger = logging.getLogger(self.__class__.__name__)
        self.precision = os.environ.get("AFT_PRECISION", "fp32")
        self._handle: Optional[C.c_void_p] = None
        self._packed_key = None
        self._workspace: Optional[torch.Tensor] = None
        self._keepalive: list = []
        self._setup_dimensions()
        self._build_architecture()
        self.to(self.device)
        self._log_initialization_info()

    # -- construction (fortitran.py:52-143) -----------------------------------------------------
    def _setup_dimensions(self) -> None:
        ofdm, pilot = self.system_config.ofdm, self.system_config.pilot
        self.ofdm_size = (ofdm.num_scs, ofdm.num_symbols)
        self.pilot_size = (pilot.num_scs, pilot.num_symbols)
        self.pilot_features = pilot.num_scs * pilot.num_symbols
        self.ofdm_features = ofdm.num_scs * ofdm.num_symbols
        self.patch_length = self.model_config.patch_size[0] * self.model_config.patch_size[1]
        self.transformer_input_dim = self.patch_length
        if self.use_channel_adaptation:
            if self.model_config.adaptive_token_length is None:
                raise ValueError("adaptive_token_length must be set when channel adaptation is enabled")
            self.transformer_input_dim += self.model_config.adaptive_token_length

    def _build_architecture(self) -> None:
        cfg = self.model_config
        self.pilot_upsampler = nn.Linear(self.pilot_features, self.ofdm_features)
        self.initial_enhancer = _ConvStackParams()
        self.patch_embedder = _PatchMap(self.ofdm_size, cfg.patch_size, inverse=False)
        if self.use_channel_adaptation:
            if cfg.channel_adaptivity_hidden_sizes is None:
                raise ValueError("channel_adaptivity_hidden_sizes must be set when channel adaptation is enabled")
            hidden = tuple(cfg.channel_adaptivity_hidden_sizes)
            if len(hidden) != 3:
                raise ValueError("channel_adaptivity_hidden_sizes must have exactly 3 values")
            self.channel_adapter = _AdapterParams(hidden)
        self.transformer_encoder = _EncoderParams(self.transformer_input_dim, self.patch_length, cfg)
        self.patch_reconstructor = _PatchMap(self.ofdm_size, cfg.patch_size, inverse=True)
        self.final_refiner = _ConvStackParams()

    def _log_initialization_info(self) -> None:
        info = self.get_model_info()
        self.logger.info("%s initialized (B200 kernels): adaptation=%s grid=%s pilots=%s patch=%s d=%d layers=%d "
                         "device=%s params=%d", info["model_name"], info["channel_adaptation"], info["ofdm_size"],
                         info["pilot_size"], info["patch_size"], info["model_dim"], info["num_layers"],
                         info["device"], info["total_parameters"])

    def get_model_info(self) -> dict:
        params = list(self.parameters())
        return {
            "model_name": self.__class__.__name__,
            "channel_adaptation": self.use_channel_adaptation,
            "ofdm_size": self.ofdm_size,
            "pilot_size": self.pilot_size,
            "patch_size": self.model_config.patch_size,
            "patch_length": self.patch_length,
            "transformer_input_dim": self.transformer_input_dim,
            "model_dim": self.model_config.model_dim,
            "num_layers": self.model_config.num_layers,
            "device": str(self.device),
            "total_parameters": sum(p.numel() for p in params),
            "trainable_parameters": sum(p.numel() for p in params if p.requires_grad),
        }

    # -- nn.Module plumbing ---------------------------------------------------------------------
    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        # parameters may have moved (``.to()``, ``.cuda()``): follow them and drop device-side state
        try:
            self.device = next(self.parameters()).device
        except StopIteration:
            pass
        self._release()
        return out

    def _release(self) -> None:
        if getattr(self, "_handle", None) is not None:
            _capi.lib().aft_destroy(self._handle)
        self._handle, self._packed_key, self._workspace, self._keepalive = None, None, None, []

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    # -- C-ABI glue -----------------------------------------------------------------------------
    def _aft_config(self) -> _capi.AftConfig:
        cfg, hidden = self.model_config, self.model_config.channel_adaptivity_hidden_sizes or [0, 0, 0]
        return _capi.AftConfig(
            num_scs=self.ofdm_size[0], num_symbols=self.ofdm_size[1],
            pilot_scs=self.pilot_size[0], pilot_symbols=self.pilot_size[1],
            patch_scs=cfg.patch_size[0], patch_symbols=cfg.patch_size[1],
            num_layers=cfg.num_layers, model_dim=cfg.model_dim, num_head=cfg.num_head, ff_dim=2 * cfg.model_dim,
            activation=_capi.AFT_ACT_GELU if cfg.activation == "gelu" else _capi.AFT_ACT_RELU,
            adaptive=int(self.use_channel_adaptation),
            adapt_h1=hidden[0], adapt_h2=hidden[1], adapt_h3=hidden[2],
            adaptive_token_length=cfg.adaptive_token_length or 0, max_seq_len=cfg.max_seq_len)

    def _ensure_handle(self) -> None:
        if self.device.type != "cuda":
            raise RuntimeError(
                f"{self.__class__.__name__}: device is '{self.device}', but this implementation runs only on "
                "CUDA sm_100 (B200) through libaft_b200.so; there is no CPU fallback. Construct the model with "
                "ModelConfig(device='cuda') or move it with .to('cuda').")
        if self._handle is None:
            with torch.cuda.device(self.device):
                handle = C.c_void_p()
                cfg = self._aft_config()
                _capi.check(_capi.lib().aft_create(C.byref(cfg), C.byref(handle)))
                self._handle = handle

    def _weight_tensors(self):
        """fp32, contiguous views of every parameter in ABI order, plus a staleness key."""
        te = self.transformer_encoder
        named = [("up_w", self.pilot_upsampler.weight), ("up_b", self.pilot_upsampler.bias)]
        for tag, stack in (("enh", self.initial_enhancer), ("ref", self.final_refiner)):
            for i, idx in enumerate((0, 2, 4, 6)):
                named += [(f"{tag}_w{i}", stack.conv_block[idx].weight), (f"{tag}_b{i}", stack.conv_block[idx].bias)]
        if self.use_channel_adaptation:
            for name in ("snr", "ds", "dop"):
                enc = getattr(self.channel_adapter, f"{name}_encoder")
                for i, idx in enumerate((0, 2, 4)):
                    named += [(f"{name}_w{i}", enc[idx].weight), (f"{name}_b{i}", enc[idx].bias)]
        named += [("l1_w", te.linear_1.weight), ("l1_b", te.linear_1.bias), ("pos", te.positional_encoding.table()),
                  ("l2_w", te.linear_2.weight), ("l2_b", te.linear_2.bias)]
        for l, layer in enumerate(te.transformer.layers):
            a = layer.self_attn
            named += [(f"L{l}_in_w", a.in_proj_weight), (f"L{l}_in_b", a.in_proj_bias),
                      (f"L{l}_out_w", a.out_proj.weight), (f"L{l}_out_b", a.out_proj.bias),
                      (f"L{l}_l1_w", layer.linear1.weight), (f"L{l}_l1_b", layer.linear1.bias),
                      (f"L{l}_l2_w", layer.linear2.weight), (f"L{l}_l2_b", layer.linear2.bias),
                      (f"L{l}_n1_w", layer.norm1.weight), (f"L{l}_n1_b", layer.norm1.bias),
                      (f"L{l}_n2_w", layer.norm2.weight), (f"L{l}_n2_b", layer.norm2.bias)]
        key = tuple((t.data_ptr(), t._version, t.dtype) for _, t in named)
        return named, key

    def invalidate_weights(self) -> None:
        """Forget the packed copies of the parameters: the next forward re-reads every parameter.

        The library computes on private packed copies (fp32 re-layouts, bf16 operand images).  They are refreshed
        automatically when a parameter's storage or version counter changes (``load_state_dict``, optimizer steps,
        in-place ops on the parameter itself) and after ``load_state_dict`` (post-hook).  Writes that bypass the version
        counter -- ``p.data.copy_(...)``, ``p.data.mul_(...)``, EMA swaps through ``.data`` -- are invisible to that
        test: call this method after them, or set ``model.weight_check = "checksum"`` (an on-device checksum of all
        parameters per forward, one small kernel + a 16-byte read-back) or ``"always"`` (repack on every forward)."""
        self._packed_key = None

    refresh_weights = invalidate_weights

    def _param_checksum(self, named) -> Tuple[float, float]:
        flat = torch.cat([t.detach().reshape(-1).to(torch.float64) for _, t in named])
        w = torch.arange(1, flat.numel() + 1, dtype=torch.float64, device=flat.device)
        return float(flat.sum().item()), float((flat * (w % 8191.0)).sum().item())

    def _sync_weights(self) -> None:
        named, key = self._weight_tensors()
        mode = getattr(self, "weight_check", "version")
        if mode not in ("version", "checksum", "always"):
            raise ValueError(f"weight_check must be 'version', 'checksum' or 'always', got {mode!r}")
        if mode == "checksum":
            key = key + (self._param_checksum(named),)
        if mode != "always" and key == self._packed_key:
            return
        keep = {n: t.detach().to(device=self.device, dtype=torch.float32).contiguous() for n, t in named}
        ptr = lambda n: C.cast(keep[n].data_ptr(), C.POINTER(C.c_float))
        w = _capi.AftWeights()
        w.upsampler_w, w.upsampler_b = ptr("up_w"), ptr("up_b")
        for tag, dst in (("enh", w.initial_enhancer), ("ref", w.final_refiner)):
            for i in range(4):
                dst.w[i], dst.b[i] = ptr(f"{tag}_w{i}"), ptr(f"{tag}_b{i}")
        if self.use_channel_adaptation:
            for name, dst in (("snr", w.snr_encoder), ("ds", w.ds_encoder), ("dop", w.dop_encoder)):
                for i in range(3):
                    dst.w[i], dst.b[i] = ptr(f"{name}_w{i}"), ptr(f"{name}_b{i}")
        w.linear_1_w, w.linear_1_b, w.pos_table = ptr("l1_w"), ptr("l1_b"), ptr("pos")
        w.linear_2_w, w.linear_2_b = ptr("l2_w"), ptr("l2_b")
        n_layers = self.model_config.num_layers
        layers = (_capi.AftEncoderLayer * n_layers)()
        for l in range(n_layers):
            for field, tag in (("in_proj_w", "in_w"), ("in_proj_b", "in_b"), ("out_proj_w", "out_w"),
                               ("out_proj_b", "out_b"), ("lin1_w", "l1_w"), ("lin1_b", "l1_b"), ("lin2_w", "l2_w"),
                               ("lin2_b", "l2_b"), ("norm1_w", "n1_w"), ("norm1_b", "n1_b"), ("norm2_w", "n2_w"),
                               ("norm2_b", "n2_b")):
                setattr(layers[l], field, ptr(f"L{l}_{tag}"))
        w.layers, w.num_layers = layers, n_layers
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(_capi.lib().aft_load_weights(self._handle, C.byref(w), C.c_void_p(stream)))
        self._keepalive = list(keep.values())   # sources must outlive the asynchronous packing kernels
        self._packed_key = key

    def _get_workspace(self, batch: int, precision: int) -> torch.Tensor:
        need = _capi.lib().aft_workspace_bytes(self._handle, batch, precision)
        if need == 0:
            raise _capi.AftError(_capi.AFT_ERR_INVALID, _capi.lib().aft_last_error().decode())
        if self._workspace is None or self._workspace.numel() < need + 256:
            self._workspace = None
            self._workspace = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
        return self._workspace

    def _precision_code(self) -> int:
        try:
            return _PRECISIONS[self.precision]
        except KeyError:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}, got {self.precision!r}") from None

    # -- argument checks shared by every entry point (fortitran.py:157-173) -----------------------
    def _check_call(self, pilot_symbols: torch.Tensor, meta_data: Optional[Tuple], where: str):
        """Validates one call and returns ``(batch, meta_1_3)``; ``where`` is "cuda" (forward) or "cpu" (forward_host)."""
        if self.use_channel_adaptation and meta_data is None:
            raise ValueError("meta_data is required when channel adaptation is enabled")
        if not self.use_channel_adaptation and meta_data is not None:
            self.logger.warning("meta_data provided but channel adaptation is disabled - ignoring meta_data")
        if where == "cpu" and self.trainable and torch.is_grad_enabled():
            raise RuntimeError("forward_host is inference-only and not differentiable: with model.trainable = True and "
                               "grad enabled, call forward() on device tensors, or run forward_host under torch.no_grad()")
        if self.training and torch.is_grad_enabled() and not (self.trainable and where == "cuda"):
            raise RuntimeError("this implementation is inference-only unless model.trainable = True: call model.eval() "
                               "and/or run under torch.no_grad(), or set model.trainable = True to train on the GPU")
        if not torch.is_tensor(pilot_symbols) or not torch.is_complex(pilot_symbols):
            raise TypeError(f"pilot_symbols must be a complex tensor, got {getattr(pilot_symbols, 'dtype', type(pilot_symbols))}")
        if pilot_symbols.dim() != 3 or tuple(pilot_symbols.shape[1:]) != self.pilot_size:
            raise ValueError(f"expected pilot_symbols of shape [batch, {self.pilot_size[0]}, {self.pilot_size[1]}], "
                             f"got {tuple(pilot_symbols.shape)}")
        if where == "cpu" and pilot_symbols.device.type != "cpu":
            raise ValueError("forward_host expects CPU tensors; use forward() for device tensors")
        batch = pilot_symbols.shape[0]
        cond = None
        if self.use_channel_adaptation:
            if not isinstance(meta_data, (tuple, list)) or len(meta_data) < 4:
                raise ValueError("meta_data must be the reference tuple (file_no, snr, delay_spread, max_dop_shift, pilot_freq, "
                                 "channel_type)")
            cond = list(meta_data[1:4])
            for t in cond:
                if not torch.is_tensor(t):
                    raise TypeError("meta_data entries 1..3 (snr, delay_spread, max_dop_shift) must be tensors")
                if t.numel() != batch:
                    raise ValueError(f"meta_data entries must have {batch} elements, got {t.numel()}")
                if where == "cpu" and t.device.type != "cpu":
                    raise ValueError("forward_host expects CPU meta_data tensors")
        return batch, cond

    def _check_host_out(self, out: Optional[torch.Tensor], batch: int) -> torch.Tensor:
        if out is None:
            return torch.empty((batch, *self.ofdm_size), dtype=torch.complex64, pin_memory=True)
        if not torch.is_tensor(out) or out.device.type != "cpu" or out.dtype != torch.complex64 or not out.is_contiguous() \
                or tuple(out.shape) != (batch, *self.ofdm_size):
            raise ValueError(f"out must be a contiguous CPU complex64 tensor of shape {(batch, *self.ofdm_size)}, got "
                             f"{getattr(out, 'dtype', None)} {tuple(getattr(out, 'shape', ()))} on "
                             f"{getattr(getattr(out, 'device', None), 'type', None)}")
        return out

    # -- forward (fortitran.py:145-182) ---------------------------------------------------------
    def forward(self, pilot_symbols: torch.Tensor, meta_data: Optional[Tuple] = None, gather=None, *,
                sample_offset: int = 0, dropout_seed: Optional[int] = None) -> torch.Tensor:
        """``pilot_symbols``: complex [batch, pilot_scs, pilot_symbols]; ``meta_data``: the reference 6-tuple
        ``(file_no, snr, delay_spread, max_dop_shift, pilot_freq, channel_type)`` (items 1..3 are used).
        Returns complex64 [batch, ofdm_scs, ofdm_symbols] on ``self.device``.

        ``gather`` (keyword, optional; not part of the reference signature): a
        :class:`adafortitran_b200.distributed.PeerGather`; the kernel that writes the estimates then also stores them into
        every rank's gather buffer (fused all-gather over NVLink) and the returned tensor is this rank's slice of the
        local gather buffer.

        ``sample_offset`` and ``dropout_seed`` (keywords, differentiable calls only): sample ``b`` of this call draws the
        dropout masks of sample ``sample_offset + b`` of a larger batch, and ``dropout_seed`` (an integer in
        ``[0, 2**64)``) replaces the seed otherwise drawn from torch's default generator.  Shards of one batch forwarded
        with their offsets and one seed get exactly the masks of a single call over the whole batch.  A non-default
        value on an inference call raises ``ValueError``."""
        precision = self._precision_code()
        batch, cond_in = self._check_call(pilot_symbols, meta_data, "cuda")
        sample_offset = operator.index(sample_offset)
        if self.trainable and torch.is_grad_enabled():
            return self._forward_differentiable(pilot_symbols, cond_in, batch, precision, gather, sample_offset,
                                                dropout_seed)
        if sample_offset != 0 or dropout_seed is not None:
            raise ValueError("sample_offset / dropout_seed select dropout masks of a differentiable call: they have no "
                             "meaning for inference (model.trainable = False or grad disabled)")
        self._ensure_handle()
        with torch.cuda.device(self.device):
            pilots = pilot_symbols.to(device=self.device, dtype=torch.complex64).contiguous()
            cond = [None, None, None]
            if cond_in is not None:
                cond = [t.to(device=self.device, dtype=torch.float32).reshape(-1).contiguous() for t in cond_in]
            self._sync_weights()
            if gather is not None:
                gather.check(self, batch)
                out = gather.local_rows(batch)
            else:
                out = torch.empty((batch, *self.ofdm_size), dtype=torch.complex64, device=self.device)
            if batch == 0:
                return out
            ws = self._get_workspace(batch, precision)
            ws_ptr = (ws.data_ptr() + 255) // 256 * 256
            stream = torch.cuda.current_stream(self.device).cuda_stream
            vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            if gather is None:
                _capi.check(_capi.lib().aft_forward(
                    self._handle, vp(pilots), vp(cond[0]), vp(cond[1]), vp(cond[2]), vp(out), batch, precision,
                    C.c_void_p(ws_ptr), ws.numel() - (ws_ptr - ws.data_ptr()), C.c_void_p(stream)))
            else:
                plan = gather.plan()
                # fused tensor-core path (AFT_BF16 on the reference default geometry): the head stores straight into the
                # gather buffers; every other path, the long-sequence bf16 path of other geometries included, computes
                # into a local stage that the library then copies to the gather buffers
                reference_geometry = (self.ofdm_size == (120, 14) and self.pilot_size == (12, 2)
                                      and tuple(self.model_config.patch_size) == (3, 2))
                fused = precision == _capi.AFT_BF16 and reference_geometry and not gather.force_staging
                stage = None if fused else torch.empty((batch, *self.ofdm_size), dtype=torch.complex64, device=self.device)
                _capi.check(_capi.lib().aft_forward_gather(
                    self._handle, vp(pilots), vp(cond[0]), vp(cond[1]), vp(cond[2]), vp(stage), batch, precision,
                    C.c_void_p(ws_ptr), ws.numel() - (ws_ptr - ws.data_ptr()), C.c_void_p(stream), C.byref(plan)))
        return out

    def _forward_differentiable(self, pilot_symbols, cond_in, batch, precision, gather, sample_offset,
                                dropout_seed) -> torch.Tensor:
        if precision != _capi.AFT_FP32:
            raise ValueError("training (trainable = True with grad enabled) runs on the fp32 CUDA-core path only; "
                             "set model.precision = 'fp32' or run under torch.no_grad()")
        if gather is not None:
            raise ValueError("gather= is an inference path: it cannot be combined with a differentiable call")
        inputs = [pilot_symbols] + list(cond_in or [])
        if any(torch.is_tensor(t) and t.requires_grad for t in inputs):
            raise ValueError("gradients with respect to the pilots or the metadata are not computed: pass inputs that "
                             "do not require grad")
        if dropout_seed is not None:
            dropout_seed = operator.index(dropout_seed)
            if not 0 <= dropout_seed < 2 ** 64:
                raise ValueError(f"dropout_seed must be in [0, 2**64), got {dropout_seed}")
        self._ensure_handle()
        with torch.cuda.device(self.device):
            pilots = pilot_symbols.to(device=self.device, dtype=torch.complex64).contiguous()
            cond = [None, None, None]
            if cond_in is not None:
                cond = [t.to(device=self.device, dtype=torch.float32).reshape(-1).contiguous() for t in cond_in]
            p = float(self.model_config.dropout) if self.training else 0.0
            if dropout_seed is None:
                dropout_seed = int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())
            named, _ = self._weight_tensors()
            return _TrainForward.apply(self, pilots, cond, batch, p, dropout_seed, sample_offset, *[t for _, t in named])

    def forward_host(self, pilot_symbols: torch.Tensor, meta_data: Optional[Tuple] = None,
                     out: Optional[torch.Tensor] = None, gather=None) -> torch.Tensor:
        """Host-buffer entry point (``aft_forward_host``): CPU tensors in (pinned for full overlap), CPU complex64
        estimates out; host<->device copies are chunked and overlapped with compute inside the library.  Same argument
        checks as :meth:`forward`; ``out`` (optional) must be a contiguous CPU complex64 ``[batch, scs, symbols]`` tensor.
        With ``gather`` the estimates are also stored into every rank's gather buffer (see :meth:`forward`)."""
        precision = self._precision_code()
        batch, cond_in = self._check_call(pilot_symbols, meta_data, "cpu")
        out = self._check_host_out(out, batch)
        self._ensure_handle()
        pilots = pilot_symbols.to(dtype=torch.complex64).contiguous()
        cond = [None, None, None]
        if cond_in is not None:
            cond = [t.to(dtype=torch.float32).reshape(-1).contiguous() for t in cond_in]
        if batch == 0:
            return out
        with torch.cuda.device(self.device):
            self._sync_weights()
            torch.cuda.current_stream(self.device).synchronize()   # packed weights visible to the internal streams
            vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            if gather is None:
                _capi.check(_capi.lib().aft_forward_host(self._handle, vp(pilots), vp(cond[0]), vp(cond[1]), vp(cond[2]),
                                                         vp(out), batch, precision))
            else:
                gather.check(self, batch)
                plan = gather.plan()
                _capi.check(_capi.lib().aft_forward_host_gather(self._handle, vp(pilots), vp(cond[0]), vp(cond[1]), vp(cond[2]),
                                                                vp(out), batch, precision, C.byref(plan)))
        return out

    def _load_from_state_dict(self, *args, **kwargs):
        out = super()._load_from_state_dict(*args, **kwargs)
        self._packed_key = None     # load_state_dict: always repack (copy_ into .data would otherwise go unnoticed)
        return out


class _TrainForward(torch.autograd.Function):
    """``aft_forward_train_offset`` / ``aft_backward`` behind autograd.  The parameters are inputs of the Function (in the order
    of ``_weight_tensors``), so ``AccumulateGrad``, ``requires_grad=False``, hooks and version checks work as for any
    torch op; their gradients are views of the flat buffer ``aft_backward`` fills."""

    @staticmethod
    def forward(ctx, model, pilots, cond, batch, p, seed, sample0, *params):
        model._sync_weights()
        out = torch.empty((batch, *model.ofdm_size), dtype=torch.complex64, device=model.device)
        ws = None
        if batch > 0:
            lib = _capi.lib()
            need = lib.aft_train_workspace_bytes(model._handle, batch)
            if need == 0:
                _capi.check(_capi.AFT_ERR_UNSUPPORTED if model._handle else _capi.AFT_ERR_INVALID)
            ws = torch.empty(need + 256, dtype=torch.uint8, device=model.device)
            ws_ptr = (ws.data_ptr() + 255) // 256 * 256
            vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            stream = torch.cuda.current_stream(model.device).cuda_stream
            _capi.check(lib.aft_forward_train_offset(model._handle, vp(pilots), vp(cond[0]), vp(cond[1]), vp(cond[2]),
                                                     vp(out), batch, sample0, p, seed, C.c_void_p(ws_ptr), need,
                                                     C.c_void_p(stream)))
        ctx.model, ctx.batch, ctx.ws = model, batch, ws
        ctx.save_for_backward(*params)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        params = ctx.saved_tensors    # raises if a parameter was modified in place since the forward
        model, batch, ws = ctx.model, ctx.batch, ctx.ws
        if ws is None and batch > 0:
            raise RuntimeError("backward through the same training forward a second time: the saved activations were "
                               "released after the first backward (retain_graph is not supported)")
        ctx.ws = None
        lib = _capi.lib()
        n = lib.aft_param_count(model._handle)
        flat = torch.zeros(n, dtype=torch.float32, device=model.device)
        if batch > 0:
            g = torch.view_as_real(grad_out.to(torch.complex64).resolve_conj()).contiguous()
            ws_ptr = (ws.data_ptr() + 255) // 256 * 256
            need = lib.aft_train_workspace_bytes(model._handle, batch)
            with torch.cuda.device(model.device):
                stream = torch.cuda.current_stream(model.device).cuda_stream
                _capi.check(lib.aft_backward(model._handle, C.c_void_p(g.data_ptr()), batch, C.c_void_p(ws_ptr), need,
                                             C.c_void_p(flat.data_ptr()), C.c_void_p(stream)))
        grads, off = [], 0
        for i, t in enumerate(params):
            k = t.numel()
            grads.append(flat[off:off + k].view(t.shape).to(t.dtype) if ctx.needs_input_grad[7 + i] else None)
            off += k
        return (None, None, None, None, None, None, None, *grads)


class FortiTranEstimator(BaseFortiTranEstimator):
    """FortiTran: no channel adaptation (reference fortitran.py:253-268)."""

    def __init__(self, system_config: SystemConfig, model_config: ModelConfig) -> None:
        super().__init__(system_config, model_config, use_channel_adaptation=False)


class AdaFortiTranEstimator(BaseFortiTranEstimator):
    """AdaFortiTran: SNR / delay-spread / Doppler conditioned (reference adafortitran.py:5-22)."""

    def __init__(self, system_config: SystemConfig, model_config: ModelConfig) -> None:
        super().__init__(system_config, model_config, use_channel_adaptation=True)


class LinearEstimator(nn.Module):
    """Learned linear estimator ``h_hat = W h_pilot + b`` (reference src/models/linear.py:15-107): same constructor,
    attributes, ``state_dict`` keys (``linear.weight`` [out, in], ``linear.bias``) and shape check; the product runs in
    ``aft_linear_forward``.  Like the reference's ``nn.Linear`` it is a real-valued map: complex input is rejected.

    ``trainable`` (default ``False``): with ``True``, a ``forward`` with grad enabled is differentiable, in ``train()`` and
    ``eval()`` mode alike (the model has no dropout): ``loss.backward()`` fills ``.grad`` of the weight, the bias and, when
    it requires grad, the input through ``aft_linear_backward``.  The output equals the ``no_grad`` output bit for bit, and
    gradients come back in the dtype of the tensor they belong to."""

    trainable = False

    def __init__(self, system_config: SystemConfig, model_config: ModelConfig) -> None:
        super().__init__()
        self.system_config = system_config
        self.model_config = model_config
        self.device = torch.device(model_config.device)
        self.logger = logging.getLogger(__name__)
        self.ofdm_size = (system_config.ofdm.num_scs, system_config.ofdm.num_symbols)
        self.pilot_size = (system_config.pilot.num_scs, system_config.pilot.num_symbols)
        self.linear = nn.Linear(self.pilot_size[0] * self.pilot_size[1], self.ofdm_size[0] * self.ofdm_size[1])
        self.to(self.device)

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.device = self.linear.weight.device    # follow .to() / .cuda() / .cpu()
        return out

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        expected = (x.size(0), self.pilot_size[0], self.pilot_size[1])
        if tuple(x.size()) != expected:
            raise ValueError(f"Expected input shape {expected}, got {tuple(x.size())}")     # linear.py:76-80
        if x.is_complex():
            raise RuntimeError("LinearEstimator is a real-valued nn.Linear: complex input has no defined result "
                               "(the reference raises a dtype mismatch inside F.linear)")
        device = self.linear.weight.device
        if device.type != "cuda" or self.linear.bias.device != device:
            raise RuntimeError(f"adafortitran_b200 has no CPU fallback: the parameters live on '{device}', move the model "
                               "to a CUDA device (.to('cuda'))")
        if self.trainable and torch.is_grad_enabled():
            out = _LinearTrain.apply(x, self.linear.weight, self.linear.bias)
            return out.reshape(-1, self.ofdm_size[0], self.ofdm_size[1])
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("adafortitran_b200 is inference-only: call model.eval() or wrap the call in torch.no_grad()")
        out, _, _ = _linear_forward(x, self.linear.weight, self.linear.bias)
        return out.reshape(-1, self.ofdm_size[0], self.ofdm_size[1])

    def __repr__(self) -> str:
        return f"LinearEstimator(\n  ofdm_size={self.ofdm_size},\n  pilot_size={self.pilot_size},\n  device={self.device}\n)"


def _linear_forward(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor):
    """``aft_linear_forward`` on fp32, contiguous copies of the operands (no-ops for the reference's own layout) instead of
    pointers to anything else.  Returns the output [batch, out] and the fp32 weight and input it was computed from."""
    device = weight.device
    w = weight.detach().to(torch.float32).contiguous()
    b = bias.detach().to(torch.float32).contiguous()
    xin = x.detach().to(device=device, dtype=torch.float32).reshape(x.size(0), w.shape[1]).contiguous()
    out = torch.empty((x.size(0), w.shape[0]), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _capi.check(_capi.lib().aft_linear_forward(
            C.c_void_p(w.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(xin.data_ptr()),
            C.c_void_p(out.data_ptr()), x.size(0), w.shape[1], w.shape[0], C.c_void_p(stream)))
    return out, w, xin


class _LinearTrain(torch.autograd.Function):
    """``aft_linear_forward`` / ``aft_linear_backward`` behind autograd for :class:`LinearEstimator` with
    ``trainable = True``.  The input gradient is computed only when the input needs one."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        out, w, xin = _linear_forward(x, weight, bias)
        ctx.save_for_backward(w, xin)
        ctx.x_meta = (x.shape, x.dtype, x.device)
        ctx.param_dtypes = (weight.dtype, bias.dtype)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        w, xin = ctx.saved_tensors
        (x_shape, x_dtype, x_device), device = ctx.x_meta, w.device
        batch, (out_dim, in_dim) = xin.shape[0], w.shape
        gy = grad_out.to(device=device, dtype=torch.float32).contiguous()
        grad_w = torch.empty((out_dim, in_dim), dtype=torch.float32, device=device)
        grad_b = torch.empty(out_dim, dtype=torch.float32, device=device)
        grad_x = torch.empty((batch, in_dim), dtype=torch.float32, device=device) if ctx.needs_input_grad[0] else None
        lib = _capi.lib()
        need = lib.aft_linear_backward_workspace_bytes(batch, in_dim, out_dim)
        if need == 0:
            _capi.check(_capi.AFT_ERR_INVALID)
        ws = torch.empty(need, dtype=torch.uint8, device=device)
        vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            _capi.check(lib.aft_linear_backward(vp(w), vp(xin), vp(gy), vp(grad_w), vp(grad_b), vp(grad_x), batch, in_dim,
                                                out_dim, vp(ws), need, C.c_void_p(stream)))
        (w_dtype, b_dtype), (_, need_w, need_b) = ctx.param_dtypes, ctx.needs_input_grad
        return (grad_x.reshape(x_shape).to(device=x_device, dtype=x_dtype) if grad_x is not None else None,
                grad_w.to(w_dtype) if need_w else None, grad_b.to(b_dtype) if need_b else None)
