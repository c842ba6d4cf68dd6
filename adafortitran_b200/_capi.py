"""ctypes binding of ``include/aft.h`` (the C-ABI of ``libaft_b200.so``).

This is the stub a maintainer of the reference would add to call the B200 library from Python; it
mirrors the header one to one (see INTEGRATION.md).  There is no fallback: if the shared object is
missing or cannot be loaded, :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

AFT_ABI_VERSION = 3
AFT_OK = 0
AFT_ERR_INVALID, AFT_ERR_UNSUPPORTED, AFT_ERR_CUDA, AFT_ERR_WORKSPACE, AFT_ERR_STATE = -1, -2, -3, -4, -5
AFT_FP32, AFT_BF16 = 0, 1
AFT_ACT_RELU, AFT_ACT_GELU = 0, 1

_fp = C.POINTER(C.c_float)


class AftConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "num_scs", "num_symbols", "pilot_scs", "pilot_symbols", "patch_scs", "patch_symbols", "num_layers",
        "model_dim", "num_head", "ff_dim", "activation", "adaptive", "adapt_h1", "adapt_h2", "adapt_h3",
        "adaptive_token_length", "max_seq_len")]


class AftConvStack(C.Structure):
    _fields_ = [("w", _fp * 4), ("b", _fp * 4)]


class AftMlp(C.Structure):
    _fields_ = [("w", _fp * 3), ("b", _fp * 3)]


class AftEncoderLayer(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
        "norm1_w", "norm1_b", "norm2_w", "norm2_b")]


class AftWeights(C.Structure):
    _fields_ = [
        ("upsampler_w", _fp), ("upsampler_b", _fp),
        ("initial_enhancer", AftConvStack), ("final_refiner", AftConvStack),
        ("snr_encoder", AftMlp), ("ds_encoder", AftMlp), ("dop_encoder", AftMlp),
        ("linear_1_w", _fp), ("linear_1_b", _fp), ("pos_table", _fp),
        ("linear_2_w", _fp), ("linear_2_b", _fp),
        ("layers", C.POINTER(AftEncoderLayer)), ("num_layers", C.c_int32),
    ]


class AftGather(C.Structure):
    """Plan of the fused all-gather (``include/aft.h``): gather buffers of all ranks as mapped into this process."""
    _fields_ = [("peer_out", C.c_void_p * 8), ("world", C.c_int32), ("rank", C.c_int32), ("rows_per_rank", C.c_int64),
                ("row0", C.c_int64)]


EXPORTS = {
    # name: (restype, argtypes)
    "aft_abi_version": (C.c_int, []),
    "aft_last_error": (C.c_char_p, []),
    "aft_create": (C.c_int, [C.POINTER(AftConfig), C.POINTER(C.c_void_p)]),
    "aft_destroy": (None, [C.c_void_p]),
    "aft_load_weights": (C.c_int, [C.c_void_p, C.POINTER(AftWeights), C.c_void_p]),
    "aft_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int]),
    "aft_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "aft_forward_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int64, C.c_int]),
    "aft_forward_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(AftGather)]),
    "aft_forward_host_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int64, C.c_int, C.POINTER(AftGather)]),
    "aft_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]),
    "aft_peer_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "aft_peer_close": (C.c_int, [C.c_void_p]),
    "aft_peer_free": (C.c_int, [C.c_void_p]),
    "aft_error_sums": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "aft_extract_pilots": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "aft_linear_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "aft_linear_backward_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "aft_linear_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                      C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "aft_synthetic_channels": (C.c_int, [C.POINTER(AftConfig), C.c_uint64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "aft_launch_count": (C.c_int64, []),
    "aft_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "aft_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "aft_selftest": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.c_void_p]),
    "aft_param_count": (C.c_int64, [C.c_void_p]),
    "aft_train_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64]),
    "aft_forward_train": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                    C.c_float, C.c_uint64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "aft_forward_train_offset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.c_int64, C.c_float, C.c_uint64, C.c_void_p, C.c_size_t,
                                           C.c_void_p]),
    "aft_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
}

_LIB = None
_LOCK = threading.Lock()


def lib_path() -> str:
    return os.environ.get("AFT_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib",
                                                         "libaft_b200.so")


class AftError(RuntimeError):
    """A C-ABI call returned a negative status."""

    def __init__(self, status: int, message: str):
        super().__init__(f"libaft_b200 status {status}: {message}")
        self.status = status


def lib() -> C.CDLL:
    """Load (once) and return the shared library.  Raises if it is missing -- no fallback."""
    global _LIB
    with _LOCK:
        if _LIB is None:
            path = lib_path()
            if not os.path.exists(path):
                raise RuntimeError(
                    f"{path} not found: build it with `python -m adafortitran_b200.build` "
                    "(the CUDA extension is mandatory; there is no CPU / PyTorch fallback path)")
            handle = C.CDLL(path)
            for name, (res, args) in EXPORTS.items():
                fn = getattr(handle, name)      # AttributeError if the symbol is not exported
                fn.restype, fn.argtypes = res, args
            if handle.aft_abi_version() != AFT_ABI_VERSION:
                raise RuntimeError(f"{path}: ABI version {handle.aft_abi_version()} != {AFT_ABI_VERSION}")
            _LIB = handle
    return _LIB


def check(status: int) -> None:
    if status != AFT_OK:
        msg = lib().aft_last_error().decode("utf-8", "replace")
        if status in (AFT_ERR_INVALID, AFT_ERR_UNSUPPORTED):
            err = ValueError(f"libaft_b200 status {status}: {msg}")
            err.status = status
            raise err
        raise AftError(status, msg)
