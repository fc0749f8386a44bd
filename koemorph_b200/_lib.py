"""ctypes binding of the C ABI declared in include/koemorph_b200.h.

There is deliberately no fallback: if the shared library is missing or no CUDA device is
present, importing the ops raises.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libkoemorph_b200.so")

KOE_NO_EDGE = -1000000
MAX_EDGE = 2
POOL_WARMUP = 1       # KOE_POOL_WARMUP: koe_stream_pool_create_ex2 flag
VARLEN_WARMUP = 1     # KOE_VARLEN_WARMUP: koe_forward_varlen_ex / koe_forward_varlen_size_ex flag
# 1 was reserved for a tf32 tensor-core core that was never built: the ABI rejects it
PRECISIONS = {"fp32": 0, "bf16": 2}


class CoreWeightsStruct(C.Structure):
    """Mirror of ``koe_core_weights`` (include/koemorph_b200.h)."""
    _fields_ = [
        ("k_mel", C.c_int32), ("k_mel_pad", C.c_int32), ("emo_in", C.c_int32), ("emo_in_pad", C.c_int32),
        ("b2", C.c_float), ("ln_eps", C.c_float),
        ("wc_t", C.c_void_p), ("bc", C.c_void_p), ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
        ("qk_t", C.c_void_p), ("wv_t", C.c_void_p), ("bv", C.c_void_p), ("wa_t", C.c_void_p),
        ("ba", C.c_void_p), ("w2", C.c_void_p), ("coef", C.c_void_p),
        ("mouth_idx", C.c_void_p), ("expr_idx", C.c_void_p),
        ("we1_t", C.c_void_p), ("be1", C.c_void_p), ("eln_g", C.c_void_p), ("eln_b", C.c_void_p),
        ("we2_t", C.c_void_p), ("be2", C.c_void_p),
        ("tc_bf16", C.c_void_p), ("tc_stages", C.c_int32), ("reserved_", C.c_int32),
        ("tc_bv", C.c_void_p),
    ]


class LogmelArgs(C.Structure):
    """Mirror of ``koe_logmel_args`` (include/koemorph_b200.h)."""
    _fields_ = [
        ("audio", C.c_void_p), ("audio_stride", C.c_int64),
        ("n_clips", C.c_int32), ("n_samples", C.c_int32), ("hop", C.c_int32), ("n_frames", C.c_int32),
        ("frame_offset", C.c_int32), ("frame_step", C.c_int32), ("sample_offset", C.c_int32),
        ("lo_rel_hops", C.c_int32), ("hi_rel_hops", C.c_int32), ("pad_mode", C.c_int32),
        ("power", C.c_void_p), ("power_clip_stride", C.c_int64),
        ("frame_max", C.c_void_p), ("frame_max_clip_stride", C.c_int64),
        ("power_b", C.c_void_p), ("power_b_clip_stride", C.c_int64),
        ("frame_max_b", C.c_void_p), ("frame_max_b_clip_stride", C.c_int64),
    ]


class StreamArgs(C.Structure):
    """koe_stream_args (include/koemorph_b200.h)."""
    _fields_ = [("frontend", C.c_void_p), ("weights", C.c_void_p),
                ("n_streams", C.c_int32), ("hop", C.c_int32), ("window_frames", C.c_int32), ("half_fft", C.c_int32),
                ("hop_audio", C.c_void_p), ("tail", C.c_void_p * 2),
                ("ring_f", C.c_void_p), ("fmax_f", C.c_void_p), ("ring_r", C.c_void_p), ("fmax_r", C.c_void_p),
                ("row_l", C.c_void_p), ("fmax_l", C.c_void_p),
                ("ring_r2", C.c_void_p), ("fmax_r2", C.c_void_p), ("row_l2", C.c_void_p), ("fmax_l2", C.c_void_p),
                ("expr_sigmoid", C.c_void_p), ("out", C.c_void_p),
                ("ema_state", C.c_void_p), ("alpha", C.c_float), ("has_state", C.c_int32), ("precision", C.c_int32),
                ("step", C.c_int64)]


class ForwardArgs(C.Structure):
    """koe_forward_args (include/koemorph_b200.h)."""
    _fields_ = [("frontend", C.c_void_p), ("weights", C.c_void_p), ("audio", C.c_void_p), ("audio_stride", C.c_int64),
                ("n_clips", C.c_int32), ("n_samples", C.c_int32), ("hop", C.c_int32),
                ("n_frames", C.c_int32), ("frames_per_window", C.c_int32), ("stride_frames", C.c_int32),
                ("n_out", C.c_int32), ("n_edge", C.c_int32),
                ("egemaps", C.c_void_p), ("power", C.c_void_p * (1 + 2 * MAX_EDGE)),
                ("frame_max", C.c_void_p * (1 + 2 * MAX_EDGE)), ("expr_sigmoid", C.c_void_p), ("out", C.c_void_p),
                ("sigmoid_out", C.c_void_p), ("attn_out", C.c_void_p), ("alpha", C.c_float), ("smooth", C.c_int32),
                ("precision", C.c_int32)]


class StreamPoolArgs(C.Structure):
    """koe_stream_pool_args (include/koemorph_b200.h)."""
    _fields_ = [("frontend", C.c_void_p), ("weights", C.c_void_p), ("hop_audio", C.c_void_p),
                ("tail", C.c_void_p), ("tail_compact", C.c_void_p), ("stage", C.c_void_p), ("stage_max", C.c_void_p),
                ("ring_f", C.c_void_p), ("fmax_f", C.c_void_p), ("ring_r", C.c_void_p), ("fmax_r", C.c_void_p),
                ("row_l", C.c_void_p), ("fmax_l", C.c_void_p),
                ("ring_r2", C.c_void_p), ("fmax_r2", C.c_void_p), ("row_l2", C.c_void_p), ("fmax_l2", C.c_void_p),
                ("expr_sigmoid", C.c_void_p), ("expr_compact", C.c_void_p), ("out", C.c_void_p),
                ("ema_state", C.c_void_p), ("tables", C.c_void_p), ("alpha", C.c_float), ("precision", C.c_int32)]


class ForwardVarlenArgs(C.Structure):
    """koe_forward_varlen_args (include/koemorph_b200.h)."""
    _fields_ = [("frontend", C.c_void_p), ("weights", C.c_void_p), ("audio", C.c_void_p), ("lengths_host", C.c_void_p),
                ("n_clips", C.c_int32), ("hop", C.c_int32), ("window_frames", C.c_int32), ("stride_frames", C.c_int32),
                ("half_fft", C.c_int32), ("smooth", C.c_int32), ("precision", C.c_int32), ("alpha", C.c_float),
                ("egemaps", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64), ("out", C.c_void_p),
                ("sigmoid_out", C.c_void_p), ("attn_out", C.c_void_p)]


class FrontendConfig(C.Structure):
    """koe_frontend_config (include/koemorph_b200.h)."""
    _fields_ = [("device", C.c_int32), ("sample_rate", C.c_int32), ("n_fft", C.c_int32), ("n_mels", C.c_int32),
                ("fmin", C.c_float), ("fmax", C.c_float), ("mel_scale", C.c_int32), ("mel_norm", C.c_int32),
                ("window_normalized", C.c_int32), ("log_mode", C.c_int32), ("log_eps", C.c_float),
                ("win_length", C.c_int32)]


_lib = None
_lock = threading.Lock()

_SIGNATURES = {
    "koe_last_error": (C.c_char_p, []),
    "koe_version": (C.c_int, []),
    "koe_launch_count": (C.c_int64, []),
    "koe_reset_launch_count": (None, []),
    "koe_frontend_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                      C.POINTER(C.c_void_p)]),
    "koe_frontend_create_ex": (C.c_int, [C.POINTER(FrontendConfig), C.POINTER(C.c_void_p)]),
    "koe_frontend_destroy": (C.c_int, [C.c_void_p]),
    "koe_frontend_filterbank_host": (C.c_int, [C.c_void_p, C.c_void_p]),
    "koe_frontend_uses_unrolled_bank": (C.c_int, [C.c_void_p]),
    "koe_logmel_power": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "koe_logmel_power_ex": (C.c_int, [C.c_void_p, C.POINTER(LogmelArgs), C.c_void_p]),
    "koe_dual_stream_ring": (C.c_int, [C.POINTER(CoreWeightsStruct), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "koe_dual_stream_ring_edges": (C.c_int, [C.POINTER(CoreWeightsStruct), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                             C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "koe_logmel_normalise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "koe_pcm16_to_float": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "koe_sizeof_struct": (C.c_int, [C.c_int]),
    "koe_stream_push": (C.c_int, [C.POINTER(StreamArgs), C.POINTER(C.c_int), C.c_void_p]),
    "koe_forward_windows": (C.c_int, [C.POINTER(ForwardArgs), C.c_void_p]),
    "koe_forward_varlen_size": (C.c_int, [C.POINTER(ForwardVarlenArgs), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                          C.POINTER(C.c_int64)]),
    "koe_forward_varlen": (C.c_int, [C.POINTER(ForwardVarlenArgs), C.c_void_p]),
    "koe_forward_varlen_size_ex": (C.c_int, [C.POINTER(ForwardVarlenArgs), C.c_int, C.POINTER(C.c_int64),
                                             C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "koe_forward_varlen_ex": (C.c_int, [C.POINTER(ForwardVarlenArgs), C.c_int, C.c_void_p]),
    "koe_stream_pool_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "koe_stream_pool_create_ex": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "koe_stream_pool_create_ex2": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(C.c_void_p)]),
    "koe_stream_pool_destroy": (C.c_int, [C.c_void_p]),
    "koe_stream_pool_open": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "koe_stream_pool_close": (C.c_int, [C.c_void_p, C.c_int]),
    "koe_stream_pool_set_egemaps": (C.c_int, [C.c_void_p, C.POINTER(StreamPoolArgs), C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_void_p]),
    "koe_stream_pool_push": (C.c_int, [C.c_void_p, C.POINTER(StreamPoolArgs), C.c_void_p, C.c_int, C.c_void_p,
                                       C.POINTER(C.c_int), C.c_void_p]),
    "koe_stream_pool_push_hops": (C.c_int, [C.c_void_p, C.POINTER(StreamPoolArgs), C.c_void_p, C.c_void_p, C.c_int,
                                            C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_void_p]),
    "koe_stream_pool_state_floats": (C.c_int, [C.c_void_p]),
    "koe_stream_pool_snapshot": (C.c_int, [C.c_void_p, C.POINTER(StreamPoolArgs), C.c_void_p, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "koe_stream_pool_restore": (C.c_int, [C.c_void_p, C.POINTER(StreamPoolArgs), C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p]),
    "koe_affine_rows": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "koe_emotion_stream": (C.c_int, [C.POINTER(CoreWeightsStruct), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "koe_dual_stream_windows": (C.c_int, [C.POINTER(CoreWeightsStruct), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p]),
    "koe_dual_stream_features": (C.c_int, [C.POINTER(CoreWeightsStruct), C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "koe_ema_scan": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p]),
}


def exported_symbols():
    """Names every build of the library must export (checked by the CPU test-suite)."""
    return sorted(_SIGNATURES)


def load() -> C.CDLL:
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"koemorph_b200: CUDA library not built ({LIB_PATH} missing). Run "
                    "`python -m koemorph_b200.build` (needs nvcc). There is no CPU fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name, None)
                if fn is None:
                    continue  # optional symbols are checked by the caller
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().koe_last_error()
        raise RuntimeError(f"koemorph_b200 {what} failed (code {rc}): {msg.decode() if msg else ''}")


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    """Validate a tensor the kernels will read: CUDA, expected dtype, contiguous."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (got {t.device}); koemorph_b200 has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def launch_count() -> int:
    return int(load().koe_launch_count())


def reset_launch_count() -> None:
    load().koe_reset_launch_count()
