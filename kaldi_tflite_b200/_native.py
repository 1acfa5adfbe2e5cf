"""
ctypes binding of libktf_b200.so (include/ktf_b200.h).

There is NO fallback: if the shared library is missing or the device is not a
CUDA device, importing the layers still works (so configs can be inspected on a
CPU box) but the first call that needs a kernel raises `KtfNativeError`.
"""

import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_int64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libktf_b200.so")

KTF_OUT_MFCC, KTF_OUT_FBANK, KTF_OUT_WINDOWED = 0, 1, 2
KTF_SAMPLE_F32, KTF_SAMPLE_S16 = 0, 1
KTF_PREC_F32, KTF_PREC_BF16 = 0, 1
KTF_ACT_NONE, KTF_ACT_RELU = 0, 1
KTF_SCORES_NATIVE, KTF_SCORES_BF16 = 0, 1
KTF_MAX_CONTEXT = 16
KTF_PLDA_TOPK_MAX = 32
KTF_NCCL_UNIQUE_ID_BYTES = 128
KTF_EINVAL, KTF_ECUDA, KTF_ENOMEM = -1, -2, -3


class KtfNativeError(RuntimeError):
    pass


class FrontendCfg(Structure):
    _fields_ = [("frame_width", c_int32), ("frame_shift", c_int32), ("fft_length", c_int32),
                ("num_mels", c_int32), ("num_ceps", c_int32), ("output", c_int32),
                ("remove_dc_offset", c_int32), ("raw_energy", c_int32), ("use_energy", c_int32),
                ("use_power", c_int32), ("use_log_fbank", c_int32), ("apply_lifter", c_int32),
                ("preemphasis", c_float), ("energy_floor", c_float), ("epsilon", c_float), ("dither", c_float)]


class VadCfg(Structure):
    _fields_ = [("energy_threshold", c_float), ("energy_mean_scale", c_float),
                ("proportion_threshold", c_float), ("frames_context", c_int32),
                ("energy_coeff", c_int32)]


class AffineCfg(Structure):
    _fields_ = [("in_dim", c_int32), ("out_dim", c_int32), ("num_context", c_int32),
                ("context", c_int32 * KTF_MAX_CONTEXT), ("subsampling_factor", c_int32),
                ("padding_valid", c_int32), ("activation", c_int32), ("precision", c_int32)]


_P = c_void_p
_SIGNATURES = {
    "ktf_last_error": (c_char_p, []),
    "ktf_version": (c_int32, []),
    "ktf_device_arch": (c_int32, []),
    "ktf_launch_count": (c_int64, []),
    "ktf_set_dither_seed": (c_int32, [ctypes.c_uint64]),
    "ktf_ctx_create": (c_int32, [c_int32, POINTER(_P)]),
    "ktf_ctx_destroy": (None, [_P]),
    "ktf_ctx_device": (c_int32, [_P]),
    "ktf_ctx_stream": (_P, [_P]),
    "ktf_ctx_synchronize": (c_int32, [_P]),
    "ktf_ctx_malloc": (c_int32, [_P, c_int64, POINTER(_P)]),
    "ktf_ctx_free": (c_int32, [_P, _P]),
    "ktf_ctx_memcpy_h2d": (c_int32, [_P, _P, _P, c_int64]),
    "ktf_ctx_memcpy_d2h": (c_int32, [_P, _P, _P, c_int64]),
    "ktf_nccl_available": (c_int32, []),
    "ktf_nccl_unique_id": (c_int32, [_P]),
    "ktf_nccl_comm_init": (c_int32, [_P, c_int32, c_int32, _P]),
    "ktf_nccl_comm_destroy": (c_int32, [_P]),
    "ktf_nccl_allgather_xvec": (c_int32, [_P, _P, _P, c_int64, c_int32, c_int32, _P]),
    "ktf_frontend_create": (c_int32, [POINTER(FrontendCfg), _P, _P, _P, _P, POINTER(_P)]),
    "ktf_frontend_destroy": (None, [_P]),
    "ktf_frontend_num_frames": (c_int64, [_P, c_int64]),
    "ktf_frontend_out_dim": (c_int32, [_P]),
    "ktf_frontend_forward": (c_int32, [_P, _P, c_int64, c_int64, c_int64, _P, _P, _P]),
    "ktf_frontend_forward_ragged": (c_int32, [_P, _P, c_int64, _P, _P, _P, _P, _P]),
    "ktf_frontend_num_frames_ex": (c_int64, [_P, c_int64, c_int32]),
    "ktf_frontend_forward_ex": (c_int32, [_P, _P, c_int32, c_int32, c_int64, c_int64, c_int64, _P, _P, _P]),
    "ktf_frontend_forward_ragged_ex": (c_int32, [_P, _P, c_int32, c_int32, c_int64, _P, _P, _P, _P, _P]),
    "ktf_framing_forward": (c_int32, [_P, c_int64, c_int64, c_int64, c_int32, c_int32, _P, _P]),
    "ktf_vad_mask": (c_int32, [POINTER(VadCfg), _P, c_int32, _P, c_int64, c_int64, _P, _P]),
    "ktf_vad_compact_workspace": (c_int64, [c_int64, c_int64]),
    "ktf_vad_compact": (c_int32, [_P, c_int32, _P, _P, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "ktf_cmvn_forward": (c_int32, [_P, c_int32, _P, c_int64, c_int64, c_int64, c_int32, c_int32, c_int32, _P, _P, _P]),
    "ktf_affine_create": (c_int32, [POINTER(AffineCfg), _P, _P, _P, _P, POINTER(_P)]),
    "ktf_affine_destroy": (None, [_P]),
    "ktf_affine_out_rows": (c_int64, [_P, c_int64]),
    "ktf_affine_forward": (c_int32, [_P, _P, _P, _P, c_int64, c_int64, c_int64, _P, _P, _P]),
    "ktf_tdnn_stack_create": (c_int32, [POINTER(_P), c_int32, c_int32, c_int32, c_float, POINTER(_P)]),
    "ktf_tdnn_stack_destroy": (None, [_P]),
    "ktf_tdnn_stack_out_dim": (c_int32, [_P]),
    "ktf_tdnn_stack_forward": (c_int32, [_P, _P, _P, c_int64, c_int64, _P, _P]),
    "ktf_tdnn_stack_forward_vad": (c_int32, [_P, _P, _P, _P, c_int64, c_int64, c_int64, c_int32, _P, _P]),
    "ktf_tdnn_stack_vad_prepass_fits": (c_int32, [_P, c_int32, c_int64]),
    "ktf_relu_forward": (c_int32, [_P, c_int64, _P, _P]),
    "ktf_scale_offset_forward": (c_int32, [_P, c_int64, c_int32, _P, _P, _P, _P]),
    "ktf_stats_finalize": (c_int32, [_P, _P, c_int64, c_int32, c_int32, c_float, c_int32, _P, _P]),
    "ktf_stats_reduce": (c_int32, [_P, _P, c_int64, c_int32, c_int32, c_int32, c_float, _P, _P]),
    "ktf_stats_windows": (c_int32, [_P, c_int64, c_int64, c_int32, c_int32, c_int32, c_int32, c_int64,
                                    c_int64, c_int32, c_int32, c_int32, c_float, _P, _P]),
    "ktf_lda_forward": (c_int32, [_P, c_int64, c_int32, c_int32, _P, _P, c_int32, _P, _P]),
    "ktf_plda_create": (c_int32, [c_int32, _P, _P, _P, c_int32, c_int32, c_int32, POINTER(_P)]),
    "ktf_plda_create_ex": (c_int32, [c_int32, _P, _P, _P, c_int32, c_int32, c_int32, c_double, POINTER(_P)]),
    "ktf_plda_destroy": (None, [_P]),
    "ktf_plda_transform": (c_int32, [_P, _P, c_int64, _P, _P]),
    "ktf_plda_score": (c_int32, [_P, _P, c_int64, _P, c_int64, _P, c_int64, _P]),
    "ktf_plda_score_ex": (c_int32, [_P, _P, c_int64, _P, c_int64, _P, c_int64, c_int32, _P]),
    "ktf_plda_score_top1": (c_int32, [_P, _P, c_int64, _P, c_int64, _P, _P, _P]),
    "ktf_plda_score_topk": (c_int32, [_P, _P, c_int64, _P, c_int64, c_int32, _P, _P, _P]),
    "ktf_topk_merge": (c_int32, [_P, _P, c_int32, c_int64, c_int32, c_int32, _P, _P, _P]),
}

_lib = None


def exported_symbols():
    """Names every entry point include/ktf_b200.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGNATURES)


def lib():
    """Loads the shared library on first use; raises KtfNativeError if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KtfNativeError(
                f"{LIB_PATH} is missing: build it with `python -m kaldi_tflite_b200.build` "
                "(there is no CPU fallback)")
        try:
            l = ctypes.CDLL(LIB_PATH)
        except OSError as e:
            raise KtfNativeError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def last_error():
    return lib().ktf_last_error().decode(errors="replace")


def check(rc):
    """Maps a ktf return code to the exception type the reference raises in the same situation."""
    if rc == 0:
        return
    msg = last_error()
    if rc == KTF_EINVAL:
        raise ValueError(msg)
    if rc == KTF_ENOMEM:
        raise MemoryError(msg)
    raise KtfNativeError(msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise KtfNativeError("no CUDA device: kaldi_tflite_b200 has no CPU path")
    lib()


def launch_count():
    return int(lib().ktf_launch_count())
