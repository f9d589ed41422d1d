"""ctypes binding of librf_b200.so (the C-ABI declared in include/rf_b200.h).

PyTorch is only plumbing here: tensors own the device memory, `data_ptr()` and the current
CUDA stream are handed to the library.  There is no CPU fallback — if the library is missing
or no sm_100 GPU is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

import numpy as np
import torch

_PKG = Path(__file__).resolve().parent.parent
_LIB_PATH = Path(os.environ.get("RF_B200_LIB", _PKG / "librf_b200.so"))


class NativeError(RuntimeError):
    pass


class PlanDesc(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int32),
        ("n_fft", C.c_int32),
        ("win_length", C.c_int32),
        ("hop_length", C.c_int32),
        ("n_mels", C.c_int32),
        ("f_min", C.c_float),
        ("f_max", C.c_float),
        ("mel_norm_slaney", C.c_int32),
        ("mel_scale_slaney", C.c_int32),
        ("full_band", C.c_int32),
    ]


class GemmDesc(C.Structure):
    _fields_ = [
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("batch1", C.c_int32), ("batch2", C.c_int32),
        ("A", C.c_void_p), ("lda", C.c_int64), ("sa1", C.c_int64), ("sa2", C.c_int64),
        ("B", C.c_void_p), ("ldb", C.c_int64), ("sb1", C.c_int64), ("sb2", C.c_int64),
        ("D", C.c_void_p), ("ldd", C.c_int64), ("sd1", C.c_int64), ("sd2", C.c_int64),
        ("bias", C.c_void_p), ("bias_mode", C.c_int32),
        ("residual", C.c_void_p), ("ldr", C.c_int64), ("sr1", C.c_int64), ("sr2", C.c_int64),
        ("alpha", C.c_float), ("act", C.c_int32), ("out_f32", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


class ConvDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C1", C.c_int32), ("C2", C.c_int32),
        ("Cout", C.c_int32), ("ksize", C.c_int32), ("stride", C.c_int32),
        ("x1", C.c_void_p), ("x2", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p),
        ("bias_per_image", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p),
        ("alpha", C.c_float), ("act", C.c_int32), ("bias_per_image_pitch", C.c_int32), ("pad_mode", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


class PlanInfo(C.Structure):
    _fields_ = [
        ("n_freq", C.c_int32),
        ("n_live", C.c_int32),
        ("k_lo", C.c_int32),
        ("k_hi", C.c_int32),
        ("n_even", C.c_int32),
        ("fb_nnz", C.c_int32),
        ("chunk_frames", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/rf_b200.h declares
SIGNATURES = {
    "rf_last_error": (C.c_char_p, []),
    "rf_version": (C.c_char_p, []),
    "rf_plan_create": (C.c_int, [C.POINTER(PlanDesc), C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "rf_plan_destroy": (None, [C.c_void_p]),
    "rf_plan_get_info": (C.c_int, [C.c_void_p, C.POINTER(PlanInfo)]),
    "rf_plan_set_decimation": (C.c_int, [C.c_void_p, C.c_int]),
    "rf_plan_table": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t]),
    "rf_inverse_mel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_griffinlim_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
    "rf_griffinlim": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rf_mel_to_wave": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rf_mel_to_wave_profiled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                          C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rf_stft_mel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_stft": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_mel_scale": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_gemm_f16": (C.c_int, [C.POINTER(GemmDesc), C.c_void_p]),
    "rf_conv2d_f16": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p]),
    "rf_gemm_workspace_bytes": (C.c_size_t, [C.POINTER(GemmDesc)]),
    "rf_conv2d_workspace_bytes": (C.c_size_t, [C.POINTER(ConvDesc)]),
    "rf_group_norm_scratch_floats": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "rf_group_norm_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float,
                                    C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rf_group_norm_cat_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rf_layer_norm_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                    C.c_void_p]),
    "rf_geglu_f16": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_softmax_rows_f16": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_upsample2x_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_concat_channels_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_conv1x1_small_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float,
                                       C.c_void_p, C.c_void_p]),
    "rf_vae_image_to_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_vae_image_to_u8_f32scale": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_conv_in_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p]),
    "rf_conv_out_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p]),
    "rf_timestep_embedding_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_silu_f16": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]),
    "rf_slerp_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_long, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                               C.c_void_p]),
    "rf_cfg_pndm_step_f16": (C.c_int, [C.c_void_p, C.c_long, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "rf_cfg_dpmpp_step_f16": (C.c_int, [C.c_void_p, C.c_long, C.c_float, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                                        C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rf_axpby_f16":(C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_long,
                               C.c_void_p, C.c_void_p]),
    "rf_add_noise_f16_seq": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_long, C.c_void_p, C.c_void_p]),
    "rf_resample_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_resample_coeffs": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rf_image_u8_to_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rf_attention_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "rf_attention_masked_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "rf_tc_profile_begin": (C.c_int, []),
    "rf_tc_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_long)]),
    "rf_image_to_mel": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p,
                                  C.c_void_p]),
    "rf_mel_to_image": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "rf_wave_to_int16": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """Load the shared library (once). Raises NativeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not _LIB_PATH.exists():
                raise NativeError(
                    f"{_LIB_PATH} not found: build it with `python riffusion-hobby_b200/build.py` "
                    "(nvcc, sm_100a). There is no CPU fallback."
                )
            handle = C.CDLL(str(_LIB_PATH))
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)  # AttributeError if a declared symbol is not exported
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().rf_last_error().decode("utf-8", "replace")
        if rc == 1:
            raise ValueError(msg)
        if rc == 3:
            raise NotImplementedError(msg)
        raise NativeError(msg)


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str, dtype: torch.dtype) -> torch.Tensor:
    if not t.is_cuda:
        raise NativeError(f"{name} must be a CUDA tensor (no CPU fallback); got device {t.device}")
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


class Plan:
    """Owns an rf_plan*. Tables are host-side until the first device call."""

    def __init__(self, desc: PlanDesc, window: np.ndarray | None = None, fb: np.ndarray | None = None):
        self._h = C.c_void_p()
        w = None if window is None else np.ascontiguousarray(window, dtype=np.float32)
        f = None if fb is None else np.ascontiguousarray(fb, dtype=np.float32)
        if w is not None and w.shape != (desc.win_length,):
            raise ValueError("window must have win_length entries")
        if f is not None and f.shape != (desc.n_fft // 2 + 1, desc.n_mels):
            raise ValueError("fb must be (n_fft//2+1, n_mels)")
        check(lib().rf_plan_create(C.byref(desc), None if w is None else w.ctypes.data,
                                   None if f is None else f.ctypes.data, C.byref(self._h)))
        self.desc = desc
        info = PlanInfo()
        check(lib().rf_plan_get_info(self._h, C.byref(info)))
        self.info = info

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def set_decimation(self, enable: bool) -> bool:
        """Griffin-Lim's half-rate inner loop (include/rf_b200.h: rf_plan_set_decimation); returns whether it is on."""
        r = lib().rf_plan_set_decimation(self._h, int(bool(enable)))
        if r < 0:
            check(r)
        return bool(r)

    def table(self, name: str, dtype, shape) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        check(lib().rf_plan_table(self._h, name.encode(), out.ctypes.data, out.nbytes))
        return out

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.rf_plan_destroy(h)
