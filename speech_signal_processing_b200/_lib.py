"""ctypes binding of ``libssp_b200.so`` (the C ABI declared in ``include/ssp_b200.h``).

There is no CPU fallback: if the library has not been built, or no CUDA device is present
when a kernel is requested, the call raises.
"""
from __future__ import annotations

import ctypes as C
import functools
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SSP_B200_LIB") or os.path.join(PKG, "libssp_b200.so")  # override: A/B a second build

PREC_FP32 = 0
PREC_TF32 = 1
PREC_TF32X2 = 2
PREC_TF32X3 = 3


class SspError(RuntimeError):
    pass


class FrontendCfg(C.Structure):
    _fields_ = [
        ("frame_len", C.c_int32), ("frame_shift", C.c_int32), ("nfft", C.c_int32), ("n_filt", C.c_int32),
        ("n_ceps", C.c_int32), ("framing", C.c_int32), ("preemph_mode", C.c_int32), ("preemph", C.c_float),
        ("spec_type", C.c_int32), ("spec_scale", C.c_float), ("log_type", C.c_int32), ("log_add", C.c_float),
        ("log_zero_floor", C.c_float), ("energy_mode", C.c_int32), ("delta_order", C.c_int32),
        ("delta_n", C.c_int32), ("cmvn", C.c_int32), ("pcm_dtype", C.c_int32),
    ]


class VadCfg(C.Structure):
    _fields_ = [("frame_len", C.c_int32), ("frame_shift", C.c_int32), ("n_blocks", C.c_int32), ("normalize_peak", C.c_int32),
                ("pcm_dtype", C.c_int32), ("eps", C.c_float)]


class GmmDims(C.Structure):
    _fields_ = [("n_models", C.c_int32), ("n_comp", C.c_int32), ("n_feat", C.c_int32)]


_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32

# name -> (restype, argtypes); mirrors include/ssp_b200.h one to one
PROTOTYPES = {
    "ssp_abi_version": (C.c_int, []),
    "ssp_last_error": (C.c_char_p, []),
    "ssp_launch_count": (_I64, []),
    "ssp_reset_launch_count": (None, []),
    "ssp_launch_log": (C.c_char_p, []),
    "ssp_frontend_num_frames": (_I64, [C.POINTER(FrontendCfg), _I64]),
    "ssp_frontend_max_frames": (_I64, [C.POINTER(FrontendCfg)]),
    "ssp_frontend_batch": (C.c_int, [_P, _P, _I64, C.POINTER(FrontendCfg), _P, _P, _P, _P, _P, _P, _P, _I64, _P, _P, _P]),
    "ssp_plp_post": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, _P, _P, _I32, _P, _P]),
    "ssp_mel_db_post": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, C.c_float, _P, _P]),
    "ssp_delta": (C.c_int, [_P, _I64, _I32, _I32, _P, _P]),
    "ssp_cmvn": (C.c_int, [_P, _P, _I64, _I32, _P, _P]),
    "ssp_vad_num_frames": (_I64, [C.POINTER(VadCfg), _I64]),
    "ssp_vad_features": (C.c_int, [_P, _P, _I64, C.POINTER(VadCfg), _P, _P, _P, _P, _P]),
    "ssp_vad_detect": (C.c_int, [_P, _P, _P, _I64, C.c_float, C.c_double, C.c_double, _I32, _P, _P]),
    "ssp_gmm_pack_bytes": (_I64, [C.POINTER(GmmDims)]),
    "ssp_gmm_pack_models": (C.c_int, [_P, _P, _P, C.POINTER(GmmDims), _P, _P]),
    "ssp_gmm_score": (C.c_int, [_P, _P, _I64, _I64, _P, C.POINTER(GmmDims), _I32, _P, _P, _P]),
    "ssp_gmm_shared_pack_bytes": (_I64, [C.POINTER(GmmDims)]),
    "ssp_gmm_pack_shared": (C.c_int, [_P, _P, _P, C.POINTER(GmmDims), _I32, _P, _P]),
    "ssp_gmm_score_shared_workspace_bytes": (_I64, [C.POINTER(GmmDims), _I64]),
    "ssp_gmm_score_shared": (C.c_int, [_P, _P, _I64, _I64, _P, C.POINTER(GmmDims), _P, _P, _P, _I64, _P]),
    "ssp_gmm_stats": (C.c_int, [_P, _P, _I64, _I64, _P, C.POINTER(GmmDims), _P, _P, _P, _P, _P, _P, _I64, _I32, _P]),
    "ssp_gmm_stats_workspace_bytes": (_I64, [C.POINTER(GmmDims), _I64, _I64]),
    "ssp_gmm_posteriors": (C.c_int, [_P, _P, _I64, _I64, _P, C.POINTER(GmmDims), _P, _P, _P, _P, _I64, _I32, _P]),
    "ssp_gmm_posteriors_workspace_bytes": (_I64, [C.POINTER(GmmDims), _I64, _I64]),
    "ssp_gmm_mstep": (C.c_int, [_P, _P, _P, _I32, _I32, _I32, C.c_double, C.c_double, _P, _P, _P, _P]),
    "ssp_gmm_map_adapt": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _P, _I32, _I32, C.c_double, _I32, _P, _P, _P, _P]),
    "ssp_dtw_max_len": (_I64, [_I32]),
    "ssp_dtw_batch": (C.c_int, [_P, _P, _I64, _P, _P, _I64, _I32, _I32, _I64, _P, _P]),
    "ssp_dtw_full": (C.c_int, [_P, _I64, _P, _I64, _I32, _I32, _P, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once) and set the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SspError(
            f"{LIB_PATH} is missing: build it with `python -m speech_signal_processing_b200.build` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ssp_abi_version() != 1:
        raise SspError(f"ABI version mismatch: library {lib.ssp_abi_version()}, binding 1")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().ssp_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(msg or what)
        if rc == -3:
            raise NotImplementedError(msg or what)
        raise SspError(f"{what}: {msg} (rc={rc})")


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise SspError("speech_signal_processing_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def on_device(fn):
    """Method decorator: run with ``self.device`` as the current CUDA device, so that the kernels launch in that
    device's context on ITS current stream (``stream_ptr``) whatever device the caller had selected."""
    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        import torch

        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


def ptr(t) -> int:
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load().ssp_launch_count())


def launch_log() -> dict:
    """{kernel name: launches} since the last ``ssp_reset_launch_count``."""
    text = load().ssp_launch_log().decode()
    return {k: int(v) for k, v in (item.rsplit(":", 1) for item in text.split(",") if item)}
