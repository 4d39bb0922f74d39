"""ctypes binding of ``libste_ukf.so`` (the C ABI declared in ``include/ste_ukf.h``).

PyTorch tensors are only the buffer carrier: every call receives ``tensor.data_ptr()`` values and
the current CUDA stream handle.  There is no CPU implementation behind these functions; if the
library is missing, or a tensor is not a CUDA tensor, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import build as _build

# --- mirror of include/ste_ukf.h ------------------------------------------------------------ #
STE_ABI_VERSION = 7
STE_OK, STE_ERR_INVALID_ARG, STE_ERR_CUDA, STE_ERR_UNSUPPORTED = 0, -1, -2, -3
STE_FLAG_GATING, STE_FLAG_FORCE_GENERIC, STE_FLAG_PACKED_COV, STE_FLAG_LONG_STEPS = 0x1, 0x2, 0x4, 0x8
STE_STATUS_NONFINITE = 0x1
STE_STATUS_INDEFINITE = 0x2
STE_STATUS_GATE_CAP = 0x4
STE_STATUS_OBS_OVERRUN = 0x8
STE_STATUS_RANK_DEFICIENT = 0x10
STE_STATUS_SMOOTH_RECOMPUTE = 0x100
STATS_PLANES = 15
STE_GEODESY_SPHERE, STE_GEODESY_WGS84 = 0, 1
STE_MODEL_GEODETIC, STE_MODEL_GEODETIC_TURN = 0, 1

_dptr = C.c_void_p  # device pointers travel as plain integers


class SteProblem(C.Structure):
    _fields_ = [
        ("n_tracks", C.c_int32),
        ("max_steps", C.c_int32),
        ("max_obs", C.c_int32),
        ("substeps", C.c_int32),
        ("rate_repeat", C.c_int32),
        ("flags", C.c_uint32),
        ("gate_max_iter", C.c_int32),
        ("reserved", C.c_int32),
        ("ld", C.c_int64),
        ("gate_chi", C.c_double),
        ("H", C.c_double * 16),
        ("Q", C.c_double * 16),
        ("R", C.c_double * 16),
        ("P0", C.c_double * 16),
    ]


class SteInputs(C.Structure):
    _fields_ = [
        ("x0", _dptr),
        ("P0", _dptr),
        ("dt", _dptr),
        ("upd_mask", _dptr),
        ("n_steps", _dptr),
        ("z", _dptr * 4),
        ("sog_rate", _dptr),
        ("cog_rate", _dptr),
        ("rate_repeat", _dptr),
        ("noise_pred", _dptr),
        ("noise_upd", _dptr),
        ("noise_bwd", _dptr),
        ("R_tracks", _dptr),
    ]


class SteOutputs(C.Structure):
    _fields_ = [
        ("mean_f", _dptr),
        ("cov_f", _dptr),
        ("mean_s", _dptr),
        ("cov_s", _dptr),
        ("status", _dptr),
        ("n_updates", _dptr),
        ("gate_iters", _dptr),
        ("gate_lambda", _dptr),
        ("gate_scale", _dptr),
        ("smooth_stats", _dptr),
    ]


class SteProblemN(C.Structure):
    _fields_ = [
        ("n", C.c_int32),
        ("model", C.c_int32),
        ("n_tracks", C.c_int32),
        ("max_steps", C.c_int32),
        ("max_obs", C.c_int32),
        ("reserved", C.c_int32),
        ("ld", C.c_int64),
        ("H", C.c_double * 64),
        ("Q", C.c_double * 64),
        ("R", C.c_double * 64),
        ("P0", C.c_double * 64),
    ]


class SteInputsN(C.Structure):
    _fields_ = [
        ("x0", _dptr),
        ("P0", _dptr),
        ("dt", _dptr),
        ("upd_mask", _dptr),
        ("n_steps", _dptr),
        ("z", _dptr * 8),
        ("sog_rate", _dptr),
        ("cog_rate", _dptr),
        ("rate_repeat", _dptr),
        ("noise_pred", _dptr),
        ("noise_upd", _dptr),
        ("noise_bwd", _dptr),
    ]


class SteNoiseN(C.Structure):
    _fields_ = [
        ("Q_tracks", _dptr),
        ("R_tracks", _dptr),
    ]


class SteInnovations(C.Structure):
    _fields_ = [
        ("nis", _dptr),
        ("loglik", _dptr),
        ("rank", _dptr),
    ]


class SteOutputsN(C.Structure):
    _fields_ = [
        ("mean_f", _dptr),
        ("cov_f", _dptr),
        ("mean_s", _dptr),
        ("cov_s", _dptr),
        ("status", _dptr),
        ("n_updates", _dptr),
    ]


STE_MAX_CANDIDATES = 32


class SteCandidates(C.Structure):
    _fields_ = [
        ("n_cand", C.c_int32),
        ("reserved", C.c_int32),
        ("Q", C.POINTER(C.c_double)),   # host [n_cand][n*n]
        ("R", C.POINTER(C.c_double)),
    ]


class SteScores(C.Structure):
    _fields_ = [
        ("loglik", _dptr),
        ("nis", _dptr),
        ("dof", _dptr),
        ("n_updates", _dptr),
        ("status", _dptr),
        ("ld_out", C.c_int64),
    ]


STE_TEXT_MAX_COLS, STE_TEXT_MAX_TABLES, STE_TEXT_MAX_VALUE_BYTES = 8, 8, 27


class SteTextTable(C.Structure):
    _fields_ = [
        ("base", _dptr),
        ("track", _dptr),
        ("ld", C.c_int64),
        ("n_tracks", C.c_int32),
        ("row_stride", C.c_int32),
        ("row_div", C.c_int32),
        ("n_cols", C.c_int32),
        ("plane", C.c_int32 * STE_TEXT_MAX_COLS),
    ]


class NativeError(RuntimeError):
    """A non-zero return code of the C ABI."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libste_ukf error {code}: {message}")
        self.code = code


_PROTOTYPES = {
    "ste_version": (C.c_int, []),
    "ste_last_error": (C.c_char_p, []),
    "ste_ukf_forward_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteOutputs), C.c_void_p]),
    "ste_urtss_backward_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteOutputs), C.c_void_p]),
    "ste_ukf_fused_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteOutputs)] * 2 + [C.c_void_p]),
    "ste_ukf_predict_f64": (C.c_int, [C.POINTER(SteProblem)] + [_dptr] * 9 + [C.c_void_p]),
    "ste_ukf_update_f64": (C.c_int, [C.POINTER(SteProblem)] + [_dptr] * 8 + [C.c_void_p]),
    "ste_ukf_predict_n_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_double)] + [_dptr] * 9 + [C.c_void_p]),
    "ste_ukf_update_n_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double)] + [_dptr] * 5 + [C.c_void_p]),
    "ste_urtss_backward_n_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_double)]
                                 + [_dptr] * 9 + [C.c_void_p]),
    "ste_ukf_forward_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteOutputsN), C.c_void_p]),
    "ste_urtss_backward_tracks_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteOutputsN), C.c_void_p]),
    "ste_ukf_forward_noise_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteNoiseN), C.POINTER(SteOutputsN),
                                              C.c_void_p]),
    "ste_urtss_backward_tracks_noise_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteNoiseN),
                                                        C.POINTER(SteOutputsN), C.c_void_p]),
    "ste_ukf_forward_innov_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteInnovations), C.POINTER(SteOutputs),
                                            C.c_void_p]),
    "ste_ukf_forward_innov_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteNoiseN), C.POINTER(SteInnovations),
                                              C.POINTER(SteOutputsN), C.c_void_p]),
    "ste_ukf_forward_noise_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteNoiseN), C.POINTER(SteInnovations),
                                            C.POINTER(SteOutputs), C.c_void_p]),
    "ste_urtss_backward_noise_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteNoiseN), C.POINTER(SteOutputs),
                                               C.c_void_p]),
    "ste_ukf_score_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs), C.POINTER(SteCandidates), C.POINTER(SteScores), C.c_void_p]),
    "ste_ukf_score_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN), C.POINTER(SteCandidates), C.POINTER(SteScores),
                                      C.c_void_p]),
    "ste_process_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64] + [_dptr] * 5 + [C.c_void_p]),
    "ste_csv_parse_rows": (C.c_int, [_dptr, _dptr, C.c_int64, C.POINTER(C.c_int32)] + [_dptr] * 9 + [C.c_void_p]),
    "ste_gate_terms_f64": (C.c_int, [C.POINTER(SteProblem)] + [_dptr] * 5 + [C.c_void_p]),
    "ste_sigma_points_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_double, _dptr, _dptr, _dptr, _dptr, C.c_void_p]),
    "ste_geodetic_f64": (C.c_int, [C.c_int32, C.c_int64, _dptr, _dptr, _dptr, _dptr, _dptr, C.c_void_p]),
    "ste_derive_inputs_f64": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32] + [_dptr] * 8 + [C.c_void_p]),
    "ste_track_metrics_f64": (C.c_int, [C.POINTER(SteProblem), C.POINTER(SteInputs)] + [_dptr] * 6 + [C.c_void_p]),
    "ste_track_metrics_n_f64": (C.c_int, [C.POINTER(SteProblemN), C.POINTER(SteInputsN)] + [_dptr] * 6 + [C.c_void_p]),
    "ste_text_convert_f64": (C.c_int, [C.POINTER(SteTextTable), C.c_int32, C.c_int32, _dptr, C.c_int64] + [_dptr] * 3 + [C.c_void_p]),
    "ste_text_write": (C.c_int, [C.c_int64] + [_dptr] * 4 + [C.c_int64, C.c_void_p]),
    "ste_probe_fastmath": (C.c_int, [C.c_int32, C.c_int32, _dptr, _dptr, _dptr, _dptr, C.c_void_p]),
    "ste_probe_fp64_latency": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _dptr, _dptr, C.c_void_p]),
    "ste_probe_fp64_fma": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _dptr, C.c_void_p]),
}

_lib: Optional[C.CDLL] = None


def library_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Load (once) the in-tree shared library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -m ship_track_estimators_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback for the UKF/URTSS path."
        )
    lib = C.CDLL(path)
    for name, (restype, argtypes) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.ste_version()
    if got != STE_ABI_VERSION:
        raise RuntimeError(f"libste_ukf.so ABI version {got}, binding expects {STE_ABI_VERSION}")
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != STE_OK:
        raise NativeError(code, load().ste_last_error().decode("utf-8", "replace"))


def ptr(t) -> Optional[int]:
    """Device pointer of a CUDA tensor (None passes NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("the UKF/URTSS path runs on CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("tensors passed to libste_ukf must be contiguous")
    return t.data_ptr()


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
