"""ctypes binding of libdpmsolver_b200.so (C-ABI: include/dpm_solver_b200.h).

The library is the product: there is no Python/PyTorch fallback. If the shared object is missing
or a symbol cannot be resolved, importing this module's `lib()` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "lib" / "libdpmsolver_b200.so"

# enums (mirror include/dpm_solver_b200.h)
DPM_F32, DPM_BF16, DPM_F16 = 0, 1, 2
FORM_NONE, FORM_LIN1, FORM_LIN2, FORM_LIN3, FORM_DIFF2, FORM_MS3, FORM_SS3T = range(7)
PARAM_NOISE, PARAM_X_START, PARAM_V, PARAM_SCORE = range(4)

PARAM_BY_NAME = {"noise": PARAM_NOISE, "x_start": PARAM_X_START, "v": PARAM_V, "score": PARAM_SCORE}


class StepDesc(C.Structure):
    """struct dpm_step_desc"""
    _fields_ = [
        ("x", C.c_void_p), ("xe", C.c_void_p), ("m0", C.c_void_p), ("m1", C.c_void_p),
        ("m2", C.c_void_p), ("m_out", C.c_void_p), ("out", C.c_void_p), ("out2", C.c_void_p),
        ("e_cond", C.c_void_p), ("e_uncond", C.c_void_p), ("thr", C.c_void_p),
        ("n", C.c_uint64), ("per_sample", C.c_uint64),
        ("state_dtype", C.c_int32), ("model_dtype", C.c_int32), ("form", C.c_int32),
        ("n_model", C.c_int32), ("param", C.c_int32), ("predict_x0", C.c_int32),
        ("c0_on_old", C.c_int32), ("raw_round", C.c_int32),
        ("guidance", C.c_float), ("alpha_e", C.c_float), ("sigma_e", C.c_float),
        ("a", C.c_float), ("c0", C.c_float), ("c1", C.c_float), ("c2", C.c_float),
        ("w0", C.c_float), ("w1", C.c_float), ("w2", C.c_float), ("w3", C.c_float),
        ("w4", C.c_float),
        ("dev_coef", C.c_void_p),
    ]


class AdaptiveCtl(C.Structure):
    """struct dpm_adaptive_ctl"""
    _fields_ = [
        ("schedule_kind", C.c_int32), ("table_len", C.c_int32),
        ("t_array", C.c_void_p), ("log_alpha_array", C.c_void_p), ("log_alpha_flipped", C.c_void_p), ("t_flipped", C.c_void_p),
        ("beta_0", C.c_float), ("beta_1_minus_beta_0", C.c_float), ("inv_total_N", C.c_float),
        ("discrete_time_input", C.c_int32), ("order", C.c_int32), ("predict_x0", C.c_int32), ("taylor", C.c_int32),
        ("t_0", C.c_float), ("theta", C.c_float), ("t_err", C.c_float),
        ("state", C.c_void_p), ("coef", C.c_void_p), ("times", C.c_void_p), ("error", C.c_void_p),
    ]


_vp, _f, _u64, _i = C.c_void_p, C.c_float, C.c_uint64, C.c_int

# name -> (restype, argtypes); every prototype of the header appears here and is checked at load
PROTOTYPES = {
    "dpm_version": (C.c_int, []),
    "dpm_last_error": (C.c_char_p, []),
    "dpm_set_tuning": (C.c_int, [_i, _i, _i]),
    "dpm_get_tuning": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "dpm_launch_count": (C.c_uint64, []),
    "dpm_step": (C.c_int, [C.POINTER(StepDesc), _vp]),
    "dpm_lincomb": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _f, _f, _f, _f, _u64, _i, _vp]),
    "dpm_solver_first_update": (C.c_int, [_vp, _vp, _vp, _f, _f, _u64, _i, _vp]),
    "dpm_multistep_second_update": (C.c_int, [_vp, _vp, _vp, _vp, _f, _f, _f, _f, _u64, _i, _vp]),
    "dpm_multistep_third_update": (C.c_int, [_vp] * 5 + [_f] * 8 + [_u64, _i, _vp]),
    "dpm_singlestep_diff_update": (C.c_int, [_vp, _vp, _vp, _vp, _f, _f, _f, _u64, _i, _vp]),
    "dpm_singlestep_third_taylor_update": (C.c_int, [_vp] * 5 + [_f] * 9 + [_u64, _i, _vp]),
    "dpm_cfg_combine": (C.c_int, [_vp, _vp, _vp, _f, _u64, _i, _vp]),
    "dpm_duplicate": (C.c_int, [_vp, _vp, _u64, _i, _vp]),
    "dpm_philox_policy": (C.c_int, [_u64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "dpm_add_noise_philox": (C.c_int, [_vp, _vp, _u64, _i, C.POINTER(C.c_float), C.POINTER(C.c_float), _u64, _u64, _i, _i, _vp]),
    "dpm_sde_step": (C.c_int, [C.POINTER(StepDesc), _f, _vp, _u64, _u64, _vp]),
    "dpm_diffedit_corrector": (C.c_int, [_vp, _vp, _vp, _vp, _u64, _u64, _f, _f, _u64, _u64, _i, _vp]),
    "dpm_data_prediction": (C.c_int, [_vp, _vp, _vp, _f, _f, _vp, _u64, _u64, _i, _vp]),
    "dpm_dynamic_threshold_workspace": (C.c_size_t, [_u64, _u64]),
    "dpm_dynamic_threshold": (C.c_int, [_vp, C.POINTER(StepDesc), _f, _f, _vp, C.c_size_t, _vp]),
    "dpm_adaptive_init": (C.c_int, [C.POINTER(AdaptiveCtl), _f, _f, _vp]),
    "dpm_adaptive_plan": (C.c_int, [C.POINTER(AdaptiveCtl), _vp]),
    "dpm_adaptive_decide": (C.c_int, [C.POINTER(AdaptiveCtl), _vp]),
    "dpm_select_copy": (C.c_int, [_vp, _vp, _vp, _u64, _vp]),
    "dpm_adaptive_error_workspace": (C.c_size_t, [_u64, _u64]),
    "dpm_adaptive_error": (C.c_int, [_vp, _vp, _vp, _vp, _f, _f, _u64, _u64, _i, _vp, C.c_size_t, _vp]),
}

_lib = None


class DpmLibraryError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("DPM_B200_LIB", LIB_PATH))
    if not path.exists():
        raise DpmLibraryError(
            f"{path} not found. Build it with `python -m dpm_solver_b200.build` "
            "(needs nvcc, sm_100a). dpm_solver_b200 has no CPU or PyTorch fallback.")
    handle = C.CDLL(str(path))
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(handle, name)
        except AttributeError as e:
            raise DpmLibraryError(f"{path} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().dpm_last_error().decode("utf-8", "replace")
        raise DpmLibraryError(f"libdpmsolver_b200 error {rc}: {msg}")
