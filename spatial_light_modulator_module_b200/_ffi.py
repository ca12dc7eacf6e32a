"""ctypes declarations of include/slm_holo.h and the loader of the CUDA library.

The package has exactly one compute backend: ``lib/libslmholo.so`` built for sm_100a by
``build.py``.  There is no CPU or eager fallback: if the library is missing or no CUDA device is
present, :func:`load` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libslmholo.so")

PREC_F32, PREC_F64 = 0, 1
QUANT_ROUND_WRAP, QUANT_PIL_FLOAT, QUANT_FLOOR, QUANT_PREVIEW = 1, 2, 3, 5
RF_GS, RF_GD_MAX, RF_GD_POST = 0, 1, 2          # slm_rows_fourier_pass modes
CLOSE_MAX, CLOSE_GS, CLOSE_GD = 0, 1, 2         # slm_rows_close kinds

_vp, _i, _d, _ll = C.c_void_p, C.c_int, C.c_double, C.c_longlong
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)

# name -> (restype, argtypes); mirrors include/slm_holo.h one to one
SIGNATURES = {
    "slm_last_error": (C.c_char_p, []),
    "slm_version": (_i, []),
    "slm_supported_lengths": (_i, [_ip, _i]),
    "slm_ctx_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _vp]),
    "slm_ctx_destroy": (None, [_vp]),
    "slm_ctx_workspace_bytes": (C.c_size_t, [_vp]),
    "slm_ctx_launch_count": (_ll, [_vp]),
    "slm_ctx_profile": (_i, [_vp, _i]),
    "slm_ctx_profile_read": (_i, [_vp, _dp, C.POINTER(_ll)]),
    "slm_fft2": (_i, [_vp, _i, _vp, _vp, _i]),
    "slm_gs_run": (_i, [_vp, _i, _vp, _vp, _vp, _dp, _dp, _vp, _vp, _i, _i, _d, _vp, _vp]),
    "slm_gsw_run": (_i, [_vp, _i, _vp, _vp, _vp, _dp, _dp, _vp, _vp, _i, _i, _d, _vp, _vp, _dp, _vp, _d]),
    "slm_gs_multiplane_run": (_i, [_vp, _i, _i, _vp, _vp, _vp, _dp, _dp, _dp, _vp, _vp, _i, _i, _d, _vp, _vp]),
    "slm_gd_run": (_i, [_vp, _i, _vp, _vp, _vp, _dp, _dp, _vp, _vp, _dp, _i, _d, _vp, _vp]),
    "slm_fourier_guess": (_i, [_vp, _i, _vp, _vp, _dp, _vp, _i, _vp]),
    "slm_gd_multiplane_run": (_i, [_vp, _i, _i, _vp, _vp, _vp, _dp, _dp, _dp, _vp, _vp, _dp, _i, _d, _vp, _vp]),
    "slm_multiplane_fourier_guess": (_i, [_vp, _i, _i, _vp, _vp, _dp, _dp, _vp, _i, _vp]),
    "slm_random_phasor": (_i, [_vp, _vp, _vp, _ll, _d]),
    "slm_mt19937_uniform": (_i, [_vp, _vp, _i, _vp, _ll, _vp]),
    "slm_phase_phasor": (_i, [_vp, _vp, _vp, _vp, _ll, _ll]),
    "slm_single_trap_phase": (_i, [_vp, _i, _i, _i, _i, _vp]),
    "slm_trap_frames": (_i, [_vp, _vp, _i, _i, _i, _vp, _i]),
    "slm_rows_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _vp]),
    "slm_rows_fft": (_i, [_vp, _vp, _vp, _dp, _vp, _i, _i, _i]),
    "slm_rows_gs_row_pass": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp]),
    "slm_rows_fourier_pass": (_i, [_vp, _i, _vp, _vp, _i, _vp, _dp, _d, _vp, _vp]),
    "slm_rows_reduce": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i]),
    "slm_rows_close": (_i, [_vp, _vp, _i, _d, _d, _i, _d, _vp]),
    "slm_rows_state": (_i, [_vp, _dp, _dp, _ip, _ip]),
    "slm_rows_reset": (_i, [_vp]),
    "slm_rows_gd_row_pass": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "slm_transpose_blocks": (_i, [_vp, _vp, _vp, _i, _i, _i, _i]),
    "slm_transpose_blocks_peer": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i]),
    "slm_read_curves": (_i, [_vp, _i, _i, _dp, _ip]),
    "slm_expected_outcome": (_i, [_vp, _i, _vp, _dp, _vp]),
    "slm_deflect_phase": (_i, [_vp, _i, _i, _d, _d, _d, _vp]),
    "slm_lens_phase": (_i, [_vp, _i, _i, _d, _d, _d, _i, _vp]),
    "slm_add_mod2pi": (_i, [_vp, _vp, _vp, _vp, _ll, _ll]),
    "slm_quantize": (_i, [_vp, _vp, _vp, _d, _i, _vp, _ll, _ll]),
    "slm_quantize_grey": (_i, [_vp, _vp, _vp, _d, _vp, _ll, _ll]),
    "slm_host_register": (_i, [_vp, C.c_size_t]),
    "slm_host_unregister": (_i, [_vp]),
}


def declare(lib: C.CDLL) -> C.CDLL:
    """Attach restype/argtypes for every symbol of include/slm_holo.h (raises if one is missing)."""
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


class EngineError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """The CUDA library, loaded once.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        path = os.environ.get("SLM_HOLO_LIB", LIB_PATH)      # another BUILD of the same CUDA library (tuning variants)
        if path != LIB_PATH:
            _lib = declare(C.CDLL(path))
            return _lib
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                f"{LIB_PATH} is missing: build it with `python -m spatial_light_modulator_module_b200.build` "
                "(nvcc, sm_100a).  This package has no CPU fallback.")
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(lib: C.CDLL, rc: int) -> None:
    if rc != 0:
        raise EngineError(f"libslmholo error {rc}: {lib.slm_last_error().decode()}")
