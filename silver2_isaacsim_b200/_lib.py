"""ctypes binding of ``libh2o_b200.so`` (the C ABI declared in ``include/h2o.h``).

There is no CPU implementation behind this package: if the CUDA library has not
been built (``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C silver2_isaacsim_b200/csrc``) importing the engine fails loudly.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# H2O_LIB_PATH: tuning experiments load a variant build (csrc/Makefile TAG=...); the product is the default path
LIB_PATH = os.environ.get("H2O_LIB_PATH") or os.path.join(_HERE, "lib", "libh2o_b200.so")

# h2o_status (include/h2o.h)
H2O_OK = 0
STATUS_NAMES = {
    0: "H2O_OK", 1: "H2O_ERR_BAD_HANDLE", 2: "H2O_ERR_BAD_ARGUMENT", 3: "H2O_ERR_BAD_SHAPE",
    4: "H2O_ERR_BAD_DTYPE", 5: "H2O_ERR_BAD_DEVICE", 6: "H2O_ERR_NOT_CONTIGUOUS",
    7: "H2O_ERR_ALIGNMENT", 8: "H2O_ERR_NOT_CONFIGURED", 9: "H2O_ERR_CUDA", 10: "H2O_ERR_NO_DEVICE",
}
H2O_F32, H2O_F64 = 0, 1
H2O_QUAT_XYZW, H2O_QUAT_WXYZ = 0, 1
H2O_KERNEL_AUTO, H2O_KERNEL_TILE, H2O_KERNEL_DIRECT = 0, 1, 2
LAYOUT_SPLIT, LAYOUT_PHYSX, LAYOUT_VIEW = 0, 1, 2
N_COEFF = 11
N_STATS = 8
STATS_FIELDS = ("sum_force_norm", "max_force_norm", "wet_bodies", "clamped_bodies",
                "nonfinite_bodies", "still_wet_bodies", "bodies", "reevaluated_bodies")


class H2OError(RuntimeError):
    """A C-ABI call returned a non-zero ``h2o_status``."""

    def __init__(self, status: int, message: str):
        self.status = status
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")


# every exported symbol of include/h2o.h + include/h2o_dlpack.h: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    "h2o_last_error": (c_char_p, []),
    "h2o_version": (c_char_p, []),
    "h2o_device_count": (c_int, []),
    "h2o_create": (c_int, [POINTER(c_void_p), c_int64, c_int, c_int]),
    "h2o_destroy": (c_int, [_P]),
    "h2o_set_globals": (c_int, [_P, c_double, c_double]),
    "h2o_set_environment": (c_int, [_P, POINTER(c_double), c_double]),
    "h2o_set_surface_heights": (c_int, [_P, _P]),
    "h2o_set_wave_field": (c_int, [_P, c_int, POINTER(c_double), c_double]),
    "h2o_wave_time_write": (c_int, [_P, c_double, _P]),
    "h2o_wave_time_read": (c_int, [_P, POINTER(c_double), _P]),
    "h2o_wave_sample": (c_int, [_P, _P, c_int64, _P, _P]),
    "h2o_set_wave_slope": (c_int, [_P, c_int]),
    "h2o_set_fluid_inertia": (c_int, [_P, c_int]),
    "h2o_set_env_conditions": (c_int, [_P, c_int64, _P]),
    "h2o_reset_envs": (c_int, [_P, _P, c_int, _P]),
    "h2o_wave_sample_env": (c_int, [_P, _P, _P, c_int64, _P, _P]),
    "h2o_set_current_grid": (c_int, [_P, _P, POINTER(c_int64), POINTER(c_double)]),
    "h2o_water_sample": (c_int, [_P, _P, _P, c_int64, _P, _P]),
    "h2o_water_slope_sample": (c_int, [_P, _P, _P, c_int64, _P, _P]),
    "h2o_fluid_accel_sample": (c_int, [_P, _P, _P, c_int64, _P, _P]),
    "h2o_set_added_mass_dense": (c_int, [_P, c_int, POINTER(c_double), c_int, POINTER(c_int32)]),
    "h2o_set_params_uniform": (c_int, [_P, POINTER(c_double), c_double]),
    "h2o_set_part_table": (c_int, [_P, c_int, POINTER(c_double), c_int, POINTER(c_int32)]),
    "h2o_set_params_per_body": (c_int, [_P, _P, c_int, _P]),
    "h2o_set_params_soa": (c_int, [_P, POINTER(c_void_p), c_int, _P]),
    "h2o_set_articulation": (c_int, [_P, c_int]),
    "h2o_set_articulation_offsets": (c_int, [_P, c_int64, POINTER(c_int64)]),
    "h2o_set_quat_order": (c_int, [_P, c_int]),
    "h2o_set_kernel": (c_int, [_P, c_int]),
    "h2o_set_tile_config": (c_int, [_P, c_int]),
    "h2o_set_warp_compat": (c_int, [_P, c_int]),
    "h2o_set_strict": (c_int, [_P, c_int]),
    "h2o_enable_stats": (c_int, [_P, c_int]),
    "h2o_reset": (c_int, [_P, _P]),
    "h2o_set_prev": (c_int, [_P, _P, _P, _P]),
    "h2o_get_prev": (c_int, [_P, _P, _P, _P]),
    "h2o_step": (c_int, [_P, _P, _P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_step_physx": (c_int, [_P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_step_view": (c_int, [_P, _P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_bind": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P]),
    "h2o_unbind": (c_int, [_P]),
    "h2o_step_bound": (c_int, [_P, c_double, _P]),
    "h2o_capture_rollout": (c_int, [_P, c_int, c_double, _P]),
    "h2o_rollout_persistent": (c_int, [_P, c_int, c_double, c_double, c_int, _P, _P]),
    "h2o_launch_rollout": (c_int, [_P, _P]),
    "h2o_set_rollout_mode": (c_int, [_P, c_int, c_double]),
    "h2o_integrate_free_bodies": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_double, c_double, _P]),
    "h2o_components": (c_int, [_P, _P, _P, _P, _P, _P, _P, POINTER(c_void_p), _P, _P, _P]),
    "h2o_step_host": (c_int, [_P, _P, _P, _P, _P, c_double, _P, _P, _P]),
    "h2o_step_host_physx": (c_int, [_P, _P, _P, c_double, _P, _P, _P]),
    "h2o_last_host_path": (c_int, [_P]),
    "h2o_stats_device_ptr": (c_int, [_P, POINTER(c_void_p)]),
    "h2o_read_stats": (c_int, [_P, POINTER(c_double), c_int, _P]),
    "h2o_launch_count": (c_int64, [_P]),
    "h2o_n_bodies": (c_int64, [_P]),
    "h2o_dtype_of": (c_int, [_P]),
    "h2o_last_kernel": (c_int, [_P]),
    "h2o_last_ctas_per_sm": (c_int, [_P]),
    "h2o_prev_device_ptr": (c_int, [_P, POINTER(c_void_p)]),
    "h2o_coeff_device_ptr": (c_int, [_P, POINTER(c_void_p), POINTER(c_int64)]),
    # include/h2o_dlpack.h
    "h2o_step_dl": (c_int, [_P, _P, _P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_step_physx_dl": (c_int, [_P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_step_view_dl": (c_int, [_P, _P, _P, _P, c_double, _P, _P, _P, _P]),
    "h2o_bind_dl": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P]),
    "h2o_components_dl": (c_int, [_P, _P, _P, _P, _P, _P, _P, POINTER(c_void_p), _P, _P, _P]),
    "h2o_set_params_per_body_dl": (c_int, [_P, _P, _P]),
    "h2o_set_prev_dl": (c_int, [_P, _P, _P, _P]),
    "h2o_export_prev_dl": (c_int, [_P, POINTER(c_void_p)]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the CUDA library; raises ImportError (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the sm_100a CUDA library has not been built. "
            "Run `python -c \"import __graft_entry__ as g; g.build()\"` at the repo root "
            "(or `make -C silver2_isaacsim_b200/csrc`). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != H2O_OK:
        msg = load().h2o_last_error()
        raise H2OError(status, msg.decode() if msg else "")


# DLPack capsule -> DLManagedTensor* (whose first member is the DLTensor)
_pyapi = ctypes.pythonapi
_pyapi.PyCapsule_GetPointer.restype = c_void_p
_pyapi.PyCapsule_GetPointer.argtypes = [ctypes.py_object, c_char_p]
_pyapi.PyCapsule_New.restype = ctypes.py_object
_pyapi.PyCapsule_New.argtypes = [c_void_p, c_char_p, c_void_p]


def capsule_pointer(capsule) -> int:
    return _pyapi.PyCapsule_GetPointer(capsule, b"dltensor")


def capsule_from_managed(ptr: int):
    """Wrap a DLManagedTensor* produced by the library into a 'dltensor' capsule."""
    return _pyapi.PyCapsule_New(ptr, b"dltensor", None)
