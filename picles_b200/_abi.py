"""ctypes mirror of include/picles_b200.h (the C ABI of libpicles_b200.so).

The shared library is the product; this module only binds it.  There is no CPU
fallback: `load_library()` raises if the CUDA library has not been built, and every
compute entry point of the library itself fails when no sm_100-class GPU is usable.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PICLES_B200_LIB", os.path.join(HERE, "libpicles_b200.so"))

ABI_VERSION = 3

# enums (include/picles_b200.h)
BND_NONPERIODIC, BND_PERIODIC, BND_TRIPOLAR_NORTH = 0, 1, 2
MASK_LAND, MASK_OCEAN, MASK_LAND_BOUNDARY, MASK_GRID_BOUNDARY = 0, 1, 2, 3
SOLVER_TSIT5, SOLVER_DP5, SOLVER_AUTOTSIT5 = 0, 1, 2
PST_OK, PST_MAXITERS, PST_DTMIN, PST_UNSTABLE = 0, 1, 2, 4
PST_NAN_RESET, PST_INF_RESET, PST_EMAX_CLAMP = 8, 16, 32
PF_ON, PF_BOUNDARY, PF_DT_RESET, PF_ACTIVE = 1, 2, 4, 8

OPT_ACCUMULATE_STATE = 1

ERR_NAMES = {0: "OK", -1: "ERR_ARG", -2: "ERR_CUDA", -3: "ERR_ALLOC", -4: "ERR_HALO", -5: "ERR_STATE", -6: "ERR_COMM"}


class PiclesParams(C.Structure):
    """picles_params_t — field order and types must match the header exactly."""

    _fields_ = [
        ("r_g", C.c_double),
        ("C_alpha", C.c_double),
        ("C_varphi", C.c_double),
        ("C_e", C.c_double),
        ("g", C.c_double),
        ("p", C.c_double),
        ("q", C.c_double),
        ("n", C.c_double),
        ("e_T", C.c_double),
        ("propagation", C.c_int32),
        ("input", C.c_int32),
        ("dissipation", C.c_int32),
        ("peak_shift", C.c_int32),
        ("direction", C.c_int32),
        ("solver", C.c_int32),
        ("abstol", C.c_double),
        ("reltol", C.c_double),
        ("dt", C.c_double),
        ("dtmin", C.c_double),
        ("dtmax", C.c_double),
        ("force_dtmin", C.c_int32),
        ("adaptive", C.c_int32),
        ("maxiters", C.c_int64),
        ("log_energy_minimum", C.c_double),
        ("log_energy_maximum", C.c_double),
        ("wind_min_squared", C.c_double),
        ("seed_timescale", C.c_double),
        ("minimal_state", C.c_double * 2),
        ("has_defaults", C.c_int32),
        ("defaults", C.c_double * 5),
        ("periodic_boundary", C.c_int32),
        ("on_persist", C.c_int32),
        ("nan_eest_rejects", C.c_int32),
    ]


class PiclesCounters(C.Structure):
    """picles_counters_t"""

    _fields_ = [
        ("n_active", C.c_int64),
        ("n_integrated", C.c_int64),
        ("n_substeps", C.c_int64),
        ("n_rejects", C.c_int64),
        ("n_rhs", C.c_int64),
        ("n_reseed_advance", C.c_int64),
        ("n_fixups", C.c_int64),
        ("n_failed", C.c_int64),
        ("n_deposited", C.c_int64),
        ("n_remesh_A", C.c_int64),
        ("n_remesh_B", C.c_int64),
        ("n_remesh_C", C.c_int64),
        ("n_remesh_D", C.c_int64),
        ("reach", C.c_int32),
        ("max_attempts", C.c_int32),
        ("ms_advance", C.c_double),
        ("ms_project", C.c_double),
        ("ms_remesh", C.c_double),
        ("n_stiff_switches", C.c_int64),
        ("n_stiff_attempts", C.c_int64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# every symbol include/picles_b200.h declares: (restype, argtypes)
_vp = C.c_void_p
_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)
SYMBOLS = {
    "picles_abi_version": (C.c_int, []),
    "picles_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "picles_destroy": (C.c_int, [_vp]),
    "picles_last_error": (C.c_char_p, [_vp]),
    "picles_set_grid": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  _vp, _vp, _vp, _vp]),
    "picles_set_grid_metric": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         _vp, _vp, _vp, _vp, _vp, C.c_double]),
    "picles_get_metric": (C.c_int, [_vp, _vp, _vp]),
    "picles_make_boundaries": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    "picles_set_params": (C.c_int, [_vp, C.POINTER(PiclesParams)]),
    "picles_set_members": (C.c_int, [_vp, C.c_int]),
    "picles_member_energy_sums": (C.c_int, [_vp, _vp]),
    "picles_seed": (C.c_int, [_vp, _vp, _vp]),
    "picles_get_row_reach": (C.c_int, [_vp, _vp]),
    "picles_halo_rows": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "picles_halo_widen": (C.c_int, [_vp, C.c_int]),
    "picles_set_global_reach": (C.c_int, [_vp, C.c_int]),
    "picles_get_attempt_histogram": (C.c_int, [_vp, _vp, C.c_int]),
    "picles_launch_count": (C.c_int64, []),
    "picles_step": (C.c_int, [_vp, C.c_double, C.c_double, _vp, _vp, _vp, _vp]),
    "picles_upload_winds": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "picles_set_wind_midlevels": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "picles_step_advance": (C.c_int, [_vp, C.c_double, C.c_double]),
    "picles_halo_buffers": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                      C.POINTER(C.c_int64)]),
    "picles_halo_pack": (C.c_int, [_vp]),
    "picles_halo_unpack": (C.c_int, [_vp]),
    "picles_step_project_remesh": (C.c_int, [_vp, C.c_double, C.c_double]),
    "picles_synchronize": (C.c_int, [_vp]),
    "picles_get_reach": (C.c_int, [_vp, _i32p]),
    "picles_comm_unique_id": (C.c_int, [C.c_char_p, C.c_char_p]),
    "picles_comm_init": (C.c_int, [_vp, C.c_char_p, C.c_int, C.c_int, C.c_char_p]),
    "picles_comm_destroy": (C.c_int, [_vp]),
    "picles_halo_exchange": (C.c_int, [_vp, C.c_int, C.c_int]),
    "picles_step_strip": (C.c_int, [_vp, C.c_double, C.c_double, _vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "picles_set_wind_mesh": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "picles_set_member_wind_meshes": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "picles_sample_wind_mesh": (C.c_int, [_vp, C.c_double, _vp, _vp]),
    "picles_seed_wind_mesh": (C.c_int, [_vp, C.c_double]),
    "picles_step_wind_mesh": (C.c_int, [_vp, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int]),
    "picles_stage_wind_mesh": (C.c_int, [_vp, C.c_double, C.c_double, C.c_int]),
    "picles_get_state": (C.c_int, [_vp, _vp]),
    "picles_set_state": (C.c_int, [_vp, _vp]),
    "picles_checkpoint_size": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "picles_checkpoint_save": (C.c_int, [_vp, _vp, C.c_int64]),
    "picles_checkpoint_load": (C.c_int, [_vp, _vp, C.c_int64]),
    "picles_get_fields": (C.c_int, [_vp, _vp, _vp, _vp]),
    "picles_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_int64]),
    "picles_host_free": (C.c_int, [_vp]),
    "picles_snapshot_begin": (C.c_int, [_vp, _vp]),
    "picles_snapshot_wait": (C.c_int, [_vp]),
    "picles_get_particles": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "picles_get_counters": (C.c_int, [_vp, C.POINTER(PiclesCounters)]),
    "picles_get_solver_state": (C.c_int, [_vp, _vp]),
    "picles_state_energy_sum": (C.c_int, [_vp, _dp]),
    "picles_state_dev": (C.c_int, [_vp, C.POINTER(_vp)]),
    "picles_wind_dev": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "picles_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "picles_zero_state": (C.c_int, [_vp]),
    "picles_copy_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64]),
    "picles_timer_start": (C.c_int, [_vp]),
    "picles_timer_stop": (C.c_int, [_vp, _dp]),
    "picles_selftest_math": (C.c_int, [_vp, C.c_uint64, C.c_int, C.POINTER(C.c_int64)]),
    "picles_measure_fp64_peak": (C.c_int, [_vp, _dp]),
    "picles_measure_hbm_copy": (C.c_int, [_vp, C.c_int, _dp]),
    "picles_measure_wind_sample": (C.c_int, [_vp, C.c_double, C.c_int, _dp]),
    # the one-dimensional model (WaveGrowth1D)
    "picles1d_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "picles1d_destroy": (C.c_int, [_vp]),
    "picles1d_last_error": (C.c_char_p, [_vp]),
    "picles1d_set_grid": (C.c_int, [_vp, C.c_int, C.c_double, C.c_double, _vp]),
    "picles1d_set_params": (C.c_int, [_vp, C.POINTER(PiclesParams)]),
    "picles1d_seed": (C.c_int, [_vp, _vp]),
    "picles1d_step": (C.c_int, [_vp, C.c_double, C.c_double, _vp, _vp]),
    "picles1d_get_state": (C.c_int, [_vp, _vp]),
    "picles1d_get_particles": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "picles1d_get_counters": (C.c_int, [_vp, C.POINTER(PiclesCounters)]),
}

_lib = None


class PiclesError(RuntimeError):
    pass


def load_library(path: str | None = None):
    """dlopen libpicles_b200.so and bind every declared symbol.  Raises (never falls
    back) when the library is missing or a symbol is absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise PiclesError(
            f"{p} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()'). "
            "There is no CPU fallback for this path."
        )
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.picles_abi_version() != ABI_VERSION:
        raise PiclesError("libpicles_b200.so ABI version mismatch")
    if path is None:
        _lib = lib
    return lib
