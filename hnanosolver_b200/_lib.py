"""ctypes binding of libhns_b200.so (include/hns_b200.h). No fallback: if the CUDA library is missing, importing
the compute entry points raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhns_b200.so")

c_f32p = C.POINTER(C.c_float)
c_i32p = C.POINTER(C.c_int32)
c_u64p = C.POINTER(C.c_uint64)

HNS_OK = 0
STATUS_NAMES = {0: "HNS_OK", -1: "HNS_ERR_INVALID_ARGUMENT", -2: "HNS_ERR_RUNTIME", -3: "HNS_ERR_CUDA", -4: "HNS_ERR_TOPOLOGY",
                -5: "HNS_ERR_UNSUPPORTED"}


class CombustionParams(C.Structure):
    """reference: struct CombustionParams, src/Cuda/Kernels.cuh:6-13"""
    _fields_ = [("expansionRate", C.c_float), ("temperatureRelease", C.c_float), ("buoyancyStrength", C.c_float),
                ("ambientTemp", C.c_float), ("vorticityScale", C.c_float), ("factorScale", C.c_float)]


# every symbol include/hns_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "hns_abi_version": (C.c_int, []),
    "hns_last_error": (C.c_char_p, []),
    "hns_launch_count": (C.c_uint64, []),
    "hns_launch_count_reset": (None, []),
    "hns_set_device": (C.c_int, [C.c_int]),
    "hns_set_packed_advection": (C.c_int, [C.c_int]),
    "hns_packed_advection_launches": (C.c_uint64, []),
    "hns_nvdb_write": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint64]),
    "hns_nvdb_file_grid_bytes": (C.c_int, [C.c_char_p, C.POINTER(C.c_uint64)]),
    "hns_nvdb_read": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint64]),
    "hns_nvdb_leaf_origins": (C.c_int, [C.c_void_p, C.c_uint64, c_i32p, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]),
    "hns_nvdb_grid_info": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_float),
                                     C.c_char_p]),
    "hns_nvdb_leaf_topology": (C.c_int, [C.c_void_p, C.c_uint64, c_i32p, c_u64p, C.POINTER(C.c_uint64)]),
    "hns_sidecar_from_nanovdb": (C.c_int, [C.c_void_p, C.c_uint64, c_i32p, C.c_uint64, C.c_int, C.c_void_p]),
    "hns_sidecar_nanovdb_bytes": (C.c_uint64, [c_i32p, C.c_uint64, C.c_int]),
    "hns_sidecar_to_nanovdb": (C.c_int, [c_i32p, C.c_uint64, c_u64p, C.c_void_p, C.c_int, C.c_float, C.c_char_p, C.c_void_p, C.c_uint64]),
    "hns_grid_create_from_coords": (C.c_int, [c_i32p, C.c_uint64, C.c_float, C.c_int, C.POINTER(C.c_void_p)]),
    "hns_grid_create_from_origins": (C.c_int, [c_i32p, C.c_uint64, C.c_float, C.POINTER(C.c_void_p)]),
    "hns_grid_destroy": (None, [C.c_void_p]),
    "hns_grid_num_leaves": (C.c_uint64, [C.c_void_p]),
    "hns_grid_num_voxels": (C.c_uint64, [C.c_void_p]),
    "hns_grid_voxel_size": (C.c_float, [C.c_void_p]),
    "hns_grid_nanovdb_bytes": (C.c_uint64, [C.c_void_p]),
    "hns_grid_nanovdb_device_ptr": (C.c_void_p, [C.c_void_p]),
    "hns_grid_nanovdb_download": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hns_grid_get_values": (C.c_int, [C.c_void_p, c_i32p, C.c_uint64, c_u64p]),
    "hns_grid_neighbors_download": (C.c_int, [C.c_void_p, c_i32p]),
    "hns_domain_build": (C.c_int, [c_i32p, c_u64p, C.c_uint64, C.c_int, c_i32p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "hns_domain_destroy": (None, [C.c_void_p]),
    "hns_domain_num_leaves": (C.c_uint64, [C.c_void_p]),
    "hns_domain_origins": (C.c_int, [C.c_void_p, c_i32p]),
    "hns_domain_create_grid": (C.c_int, [C.c_void_p, C.c_float, C.POINTER(C.c_void_p)]),
    "hns_release_scratch": (None, []),
    "hns_compute_sim": (C.c_int, [C.c_void_p, c_f32p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(c_f32p), C.c_int, C.c_float, C.c_float,
                                  C.POINTER(CombustionParams), C.c_int, C.c_void_p]),
    "hns_advect_index_grid": (C.c_int, [c_i32p, C.c_uint64, c_f32p, C.c_int, C.POINTER(c_f32p), C.c_float, C.c_float, C.c_void_p]),
    "hns_advect_index_grid_velocity": (C.c_int, [c_i32p, C.c_uint64, c_f32p, C.c_float, C.c_float, C.c_void_p]),
    "hns_project_non_divergent": (C.c_int, [c_i32p, C.c_uint64, c_f32p, C.c_uint64, C.c_float, C.c_void_p]),
    "hns_divergence": (C.c_int, [c_i32p, C.c_uint64, c_f32p, c_f32p, C.c_float, C.c_void_p]),
    "hns_combustion_kernel": (C.c_int, [C.c_void_p, c_f32p, C.c_uint64, C.c_float, C.c_float, C.c_void_p]),
    "hns_state_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "hns_state_destroy": (None, [C.c_void_p]),
    "hns_state_upload_velocity": (C.c_int, [C.c_void_p, c_f32p]),
    "hns_state_download_velocity": (C.c_int, [C.c_void_p, c_f32p]),
    "hns_state_upload_scalar": (C.c_int, [C.c_void_p, C.c_int, c_f32p]),
    "hns_state_download_scalar": (C.c_int, [C.c_void_p, C.c_int, c_f32p]),
    "hns_state_download_aux": (C.c_int, [C.c_void_p, C.c_int, c_f32p]),
    "hns_source_create": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "hns_source_destroy": (None, [C.c_void_p]),
    "hns_source_components": (C.c_int, [C.c_void_p]),
    "hns_source_num_leaves": (C.c_uint64, [C.c_void_p]),
    "hns_source_leaves_outside": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "hns_state_add_source_velocity": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "hns_state_add_source_scalar": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "hns_value_grid_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "hns_value_grid_destroy": (None, [C.c_void_p]),
    "hns_value_grid_bytes": (C.c_uint64, [C.c_void_p]),
    "hns_value_grid_num_leaves": (C.c_uint64, [C.c_void_p]),
    "hns_value_grid_device_ptr": (C.c_void_p, [C.c_void_p]),
    "hns_value_grid_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "hns_state_export_velocity": (C.c_int, [C.c_void_p, C.c_float, C.c_char_p, C.c_void_p, C.c_void_p]),
    "hns_state_export_scalar": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_char_p, C.c_void_p, C.c_void_p]),
    "hns_state_domain_build": (C.c_int, [C.c_void_p, C.c_float, C.c_int, C.c_int, C.POINTER(C.c_void_p), c_i32p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "hns_state_create_remapped": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "hns_state_set_combustion": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CombustionParams)]),
    "hns_state_step": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_uint, C.c_void_p]),
    "hns_state_advect_velocity": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p]),
    "hns_state_vorticity_confinement": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "hns_state_set_collision": (C.c_int, [C.c_void_p, C.c_int]),
    "hns_state_collision_active": (C.c_int, [C.c_void_p]),
    "hns_state_enforce_collision": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hns_state_vorticity_active": (C.c_int, [C.c_void_p]),
    "hns_state_vorticity_mag": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hns_state_vorticity_force": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "hns_state_divergence": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "hns_state_pressure_solve": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_uint, C.c_void_p]),
    "hns_state_subtract_gradient": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "hns_state_pressure_init": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hns_state_pressure_half_sweep": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "hns_state_combustion_buoyancy": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p]),
    "hns_omega_compute": (C.c_float, [C.c_float]),
    "hns_omega_project": (C.c_float, [C.c_float]),
    "hns_state_advect_scalars": (C.c_int, [C.c_void_p, C.c_float, C.c_int, C.c_void_p]),
    "hns_state_sync": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hns_state_time_frames": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_uint, C.c_void_p, c_f32p, c_f32p]),
    "hns_state_pack_leaves": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "hns_state_unpack_leaves": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "hns_state_field_device_ptr": (C.c_void_p, [C.c_void_p, C.c_int]),
    "hns_state_field_floats_per_leaf": (C.c_int, [C.c_int]),
    "hns_dist_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "hns_dist_create": (C.c_int, [C.POINTER(C.c_uint8), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "hns_dist_destroy": (None, [C.c_void_p]),
    "hns_dist_set_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.POINTER(c_i32p),
                                    C.POINTER(C.c_uint64), C.POINTER(c_i32p), C.c_uint64, c_i32p]),
    "hns_dist_ipc_prepare": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64)]),
    "hns_dist_ipc_connect": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_uint64, c_i32p]),
    "hns_dist_ipc_finish": (C.c_int, [C.c_void_p]),
    "hns_dist_error": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "hns_dist_reset_error": (C.c_int, [C.c_void_p]),
    "hns_dist_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p]),
    "hns_dist_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p]),
    "hns_dist_cook": (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, C.c_int, C.POINTER(c_f32p), C.c_int, C.c_float, C.c_void_p]),
    "hns_dist_frame_timed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, c_f32p]),
    "hns_dist_allreduce_sum": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int, C.c_void_p]),
    "hns_state_residual_sums": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "hns_state_divergence_sum_squares": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.c_void_p]),
    "hns_mg_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "hns_mg_destroy": (None, [C.c_void_p]),
    "hns_mg_num_levels": (C.c_int, [C.c_void_p]),
    "hns_mg_level_leaves": (C.c_uint64, [C.c_void_p, C.c_int]),
    "hns_mg_level_cells": (C.c_uint64, [C.c_void_p, C.c_int]),
    "hns_mg_set_coarsest_iterations": (C.c_int, [C.c_void_p, C.c_int]),
    "hns_state_pressure_solve_mg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "hns_mg_last_cycles": (C.c_int, [C.c_void_p]),
    "hns_mg_last_relative_residual": (C.c_double, [C.c_void_p]),
    "hns_state_set_pressure_solver": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float]),
    "hns_dist_bytes_sent": (C.c_uint64, [C.c_void_p]),
    "hns_dist_exchanges": (C.c_uint64, [C.c_void_p]),
    "hns_dist_set_pressure_solver": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_i32p, C.c_int, C.c_int, C.c_int, C.c_float,
                                               C.POINTER(C.c_uint8)]),
    "hns_dist_mg_connect": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint8)]),
    "hns_dist_mg_finish": (C.c_int, [C.c_void_p]),
    "hns_dist_mg_gathers": (C.c_uint64, [C.c_void_p]),
    "hns_dist_mg_gather_bytes": (C.c_uint64, [C.c_void_p]),
}

_lib = None


class HnsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {message}")
        self.code = code
        self.message = message


class HnsInvalidArgument(HnsError, ValueError):
    """maps the reference's std::invalid_argument"""


def lib() -> C.CDLL:
    """Loads libhns_b200.so. Raises if it has not been built -- there is no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m hnanosolver_b200.build` (nvcc, sm_100a). "
                              "hnanosolver_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.hns_abi_version() != 1:
            raise ImportError("libhns_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != HNS_OK:
        msg = lib().hns_last_error().decode(errors="replace")
        raise (HnsInvalidArgument if rc == -1 else HnsError)(rc, msg)
