"""ctypes binding of include/luw_cuda.h -- the same C ABI the C++ host layer (host/lbm.hpp) links against.

There is no CPU fallback: if the shared library has not been built, importing this module raises; if no CUDA device is present,
every compute entry point returns LUW_ERR_NO_DEVICE and `check()` raises LuwError.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LUW_CUDA_LIB") or os.path.join(HERE, "lib", "libluw_cuda.so")  # override: development builds only

OK, ERR_INVALID, ERR_NO_DEVICE, ERR_OOM, ERR_CUDA = 0, 1, 2, 3, 4
FP32, FP16S, FP16C = 0, 1, 2
UPDATE_FIELDS, VOLUME_FORCE, EQUILIBRIUM_BOUNDARIES, SUBGRID, BUFFER_NUDGING, TOP_SPONGE = 1, 2, 4, 8, 16, 32
TEMPERATURE = 64
ARITH_STRICT, ARITH_FAST = 0, 1
FIELD_RHO, FIELD_U, FIELD_FLAGS, FIELD_FI, FIELD_T, FIELD_GI = 0, 1, 2, 3, 4, 5
HALO_FI, HALO_RHO_U_FLAGS, HALO_GI, HALO_T = 0, 1, 2, 3


class LuwError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"luw_cuda error {code}: {message}")
        self.code = code


class DeviceInfo(C.Structure):
    _fields_ = [("name", C.c_char * 256), ("memory_bytes", C.c_uint64), ("compute_units", C.c_uint32), ("clock_mhz", C.c_uint32),
                ("cc_major", C.c_uint32), ("cc_minor", C.c_uint32)]


class DomainParams(C.Structure):
    _fields_ = [("Nx", C.c_uint32), ("Ny", C.c_uint32), ("Nz", C.c_uint32), ("Dx", C.c_uint32), ("Dy", C.c_uint32), ("Dz", C.c_uint32),
                ("Ox", C.c_int32), ("Oy", C.c_int32), ("Oz", C.c_int32), ("precision", C.c_uint32), ("features", C.c_uint32),
                ("arith", C.c_uint32), ("w", C.c_float), ("downstream_face", C.c_int32), ("buffer_N", C.c_uint32),
                ("buffer_inv_tau", C.c_float), ("buffer_nudge_vertical", C.c_int32), ("sponge_N", C.c_uint32),
                ("sponge_inv_tau", C.c_float), ("device", C.c_int32)]


EXPORTS = {  # name -> argtypes; every symbol include/luw_cuda.h declares
    "luw_device_count": [C.POINTER(C.c_int)],
    "luw_get_device_info": [C.c_int, C.POINTER(DeviceInfo)],
    "luw_domain_create": [C.POINTER(DomainParams), C.POINTER(C.c_void_p)],
    "luw_domain_destroy": [C.c_void_p],
    "luw_domain_set_stream": [C.c_void_p, C.c_void_p],
    "luw_domain_bytes": [C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_domain_step_kernel": [C.c_void_p, C.POINTER(C.c_int)],
    "luw_upload": [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64],
    "luw_download": [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64],
    "luw_device_ptr": [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)],
    "luw_thermal_params": [C.c_void_p, C.c_float, C.c_float, C.c_float],
    "luw_initialize": [C.c_void_p],
    "luw_stream_collide": [C.c_void_p, C.c_uint64] + [C.c_float] * 6,
    "luw_update_fields": [C.c_void_p, C.c_uint64] + [C.c_float] * 6,
    "luw_run_steps": [C.c_void_p, C.c_uint64, C.c_uint64] + [C.c_float] * 6,
    "luw_halo_bytes": [C.c_void_p, C.c_int, C.c_uint32, C.POINTER(C.c_uint64)],
    "luw_halo_extract": [C.c_void_p, C.c_int, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p],
    "luw_halo_insert": [C.c_void_p, C.c_int, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p],
    "luw_halo_exchange": [C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.c_uint64],
    "luw_halo_ipc_export": [C.c_void_p, C.c_uint32, C.c_void_p],
    "luw_halo_ipc_connect": [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p],
    "luw_halo_ipc_exchange": [C.c_void_p, C.c_int, C.c_uint32, C.c_uint64],
    "luw_step_halo_ipc": [C.c_void_p, C.c_uint64] + [C.c_float] * 6,
    "luw_overlapped_steps": [C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_run_steps_multi": [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64] + [C.c_float] * 6,
    "luw_vk_inlet_create": [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)],
    "luw_vk_inlet_apply": [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float],
    "luw_vk_inlet_destroy": [C.c_void_p],
    "luw_voxelize_mesh": [C.c_void_p, C.c_uint32, C.c_uint8, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p],
    "luw_inlet_nearest": [C.c_int, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p],
    "luw_inlet_knn": [C.c_int, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p],
    "luw_inlet_launch_count": [C.POINTER(C.c_uint64)],
    "luw_cellset_create": [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)],
    "luw_cellset_upload": [C.c_void_p, C.c_int, C.c_void_p],
    "luw_cellset_download": [C.c_void_p, C.c_int, C.c_void_p],
    "luw_cellset_destroy": [C.c_void_p],
    "luw_stats_create": [C.c_void_p, C.POINTER(C.c_void_p)],
    "luw_stats_accumulate": [C.c_void_p],
    "luw_stats_reset": [C.c_void_p],
    "luw_stats_download": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_stats_download_temperature": [C.c_void_p, C.c_void_p],
    "luw_stats_destroy": [C.c_void_p],
    "luw_column_ground": [C.c_void_p, C.c_void_p],
    "luw_wind_stats_create": [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)],
    "luw_wind_stats_accumulate": [C.c_void_p],
    "luw_wind_stats_reset": [C.c_void_p],
    "luw_wind_stats_download": [C.c_void_p] + [C.c_void_p] * 6 + [C.POINTER(C.c_uint64)],
    "luw_wind_stats_destroy": [C.c_void_p],
    "luw_solid_surface": [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_wall_loads_create": [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)],
    "luw_wall_loads_accumulate": [C.c_void_p, C.c_uint64],
    "luw_wall_loads_drain": [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_wall_loads_download_cells": [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_wall_loads_reset": [C.c_void_p],
    "luw_wall_loads_destroy": [C.c_void_p],
    "luw_probes_create": [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)],
    "luw_probes_sample": [C.c_void_p, C.c_uint64] + [C.c_float] * 6,
    "luw_probes_drain": [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_probes_reset": [C.c_void_p],
    "luw_probes_destroy": [C.c_void_p],
    "luw_particles_create": [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)],
    "luw_particles_emit": [C.c_void_p, C.c_uint64, C.c_uint32],
    "luw_particles_advance": [C.c_void_p, C.c_uint64] + [C.c_float] * 7 + [C.c_double],
    "luw_particles_count": [C.c_void_p],
    "luw_particles_download": [C.c_void_p] * 5,
    "luw_particles_download_bins": [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)],
    "luw_particles_reset_bins": [C.c_void_p],
    "luw_particles_destroy": [C.c_void_p],
    "luw_host_alloc": [C.POINTER(C.c_void_p), C.c_uint64],
    "luw_host_free": [C.c_void_p],
    "luw_sync": [C.c_void_p],
    "luw_timer_begin": [C.c_void_p],
    "luw_timer_end": [C.c_void_p, C.POINTER(C.c_float)],
    "luw_kernel_timing": [C.c_void_p, C.c_int],
    "luw_kernel_timing_read": [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint64)],
    "luw_launch_count": [C.c_void_p, C.POINTER(C.c_uint64)],
}

_lib = None


def lib():
    """Load libluw_cuda.so (built by `make -C latticeurbanwind_b200/csrc` or __graft_entry__.build()). Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with __graft_entry__.build(); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, argtypes in EXPORTS.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        L.luw_last_error_string.restype = C.c_char_p
        L.luw_last_error_string.argtypes = []
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise LuwError(rc, lib().luw_last_error_string().decode(errors="replace"))


def device_count():
    n = C.c_int(0)
    rc = lib().luw_device_count(C.byref(n))
    return n.value if rc == OK else 0


def device_info(device=0):
    info = DeviceInfo()
    check(lib().luw_get_device_info(device, C.byref(info)))
    return info
