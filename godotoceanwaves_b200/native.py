"""ctypes binding of libocean.so (include/ocean.h).  Fails loudly when the library is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("OCEAN_LIB") or os.path.join(_HERE, "libocean.so")   # OCEAN_LIB: A/B builds while tuning
_lib = None


class OceanError(RuntimeError):
    """Raised for every non-zero status returned by the C ABI (message = ocean_last_error())."""


class CascadeParamsC(C.Structure):
    """struct ocean_cascade_params (include/ocean.h) <- wave_cascade_parameters.gd:2-42"""
    _fields_ = [("tile_length", C.c_float * 2),
                ("displacement_scale", C.c_double), ("normal_scale", C.c_double),
                ("wind_speed", C.c_double), ("wind_direction", C.c_double), ("fetch_length", C.c_double),
                ("swell", C.c_double), ("spread", C.c_double), ("detail", C.c_double),
                ("whitecap", C.c_double), ("foam_amount", C.c_double),
                ("spectrum_seed", C.c_int32 * 2), ("should_generate_spectrum", C.c_int32),
                ("time", C.c_double), ("foam_grow_rate", C.c_double), ("foam_decay_rate", C.c_double)]


class SchedulerC(C.Structure):
    """struct ocean_scheduler (include/ocean.h) <- water.gd:51,62-63"""
    _fields_ = [("updates_per_second", C.c_double), ("time", C.c_double), ("next_update_time", C.c_double)]


class InfoC(C.Structure):
    _fields_ = [("device", C.c_int32), ("map_size", C.c_int32), ("num_cascades", C.c_int32),
                ("pending_cascades", C.c_int32), ("kernel_launches", C.c_uint64),
                ("cascade_updates", C.c_uint64), ("device_bytes", C.c_uint64)]


# every symbol include/ocean.h declares: name -> (restype, argtypes)
_H = C.c_void_p
_P = C.POINTER
SIGNATURES = {
    "ocean_default_cascade_params": (C.c_int, [_P(CascadeParamsC)]),
    "ocean_create": (C.c_int, [C.c_int, C.c_int, C.c_int, _P(_H)]),
    "ocean_destroy": (C.c_int, [_H]),
    "ocean_update": (C.c_int, [_H, C.c_double, _P(CascadeParamsC), C.c_int]),
    "ocean_process": (C.c_int, [_H, _P(CascadeParamsC), C.c_int]),
    "ocean_update_all": (C.c_int, [_H, C.c_double, _P(CascadeParamsC), C.c_int]),
    "ocean_update_frames": (C.c_int, [_H, C.c_double, _P(CascadeParamsC), C.c_int, C.c_int]),
    "ocean_scheduler_init": (C.c_int, [_P(SchedulerC), C.c_double]),
    "ocean_scheduler_set_rate": (C.c_int, [_P(SchedulerC), C.c_double]),
    "ocean_scheduler_tick": (C.c_int, [_P(SchedulerC), C.c_double, _P(C.c_double)]),
    "ocean_water_frame": (C.c_int, [_H, _P(SchedulerC), C.c_double, _P(CascadeParamsC), C.c_int, _P(C.c_int)]),
    "ocean_map_scales": (C.c_int, [_P(CascadeParamsC), C.c_int, C.c_void_p]),
    "ocean_water_default_time": (C.c_double, [C.c_int]),
    "ocean_get_maps": (C.c_int, [_H, _P(C.c_void_p), _P(C.c_void_p), _P(C.c_size_t)]),
    "ocean_copy_maps_to_host": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_copy_maps_to_host_async": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_snapshot_maps_to_host_async": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_wait_snapshot": (C.c_int, [_H]),
    "ocean_synchronize": (C.c_int, [_H]),
    "ocean_host_alloc": (C.c_int, [_P(C.c_void_p), C.c_size_t]),
    "ocean_host_free": (C.c_int, [C.c_void_p]),
    "ocean_copy_spectrum_to_host": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "ocean_set_spectrum_amplitudes": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "ocean_enable_f32_taps": (C.c_int, [_H, C.c_int]),
    "ocean_copy_f32_maps_to_host": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_copy_rowpass_to_host": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "ocean_copy_twiddles_to_host": (C.c_int, [_H, C.c_void_p]),
    "ocean_detmath_expf": (C.c_float, [C.c_float]),
    "ocean_debug_frame_protocol": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_debug_work_queue": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "ocean_sample_maps": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ocean_sample_maps_device": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ocean_query_surface": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ocean_query_surface_device": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ocean_spray_grid": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_extract_spray": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, _P(C.c_int)]),
    "ocean_extract_spray_device": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ocean_get_foam_state": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "ocean_set_foam_state": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "ocean_jonswap_alpha": (C.c_double, [C.c_double, C.c_double]),
    "ocean_jonswap_peak_angular_frequency": (C.c_double, [C.c_double, C.c_double]),
    "ocean_timer_start": (C.c_int, [_H]),
    "ocean_timer_stop": (C.c_int, [_H, _P(C.c_float)]),
    "ocean_set_profiling": (C.c_int, [_H, C.c_int]),
    "ocean_get_last_kernel_times": (C.c_int, [_H, _P(C.c_float), _P(C.c_float), _P(C.c_float), _P(C.c_int)]),
    "ocean_selftest_math": (C.c_int, [_H, _P(C.c_uint64), _P(C.c_uint64)]),
    "ocean_get_info": (C.c_int, [_H, _P(InfoC)]),
    "ocean_last_error": (C.c_char_p, []),
    "ocean_version": (C.c_char_p, []),
}


def native_library_path() -> str:
    return _LIB_PATH


def load_library() -> C.CDLL:
    """Loads libocean.so from the package directory.  No fallback: a missing library is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise OceanError(
                f"{_LIB_PATH} is missing: build it with `python -m godotoceanwaves_b200.build` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        lib = C.CDLL(_LIB_PATH)
        tolerant = bool(os.environ.get("OCEAN_LIB")) and os.environ.get("OCEAN_ALLOW_MISSING") == "1"   # A/B timing of OLDER builds only
        for name, (restype, argtypes) in SIGNATURES.items():
            if tolerant and not hasattr(lib, name):
                continue
            fn = getattr(lib, name)          # AttributeError if the export is missing
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def check(status: int) -> None:
    if status != 0:
        msg = load_library().ocean_last_error()
        raise OceanError(f"libocean status {status}: {msg.decode() if msg else '?'}")
