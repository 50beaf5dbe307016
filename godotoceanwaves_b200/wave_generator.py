"""WaveGenerator -- mirror of assets/water/wave_generator.gd on top of libocean.so.

Same public surface as the reference node: ``map_size``, ``init_gpu(num_cascades)``,
``update(delta, parameters)``, ``_process(delta)`` (one pending cascade per call, highest index
first), ``descriptors['displacement_map' | 'normal_map']`` and the two static JONSWAP helpers.
All numerics happen in the CUDA library; this class only marshals parameters."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import native
from .native import CascadeParamsC, InfoC, OceanError, check, load_library

G = 9.81        # wave_generator.gd:5
DEPTH = 20.0    # wave_generator.gd:6


class _Descriptor:
    """Stand-in for RenderingContext.Descriptor (render_context.gd:23-28): ``rid`` is the device
    pointer of the layered RGBA16F map instead of a Vulkan RID."""

    def __init__(self, rid: int, layer_bytes: int):
        self.rid = rid
        self.layer_bytes = layer_bytes


def _same_record(a, b) -> bool:
    """ctypes hands out a fresh wrapper object per array access: compare the addresses of the underlying C records."""
    return C.addressof(a) == C.addressof(b)


class WaveGenerator:
    def __init__(self, device: int = 0):
        self.map_size = 0                       # wave_generator.gd:8
        self.device = device
        self.context = None                     # :9 (the native handle once init_gpu ran)
        self.descriptors = {}                   # :11
        self.pass_parameters = []               # :14
        self._num_cascades = 0
        self._carr = None
        self._seen = None

    # ---- wave_generator.gd:17-54
    def init_gpu(self, num_cascades: int) -> None:
        lib = load_library()
        if self.context:
            self.free()
        h = C.c_void_p()
        check(lib.ocean_create(int(self.device), int(self.map_size), int(num_cascades), C.byref(h)))
        self.context = h
        self._num_cascades = int(num_cascades)
        disp, norm, layer = C.c_void_p(), C.c_void_p(), C.c_size_t()
        check(lib.ocean_get_maps(h, C.byref(disp), C.byref(norm), C.byref(layer)))
        self.descriptors = {"displacement_map": _Descriptor(disp.value, layer.value),
                            "normal_map": _Descriptor(norm.value, layer.value)}

    # ---- parameter marshalling
    def _marshal(self, parameters):
        n = len(parameters)
        if self._carr is None or len(self._carr) != n:
            self._carr = (CascadeParamsC * n)()
            self._seen = [None] * n
        seen = self._seen
        for i, p in enumerate(parameters):
            key = (id(p), p._version)
            # untouched objects are already current in the C array -- provided the library-mutated fields (time, dirty
            # flag) were last exchanged with THIS record and not with another generator's
            if seen[i] != key or (p._synced is not None and not _same_record(p._synced, self._carr[i])):
                p.to_c(self._carr[i])
                seen[i] = key
        return self._carr

    def _readback(self, parameters):
        for i, p in enumerate(parameters):
            p.from_c(self._carr[i])

    # ---- wave_generator.gd:56-63
    def _process(self, delta: float = 0.0) -> None:
        if not self.context or not self.pass_parameters:
            return
        arr = self._marshal(self.pass_parameters)
        check(load_library().ocean_process(self.context, arr, len(self.pass_parameters)))
        self._readback(self.pass_parameters)

    # ---- wave_generator.gd:90-109
    def _auto_init(self, parameters) -> None:
        """wave_generator.gd:92-93 creates the resources on the first update; a NEW generator has empty spectrum textures,
        so every cascade must regenerate (what water.gd:84-87 does when it sets the generator up)."""
        if not self.context:
            self.init_gpu(max(2, len(parameters)))
            for p in parameters:
                p.should_generate_spectrum = True

    def update(self, delta: float, parameters) -> None:
        assert len(parameters) != 0
        self._auto_init(parameters)
        arr = self._marshal(parameters)
        check(load_library().ocean_update(self.context, float(delta), arr, len(parameters)))
        self._readback(parameters)
        self.pass_parameters = parameters

    def update_all(self, delta: float, parameters) -> None:
        """update() + every pending cascade in one batched launch (the throughput path)."""
        assert len(parameters) != 0
        self._auto_init(parameters)
        arr = self._marshal(parameters)
        check(load_library().ocean_update_all(self.context, float(delta), arr, len(parameters)))
        self._readback(parameters)
        self.pass_parameters = parameters

    def update_frames(self, delta: float, parameters, frames: int) -> None:
        """`frames` consecutive update_all(delta) calls fused into a few launches (ocean_update_frames): bit-identical
        results, without the per-frame launch and host latency."""
        assert len(parameters) != 0
        self._auto_init(parameters)
        arr = self._marshal(parameters)
        check(load_library().ocean_update_frames(self.context, float(delta), arr, len(parameters), int(frames)))
        self._readback(parameters)
        self.pass_parameters = parameters

    @property
    def pass_num_cascades_remaining(self) -> int:      # wave_generator.gd:15
        return self.info().pending_cascades if self.context else 0

    # ---- wave_generator.gd:111-113
    def free(self) -> None:
        if self.context:
            check(load_library().ocean_destroy(self.context))
            self.context = None
            self.descriptors = {}

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # ---- wave_generator.gd:116-121
    @staticmethod
    def JONSWAP_alpha(wind_speed: float = 20.0, fetch_length: float = 550e3) -> float:
        return load_library().ocean_jonswap_alpha(float(wind_speed), float(fetch_length))

    @staticmethod
    def JONSWAP_peak_angular_frequency(wind_speed: float = 20.0, fetch_length: float = 550e3) -> float:
        return load_library().ocean_jonswap_peak_angular_frequency(float(wind_speed), float(fetch_length))

    # ---- host hand-off and taps
    def _require(self):
        if not self.context:
            raise OceanError("init_gpu() has not been called")

    def synchronize(self) -> None:
        self._require()
        check(load_library().ocean_synchronize(self.context))

    def info(self) -> InfoC:
        self._require()
        out = InfoC()
        check(load_library().ocean_get_info(self.context, C.byref(out)))
        return out

    def maps_to_host(self, first: int = 0, count: int | None = None):
        """(displacement, normal) as float16 arrays [count, N, N, 4] (what texture_update would upload)."""
        self._require()
        count = self._num_cascades - first if count is None else count
        N = self.map_size
        d = np.empty((count, N, N, 4), np.float16)
        n = np.empty((count, N, N, 4), np.float16)
        check(load_library().ocean_copy_maps_to_host(self.context, first, count, d.ctypes.data, n.ctypes.data))
        return d, n

    def spectrum_to_host(self, cascade: int) -> np.ndarray:
        self._require()
        N = self.map_size
        out = np.empty((N, N, 4), np.float32)
        check(load_library().ocean_copy_spectrum_to_host(self.context, cascade, out.ctypes.data))
        return out

    def set_spectrum_amplitudes(self, cascade: int, amplitudes) -> None:
        """Replaces spectrum_compute's output of one cascade by amplitudes [N][N] complex64 (or [N][N][2] float32): A(id) per
        texel; the library completes the texture with conj A(mod(-id, N)) (spectrum_compute.glsl:121-124)."""
        self._require()
        a = np.ascontiguousarray(np.asarray(amplitudes).astype(np.complex64)).view(np.float32).reshape(self.map_size, self.map_size, 2)
        check(load_library().ocean_set_spectrum_amplitudes(self.context, cascade, a.ctypes.data))

    def enable_f32_taps(self, enable: bool = True) -> None:
        self._require()
        check(load_library().ocean_enable_f32_taps(self.context, 1 if enable else 0))

    def f32_maps_to_host(self, cascade: int):
        self._require()
        N = self.map_size
        d = np.empty((N, N, 4), np.float32)
        n = np.empty((N, N, 4), np.float32)
        check(load_library().ocean_copy_f32_maps_to_host(self.context, cascade, d.ctypes.data, n.ctypes.data))
        return d, n

    def rowpass_to_host(self, cascade: int) -> np.ndarray:
        self._require()
        N = self.map_size
        out = np.empty((4, N, N, 2), np.float32)
        check(load_library().ocean_copy_rowpass_to_host(self.context, cascade, out.ctypes.data))
        return out

    # -- map queries: the water shader's sampling contract as an op (water.gdshader:27-39,42-84) ----------------
    @staticmethod
    def map_scales(parameters) -> np.ndarray:
        """map_scales[i] = (1/tile_length.x, 1/tile_length.y, displacement_scale, normal_scale), water.gd:102-110
        (the divisions are float32, as Vector2.ONE / tile_length is in Godot)."""
        out = np.empty((len(parameters), 4), np.float32)
        for i, p in enumerate(parameters):
            out[i, 0] = np.float32(1.0) / np.float32(p.tile_length[0])
            out[i, 1] = np.float32(1.0) / np.float32(p.tile_length[1])
            out[i, 2] = p.displacement_scale
            out[i, 3] = p.normal_scale
        return out

    def sample(self, points_xz, map_scales) -> tuple:
        """(displacement [n][3], gradient_foam [n][3]) float32 at world positions points_xz [n][2], summed over the
        len(map_scales) first cascades: what vertex() and fragment() of water.gdshader read at UV = VERTEX.xz."""
        self._require()
        pts = np.ascontiguousarray(points_xz, np.float32).reshape(-1, 2)
        sc = np.ascontiguousarray(map_scales, np.float32).reshape(-1, 4)
        n = pts.shape[0]
        disp = np.empty((n, 3), np.float32)
        grad = np.empty((n, 3), np.float32)
        check(load_library().ocean_sample_maps(self.context, n, pts.ctypes.data, sc.shape[0], sc.ctypes.data,
                                               disp.ctypes.data, grad.ctypes.data))
        return disp, grad

    # -- surface query: the map query above a world position, the horizontal displacement of water.gdshader:31-37 inverted --
    SURFACE_POINT = np.dtype([("height", np.float32), ("source_x", np.float32), ("source_z", np.float32), ("residual", np.float32),
                              ("gradient_foam", np.float32, 3), ("jacobian", np.float32)])      # struct ocean_surface_point

    def query_surface(self, points_xz, map_scales, iterations: int = 8) -> np.ndarray:
        """The water surface above the world positions points_xz [n][2] as SURFACE_POINT rows: height, the undisplaced
        source point whose displaced vertex lands there, the residual |source + D.xz(source) - q| in metres, the
        gradient/foam of sample() at the source point and the Jacobian determinant there (<= 0: folded surface).
        `iterations` damped Newton steps (0..32) solve source + D.xz(source) = q; see ocean_query_surface in ocean.h."""
        self._require()
        pts = np.ascontiguousarray(points_xz, np.float32).reshape(-1, 2)
        sc = np.ascontiguousarray(map_scales, np.float32).reshape(-1, 4)
        out = np.empty(pts.shape[0], self.SURFACE_POINT)
        check(load_library().ocean_query_surface(self.context, pts.shape[0], pts.ctypes.data, sc.shape[0], sc.ctypes.data, int(iterations),
                                                 out.ctypes.data))
        return out

    # -- spray candidates: the spawn test of sea_spray_particle.gdshader:80-94 as a stream compaction --------------
    SPRAY_RECORD = np.dtype([("index", np.uint32), ("start_x", np.float32), ("start_z", np.float32), ("scale_factor", np.float32),
                             ("particle_scale", np.float32, 3), ("foam", np.float32)])     # struct ocean_spray_record

    @staticmethod
    def spray_grid(num_particles: int, emission_transform=None) -> np.ndarray:
        """START_POS.xz of the emitter's particle grid (sea_spray_particle.gdshader:47,52-54), float32 [num_particles][2]."""
        out = np.empty((num_particles, 2), np.float32)
        et = None if emission_transform is None else np.ascontiguousarray(emission_transform, np.float32).reshape(12)
        check(load_library().ocean_spray_grid(num_particles, None if et is None else et.ctypes.data, out.ctypes.data))
        return out

    def extract_spray(self, points_xz, map_scales, particle_scale=(1.0, 1.0, 1.0), max_records: int | None = None):
        """The ACTIVE spray candidates among points_xz [n][2] as SPRAY_RECORD rows in candidate order, and their total
        number (which exceeds len(records) when max_records cut the output)."""
        self._require()
        pts = np.ascontiguousarray(points_xz, np.float32).reshape(-1, 2)
        sc = np.ascontiguousarray(map_scales, np.float32).reshape(-1, 4)
        ps = np.ascontiguousarray(particle_scale, np.float32).reshape(3)
        n = pts.shape[0]
        cap = n if max_records is None else int(max_records)
        recs = np.zeros(cap, self.SPRAY_RECORD)
        count = C.c_int(0)
        check(load_library().ocean_extract_spray(self.context, n, pts.ctypes.data, sc.shape[0], sc.ctypes.data, ps.ctypes.data, cap,
                                                 recs.ctypes.data, C.byref(count)))
        return recs[:min(count.value, cap)], count.value

    def twiddles_to_host(self) -> np.ndarray:
        self._require()
        out = np.empty((self.map_size - 1, 2), np.float32)
        check(load_library().ocean_copy_twiddles_to_host(self.context, out.ctypes.data))
        return out

    def get_foam_state(self, cascade: int) -> np.ndarray:
        self._require()
        out = np.empty((self.map_size, self.map_size), np.float16)
        check(load_library().ocean_get_foam_state(self.context, cascade, out.ctypes.data))
        return out

    def set_foam_state(self, cascade: int, foam: np.ndarray) -> None:
        self._require()
        foam = np.ascontiguousarray(foam, np.float16)
        assert foam.shape == (self.map_size, self.map_size)
        check(load_library().ocean_set_foam_state(self.context, cascade, foam.ctypes.data))

    def timer_start(self) -> None:
        check(load_library().ocean_timer_start(self.context))

    def timer_stop(self) -> float:
        ms = C.c_float()
        check(load_library().ocean_timer_stop(self.context, C.byref(ms)))
        return ms.value

    def set_profiling(self, enable: bool = True) -> None:
        check(load_library().ocean_set_profiling(self.context, 1 if enable else 0))

    def last_kernel_times(self):
        """(spectrum_ms, rowpass_ms, colpass_ms, chunk_cascades) of the most recent launch sequence; the two
        kernel times are those of the first L2-sized chunk of `chunk_cascades` cascades."""
        a, b, c, n = C.c_float(), C.c_float(), C.c_float(), C.c_int()
        check(load_library().ocean_get_last_kernel_times(self.context, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return a.value, b.value, c.value, n.value
