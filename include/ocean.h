/*
 * include/ocean.h -- C ABI of libocean.so, the B200-native drop-in for the wave-generation
 * hot path of 2Retr0/GodotOceanWaves (spectrum -> time propagation -> 4 packed N x N inverse
 * FFTs -> displacement / normal / Jacobian-foam maps).
 *
 * Each entry point names the reference interface it replaces (paths relative to the
 * reference repository).  Everything is plain C: opaque handle, POD structs, raw pointers
 * and sizes.  Every function returns an int status (OCEAN_OK == 0) and never throws or
 * aborts; ocean_last_error() returns a thread-local description of the last failure.
 *
 * Threading: a generator is NOT thread-safe (the reference runs on Godot's main thread,
 * assets/water/wave_generator.gd:19).  All GPU work of a generator is issued on its own
 * CUDA stream; calls are asynchronous w.r.t. the GPU until ocean_synchronize() or a
 * *_to_host call without the _async suffix.
 *
 * Ownership: the library owns all device memory (cf. RenderingContext's DeletionQueue,
 * assets/render_context.gd:4-21,40-46); callers borrow device pointers that stay valid until
 * ocean_destroy().  Changing map_size or the cascade count = destroy + create, as in
 * assets/water/water.gd:22-41,84-91.
 */
#ifndef OCEAN_H
#define OCEAN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCEAN_OK 0
#define OCEAN_ERR_INVALID_ARGUMENT 1
#define OCEAN_ERR_CUDA 2
#define OCEAN_ERR_UNSUPPORTED 3
#define OCEAN_ERR_STATE 4

#define OCEAN_MAX_MAP_SIZE 1024 /* assets/shaders/compute/fft_compute.glsl:9 */
#define OCEAN_MIN_MAP_SIZE 128  /* assets/water/water.gd:38, wave_generator.gd:46 */

typedef struct ocean_generator ocean_generator; /* replaces the WaveGenerator node, wave_generator.gd:2 */

/* POD mirror of the WaveCascadeParameters resource, assets/water/wave_cascade_parameters.gd:2-42.
 * GDScript floats are binary64; Vector2 components are binary32.  The library rounds to
 * binary32 exactly where RenderingContext.create_push_constant does (render_context.gd:122-135). */
typedef struct ocean_cascade_params {
    float tile_length[2];             /* :7   metres */
    double displacement_scale;        /* :9   render-side only (map_scales, water.gd:102-110) */
    double normal_scale;              /* :11  render-side only */
    double wind_speed;                /* :15  m/s, clamped >= 1e-4 by the setter */
    double wind_direction;            /* :17  degrees */
    double fetch_length;              /* :20  kilometres, clamped >= 1e-4 */
    double swell;                     /* :22 */
    double spread;                    /* :25 */
    double detail;                    /* :28 */
    double whitecap;                  /* :32 */
    double foam_amount;               /* :34 */
    int32_t spectrum_seed[2];         /* :37 */
    int32_t should_generate_spectrum; /* :38  dirty flag; cleared by the library when it regenerates */
    double time;                      /* :40  advanced by ocean_update */
    double foam_grow_rate;            /* :41  written by ocean_update */
    double foam_decay_rate;           /* :42  written by ocean_update */
} ocean_cascade_params;

typedef struct ocean_info {
    int32_t device;
    int32_t map_size;
    int32_t num_cascades;
    int32_t pending_cascades;      /* pass_num_cascades_remaining, wave_generator.gd:15 */
    uint64_t kernel_launches;      /* kernels launched by this generator since creation */
    uint64_t cascade_updates;      /* cascade updates executed since creation */
    uint64_t device_bytes;         /* device memory owned by the generator */
} ocean_info;

/* class defaults of wave_cascade_parameters.gd:7-42 */
int ocean_default_cascade_params(ocean_cascade_params* out);

/* WaveGenerator.map_size + WaveGenerator.init_gpu(num_cascades), wave_generator.gd:8,17-54.
 * map_size in {128,256,512,1024} (water.gd:38); num_cascades >= 1 (the reference passes
 * max(2, n), water.gd:91 -- callers may do the same).  Allocates the spectrum (RGBA32F x
 * layers), the row-pass scratch, the two RGBA16F layered maps and the twiddle table. */
int ocean_create(int device, int map_size, int num_cascades, ocean_generator** out);

/* NOTIFICATION_PREDELETE -> context.free(), wave_generator.gd:111-113, render_context.gd:40-46 */
int ocean_destroy(ocean_generator* gen);

/* WaveGenerator.update(delta, parameters), wave_generator.gd:90-109: flushes cascades
 * 0..remaining-1 left from the previous pass, then time += delta and the foam rates for every
 * element of parameters[0..count), then arms `count` pending cascades.  `parameters` is in/out
 * (time, foam rates and the dirty flags of flushed cascades are written back). */
int ocean_update(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count);

/* WaveGenerator._process, wave_generator.gd:56-63: runs ONE pending cascade (highest index
 * first).  If `parameters` is non-NULL the live values are re-read (the reference dereferences the
 * live Resource objects) and the dirty flag is written back.  No-op when nothing is pending. */
int ocean_process(ocean_generator* gen, ocean_cascade_params* parameters, int count);

/* Batched fast path: ocean_update() followed by all pending cascades in one fused launch pair
 * (what `count` rendered frames of _process produce; cascades are independent,
 * wave_generator.gd:96-97). */
int ocean_update_all(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count);

/* `frames` consecutive ocean_update_all(delta) calls of the same resident cascades, fused: after the first frame the
 * remaining ones run `256 / count` frames per launch, chained on the device through per-cascade completion counters (consecutive
 * frames use alternate halves of the row-pass scratch: the row pass of frame f+1 runs beside the column pass of frame f and only
 * waits for the column pass of frame f-1, the column pass of frame f+1 for its own row pass and -- foam plane -- for the column
 * pass of frame f; the times are accumulated on the host in binary64, one addition per frame, exactly as wave_generator.gd:103 does).  Results are bit-identical to the frame-by-frame
 * calls; what it removes is the per-frame launch and host latency (SURVEY 8d cfg3: 1000-frame foam accumulate/decay loop). */
int ocean_update_frames(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count, int frames);

/* ---- the Water node's side of the hand-off (assets/water/water.gd), for hosts that do not bring their own ----
 * ocean_scheduler: the fixed-rate update accumulator of water.gd:51-54,62-63,75-82 as a POD state machine (binary64, the
 * arithmetic of the GDScript).  ocean_scheduler_tick(delta) is Water._process(delta) without the generator call: it returns 1
 * when an update is due and writes the delta to pass to WaveGenerator.update (target period + overshoot, or the frame delta
 * when updates_per_second == 0), then advances the clock.  ocean_scheduler_set_rate is the updates_per_second setter (:52-54).
 * ocean_water_frame is one rendered frame of the node pair: Water._process (tick, ocean_update when due) followed by the child
 * WaveGenerator._process (ocean_process: one pending cascade).  ocean_map_scales fills map_scales[i] = (1 / tile_length.xy,
 * displacement_scale, normal_scale) (water.gd:102-110; the quotients are binary32 as Vector2.ONE / tile_length is).
 * ocean_water_default_time(i) = 120.0 + PI * i, the cascade start time of water.gd:32. */
typedef struct ocean_scheduler {
    double updates_per_second;   /* water.gd:51, default 50 */
    double time;                 /* :62 */
    double next_update_time;     /* :63 */
} ocean_scheduler;
int ocean_scheduler_init(ocean_scheduler* s, double updates_per_second);
int ocean_scheduler_set_rate(ocean_scheduler* s, double updates_per_second);
int ocean_scheduler_tick(ocean_scheduler* s, double delta, double* update_delta);
int ocean_water_frame(ocean_generator* gen, ocean_scheduler* s, double delta, ocean_cascade_params* parameters, int count,
                      int* did_update);
int ocean_map_scales(const ocean_cascade_params* parameters, int count, float* map_scales /* [count][4] */);
double ocean_water_default_time(int cascade);

/* descriptors[&'displacement_map'].rid / descriptors[&'normal_map'].rid, wave_generator.gd:34-35,
 * water.gd:95-96.  Device pointers to [num_cascades][map_size][map_size][4] IEEE half (RGBA16F),
 * layer-major, tightly packed: displacement = (hx,hy,hz,0), normal = (dy/dx/(1+|dxx|),
 * dy/dz/(1+|dzz|), dhx_dx, foam) (fft_unpack.glsl:50,66-67). */
int ocean_get_maps(ocean_generator* gen, void** displacement_dev, void** normal_dev, size_t* layer_bytes);

/* Host hand-off for RenderingDevice.texture_update(rid, layer, bytes) (the maps are created with
 * TEXTURE_USAGE_CAN_UPDATE_BIT, wave_generator.gd:34-35).  Copies layers [first, first+count).
 * Either destination may be NULL.  The _async form returns after enqueueing on the generator's
 * stream (use pinned memory from ocean_host_alloc and ocean_synchronize). */
int ocean_copy_maps_to_host(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host);
int ocean_copy_maps_to_host_async(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host);
/* Overlapped hand-off: snapshots the layers on the device (one device-to-device copy on the generator's stream) and moves the
 * snapshot to (pinned) host memory on a second stream, so the NEXT update runs while the maps of this one cross PCIe.
 * ocean_wait_snapshot() returns when the most recent snapshot has arrived; a new snapshot waits for the previous one to have left
 * the device.  Use two host buffers alternately. */
int ocean_snapshot_maps_to_host_async(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host);
int ocean_wait_snapshot(ocean_generator* gen);
int ocean_synchronize(ocean_generator* gen);
int ocean_host_alloc(void** ptr, size_t bytes); /* pinned host memory */
int ocean_host_free(void* ptr);

/* descriptors[&'spectrum'] (RGBA32F, TEXTURE_USAGE_CAN_COPY_FROM_BIT, wave_generator.gd:31):
 * [map_size][map_size][4] float = (Re h0(k), Im h0(k), Re h0(-k), -Im h0(-k)) for one cascade. */
int ocean_copy_spectrum_to_host(ocean_generator* gen, int cascade, float* host);

/* Injects wave amplitudes in place of spectrum_compute's output (test / authoring tap): amplitudes = [map_size][map_size][2]
 * float, A(id) for every texel id = (x, y) (the value get_spectrum_amplitude(id) would return, spectrum_compute.glsl:103-115).
 * The library stores spectrum[id] = (A(id), conj A(mod(-id, N))) exactly as spectrum_compute.glsl:121-124 does, so the texture stays
 * consistent with what the time-propagation stage assumes.  Pass should_generate_spectrum = 0 for that cascade afterwards, or the
 * next update regenerates the spectrum from the parameters. */
int ocean_set_spectrum_amplitudes(ocean_generator* gen, int cascade, const float* amplitudes);

/* Host evaluation of the DETMATH exp (DESIGN.md): the library computes exp(-foam_decay_rate), uniform per dispatch
 * (fft_unpack.glsl:62), on the host with the same binary64 operation sequence the device functions use.  Exported so
 * that the agreement can be checked without a GPU (tests/test_abi_cpu.py). */
float ocean_detmath_expf(float x);

/* Batched map queries -- the sampling contract of the water shader as an op (what buoyancy / gameplay code needs):
 *   displacement[p]   = sum_i texture(displacements, vec3(xz*scales_i.xy, i)).xyz * scales_i.z         water.gdshader:27-39
 *   gradient_foam[p]  = sum_i mix(texture_bicubic(normals, c_i), texture(normals, c_i), min(1, ppm_i*0.1)).xyw
 *                             * vec3(scales_i.ww, 1),  ppm_i = map_size * min(scales_i.x, scales_i.y)   water.gdshader:42-84
 * over the first num_cascades layers, map_scales[i] = (1/tile_length.x, 1/tile_length.y, displacement_scale,
 * normal_scale) as in assets/water/water.gd:102-110.  points_xz: [num_points][2] world x,z (UV = VERTEX.xz);
 * outputs: [num_points][3] float each.  texture() = exact-weight bilinear filter with REPEAT addressing, binary32,
 * shader operation order (oracle/sampling.py is the specification).  |xz * scale * map_size| must stay below 2^31.
 * ocean_sample_maps takes host buffers (copies inside, synchronous); ocean_sample_maps_device takes device pointers for
 * points and outputs (map_scales stays a host array) and is asynchronous on the generator's stream. */
int ocean_sample_maps(ocean_generator* gen, int num_points, const float* points_xz_host, int num_cascades, const float* map_scales_host,
                      float* displacement_host, float* gradient_foam_host);
int ocean_sample_maps_device(ocean_generator* gen, int num_points, const float* points_xz_dev, int num_cascades, const float* map_scales_host,
                             float* displacement_dev, float* gradient_foam_dev);

/* Surface query -- where is the water surface above the world point q = (x, z)?  The water shader moves every vertex
 * sideways as well as up (water.gdshader:31-37, VERTEX += displacement), so ocean_sample_maps at q returns the displacement of
 * a surface point that has moved away from q.  This op finds the undisplaced position p whose vertex lands over q,
 *   p + D.xz(p) = q,   D(p) = sum_i texture(displacements, vec3(p * map_scales[i].xy, i)).xyz * map_scales[i].z,
 * and returns the height D.y(p) and ocean_sample_maps' gradient/foam at p (all over the first num_cascades layers, map_scales as
 * for ocean_sample_maps).  Solver: from p_0 = q, exactly `iterations` (K, in [0, OCEAN_SURFACE_MAX_ITERATIONS]) damped Newton
 * steps on the exact Jacobian J = I + dD.xz/dxz of the bilinear filter (it reads the same four texels as D): where det J > 0.05
 * the step is J^-1 r with r = p + D.xz(p) - q, elsewhere (folds, NaN) the fixed-point step r; a step longer than 2|r| is
 * shortened to 2|r|.  No early exit, so results are deterministic; binary32 with the operation order oracle/surface.py
 * specifies.  K = 8 (the Python default) leaves a residual of at most 1 mm on 98.5 % (512 x 512 x 4 demo cascades) to 99.8 %
 * (128 x 128 x 3) of random points, K = 12 on 99.5 %; a choppier sea needs more steps (8 demo cascades of 1024 x 1024: 85.5 %
 * at K = 8).  K = 0 returns ocean_sample_maps(q) at the source point q.
 * Folds: where the surface folds over itself (jacobian <= 0, the foam regions) q can have zero or several preimages.  The op
 * does not hide this: `residual` and `jacobian` describe the point where the K steps ended and the caller decides (a float can,
 * for instance, keep its previous source point or accept a residual of a few centimetres).
 * ocean_query_surface takes host buffers (copies inside, synchronous); ocean_query_surface_device takes device pointers for the
 * points and the records (map_scales stays a host array) and is asynchronous on the generator's stream. */
#define OCEAN_SURFACE_MAX_ITERATIONS 32
typedef struct ocean_surface_point {  /* 32 B */
    float height;                     /* D.y at the solved source point: surface height above q */
    float source_x, source_z;         /* p, the undisplaced position whose vertex lands over q (feed it to ocean_sample_maps) */
    float residual;                   /* |p + D.xz(p) - q|, metres */
    float gradient_foam[3];           /* ocean_sample_maps' gradient/foam at p */
    float jacobian;                   /* det(I + dD.xz/dxz) at p; <= 0: folded surface */
} ocean_surface_point;
int ocean_query_surface(ocean_generator* gen, int num_points, const float* points_xz_host, int num_cascades, const float* map_scales_host,
                        int iterations, ocean_surface_point* out_host);
int ocean_query_surface_device(ocean_generator* gen, int num_points, const float* points_xz_dev, int num_cascades,
                               const float* map_scales_host, int iterations, ocean_surface_point* out_dev);

/* Spray candidates -- the spawn test of the sea-spray particle shader as a stream-compaction op
 * (assets/shaders/spatial/sea_spray_particle.gdshader:80-94; the reference evaluates it for every particle of the emitter and
 * culls the inactive ones, README.md:29).  For each candidate START_POS.xz:
 *   gradient = sum_i texture(normals, vec3(xz * map_scales[i].xy, i)).xyw;  normal = normalize(vec3(-gradient.x, 1, -gradient.y));
 *   foam = gradient.z;  normal_factor = mix(.25, 1, min((normal.y - .92) / (.99 - .92), 1));  foam_factor likewise on [.9, 1];
 *   ACTIVE = normal_factor in [0, 1] && foam > .9;  SCALE_FACTOR = normal_factor * foam_factor;
 *   PARTICLE_SCALE = vec3(foam_factor * (1 + 1e-3)) * vec3(1, normal_factor, 1) * particle_scale
 * Only the ACTIVE candidates are returned, in candidate order (stable compaction, deterministic).  *num_active receives their
 * number even when it exceeds max_records (records beyond max_records are dropped).  oracle/spray.py is the specification.
 * ocean_spray_grid fills the start positions of the emitter's particle grid (sea_spray_particle.gdshader:47,52-54):
 * emission_transform = 3 x 4 row-major (basis columns, origin), NULL = identity; points_xz_host: [num_particles][2]. */
typedef struct ocean_spray_record {
    uint32_t index;            /* candidate (particle INDEX) */
    float start_x, start_z;    /* START_POS.xz */
    float scale_factor;        /* SCALE_FACTOR (:90) */
    float particle_scale[3];   /* PARTICLE_SCALE (:92-94) */
    float foam;                /* summed normal_map.a at the start position */
} ocean_spray_record;
int ocean_spray_grid(int num_particles, const float* emission_transform, float* points_xz_host);
int ocean_extract_spray(ocean_generator* gen, int num_candidates, const float* points_xz_host, int num_cascades,
                        const float* map_scales_host, const float* particle_scale, int max_records,
                        ocean_spray_record* records_host, int* num_active);
/* device pointers for the candidates, the records and the count (asynchronous on the generator's stream) */
int ocean_extract_spray_device(ocean_generator* gen, int num_candidates, const float* points_xz_dev, int num_cascades,
                               const float* map_scales_host, const float* particle_scale, int max_records,
                               ocean_spray_record* records_dev, int* num_active_dev);

/* Parity/debug taps (not timed): binary32 maps before the half conversion, the row-pass output
 * ([4][N][N][2] float, == fft_buffer half 1 after the first fft_compute, wave_generator.gd:79) and
 * the twiddle table ([N-1][2] float: stage s, index j at (1<<s)-1+j; fft_butterfly.glsl:27).
 * The row-pass scratch is only preserved while the taps are enabled (otherwise the column pass discards it from
 * L2 as soon as it is consumed): ocean_copy_rowpass_to_host returns OCEAN_ERR_STATE with the taps off. */
int ocean_enable_f32_taps(ocean_generator* gen, int enable);
int ocean_copy_f32_maps_to_host(ocean_generator* gen, int cascade, float* displacement_host, float* normal_host);
int ocean_copy_rowpass_to_host(ocean_generator* gen, int cascade, float* host);
int ocean_copy_twiddles_to_host(ocean_generator* gen, float* host);

/* Checkpoint/resume of the only frame-to-frame state, normal_map.a (fft_unpack.glsl:61-64):
 * [map_size][map_size] IEEE half for one cascade. */
int ocean_get_foam_state(ocean_generator* gen, int cascade, uint16_t* host);
int ocean_set_foam_state(ocean_generator* gen, int cascade, const uint16_t* host);

/* static func JONSWAP_alpha / JONSWAP_peak_angular_frequency, wave_generator.gd:116-121
 * (fetch_length in metres, binary64). */
double ocean_jonswap_alpha(double wind_speed, double fetch_length);
double ocean_jonswap_peak_angular_frequency(double wind_speed, double fetch_length);

/* Device-side timing on the generator's stream (CUDA events), used by bench.py. */
int ocean_timer_start(ocean_generator* gen);
int ocean_timer_stop(ocean_generator* gen, float* elapsed_ms); /* synchronizes */

/* Per-kernel device times of the most recent launch sequence (CUDA events between the kernels):
 * spectrum generation, then kernel A (time propagation + row IFFT) and kernel B (column IFFT + maps)
 * of the FIRST L2-sized chunk, whose cascade count is returned through chunk_cascades. */
int ocean_set_profiling(ocean_generator* gen, int enable);
int ocean_get_last_kernel_times(ocean_generator* gen, float* spectrum_ms, float* rowpass_ms, float* colpass_ms,
                                int* chunk_cascades);

/* Device self-test: the kernels' branch-free correctly-rounded sqrt/div against the IEEE intrinsics
 * (every binary32 in [2^-100, 2^100] for sqrt, ~1.2e9 random pairs for div). */
int ocean_selftest_math(ocean_generator* gen, uint64_t* failures, uint64_t* tested);

/* Host-side view of the persistent kernel's work queue for `count` cascades of `map_size` (no GPU needed): writes up to `capacity`
 * packed items (bit 31 = column-pass item, bits 16..30 = dispatch slot, bits 0..15 = block) in hand-out order and returns the item
 * count (negative status on error).  frames == 0: the order of a single update for the given group size and lag (0 = the library's
 * defaults for that map size, after OCEAN_QUEUE_GROUP / OCEAN_QUEUE_LAG), slot = cascade position.  frames >= 1: the order of a
 * fused launch of that many consecutive updates (ocean_update_frames), slot = frame * count + cascade position.  Lets the
 * deadlock-freedom invariant -- whatever an item waits for was handed out before it, each item exactly once -- be checked on the
 * CPU (tests/test_abi_cpu.py). */
int ocean_debug_work_queue(int map_size, int count, int group, int lag, int frames, int32_t* items, int capacity);

/* Host-side view of the completion-counter protocol of a fused launch (ocean_update_frames; no GPU needed).  `counters` holds
 * 3 * num_cascades values -- [c] row passes of cascade c in scratch half 0, [num_cascades + c] its column passes,
 * [2 * num_cascades + c] its row passes in half 1 -- as they stand when a launch of `frames` frames (frame indices first_frame,
 * first_frame + 1, ... of the call) over cascades 0..count-1 starts; on return they hold the values after the launch.  `records`
 * receives, per (frame, cascade) in the dispatch-slot order of ocean_debug_work_queue(frames >= 1), six int32:
 * cascade, counter the row pass bumps / the column pass waits on, its target, the column-pass count the row pass waits for, the
 * column-pass count the column pass waits for, first scratch layer pair.  tests/test_queue_protocol_cpu.py runs this protocol on
 * the CPU against random team schedules and checks that no item ever reads unfinished or overwritten data and that nobody waits forever. */
int ocean_debug_frame_protocol(int map_size, int num_cascades, int count, int first_frame, int frames, uint32_t* counters, int32_t* records);

int ocean_get_info(ocean_generator* gen, ocean_info* out);
const char* ocean_last_error(void);
const char* ocean_version(void);

#ifdef __cplusplus
}
#endif
#endif /* OCEAN_H */
