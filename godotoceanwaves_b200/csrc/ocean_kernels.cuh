// ocean_kernels.cuh -- launch interface between the C-ABI layer (ocean_api.cu) and the
// sm_100a kernels (ocean_kernels.cu).  Internal; the public surface is include/ocean.h.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace ocean {

constexpr int kMaxMapSize = 1024;
constexpr int kTwiddleCount = kMaxMapSize - 1;   // stage s, index j (< 2^s) lives at (1<<s)-1+j

// Push constants of spectrum_compute.glsl:18-30 for one dirty cascade (already binary32).
struct SpectrumDispatch {
    int32_t cascade;
    int32_t seed_x, seed_y;
    float tile_x, tile_y;
    float alpha, peak_frequency, wind_speed, angle, depth, swell, detail, spread;
};

// Push constants of spectrum_modulate.glsl:24-29 and fft_unpack.glsl:20-25 for one cascade update.  tile_length and
// depth do not travel per update: everything spectrum_modulate derives from them (k_vec, k_unit, the dispersion
// relation, :59-61,49) is time-invariant and lives in the dispersion table `table_slot` points at (TableDispatch).
struct CascadeDispatch {
    int32_t cascade;
    int32_t table_slot;
    float time;
    float whitecap, foam_grow_rate, foam_decay_factor;   // factor = DETMATH exp(-foam_decay_rate), fft_unpack.glsl:62 (uniform per dispatch)
    uint32_t done_target;  // persistent kernel: value of done[done_slot] once this update's row pass is complete (wraps)
    uint32_t wait_target;  // multi-frame launches: value of colpass_done[cascade] once the column pass that last READ this update's
                           // half of the scratch (two frames back) is complete -- the row pass may then overwrite it
    uint32_t col_wait_target;  // multi-frame launches: value of colpass_done[cascade] once the PREVIOUS frame's column pass is complete
                               // (it owns the foam plane this update's column pass reads and the maps it overwrites)
    int32_t done_slot;     // row-pass completion counter of this update: cascade (scratch half 0) or 2 * num_cascades + cascade
                           // (half 1) -- one counter per half, because the row pass of frame f+1 runs beside the column pass
                           // of frame f and its items must not be counted towards frame f's row pass
    int32_t scratch_layer; // first of the cascade's two layer pairs in the row-pass scratch: 2 * cascade in half 0,
                           // 2 * (num_cascades + cascade) in half 1 (consecutive frames of a multi-frame launch alternate)
};
constexpr int kScratchHalves = 2;

// One dispersion table to (re)build: spectrum_modulate.glsl:59-61,49 for every wave vector of a tile.
struct TableDispatch {
    int32_t slot;
    float tile_x, tile_y, depth;
};

struct DeviceBuffers {
    int map_size;
    int num_cascades;
    float4* spectrum;      // [C][N][N] (Re h0(k), Im h0(k), Re h0(-k), -Im h0(-k))      RGBA32F
    float4* rowpass;       // [kScratchHalves][C][2][N][N] (re_a, re_b, im_a, im_b), pair p = layers (2p, 2p+1)
    uint2* displacement;   // [C][N][N] 4 x half                                          RGBA16F
    uint2* normal;         // [C][N][N] 4 x half, .a = foam state                         RGBA16F
    float4* displacement_f32;  // optional taps (nullptr when disabled)
    float4* normal_f32;
    const float2* twiddles;    // [kTwiddleCount] global copy of the universal twiddle table
    float4* disp_table;        // [slots][N/2+1][N] (omega, k_vec.x, k_unit.y, k_unit.x) of texel (x, y), y <= N/2
    float* disp_kvy;           // [slots][N] k_vec.y of row y (first N/2+1 entries used)
    alignas(64) CUtensorMap rowpass_tmap;   // TMA descriptor of `rowpass` (kernel B panel loads)
};

// Builds the TMA descriptor of the row-pass scratch (driver entry point cuTensorMapEncodeTiled).
cudaError_t make_rowpass_tensor_map(void* rowpass, int map_size, int num_cascades, CUtensorMap* out);

// Opts the kernels of `map_size` into their dynamic shared-memory footprint (once per device).
cudaError_t configure_kernels(int map_size);

// Computes the universal twiddle table (fft_butterfly.glsl:27) into `twiddles_dev` and into the
// module's __constant__ copy used for warp-uniform lookups.
cudaError_t init_twiddles(float2* twiddles_dev, cudaStream_t stream);

// spectrum_compute.glsl for `count` dirty cascades (dispatch records in device memory).
cudaError_t launch_spectrum_compute(const DeviceBuffers& b, const SpectrumDispatch* dispatch_dev, int count,
                                    cudaStream_t stream);

// Dispersion tables (time-invariant part of spectrum_modulate.glsl: k_vec, k_unit, dispersion_relation) for `count`
// (tile_length, depth) keys, IEEE-exact operations in the shader's order.
cudaError_t launch_dispersion_tables(const DeviceBuffers& b, const TableDispatch* jobs_dev, int count, cudaStream_t stream);

// spectrum_modulate + row IFFT (kernel A) and column IFFT + fft_unpack (kernel B) for `count`
// cascades, issued as L2-sized chunks (chunk_cascades) of one launch pair each.
// Returns the number of kernels launched through *launched.  `mid` / `mid2` (optional) are recorded
// after kernel A / kernel B of the FIRST chunk (per-kernel timing for bench.py).
cudaError_t launch_cascade_update(const DeviceBuffers& b, const CascadeDispatch* dispatch_dev, int count,
                                  cudaStream_t stream, int* launched, cudaEvent_t mid = nullptr, cudaEvent_t mid2 = nullptr);
int chunk_cascades(int map_size);

// Same work as launch_cascade_update in ONE persistent launch (work queue over A and B items, B items
// wait on per-cascade completion counters).  `dispatch_host` (<= kMaxPersistentCascades records) travels by
// value as a kernel parameter (constant bank).  queue_dev: [0] = work counter, [1 + s] = completion counter s (row pass of
// cascade c in scratch half 0: s = c, column pass: C + c, row pass in half 1: 2C + c; monotonic modulo 2^32;
// dispatch[i].done_target is the value of counter done_slot to wait for).  item_table_dev/total_items from
// build_item_table(map_size, count, persistent_group(map_size)); resident_ctas from persistent_grid_size().
constexpr int kMaxPersistentCascades = 256;
// multi_frame: the records describe several consecutive updates of the same cascades (build_item_table_frames): B items then
// publish their completion in queue_dev[1 + num_cascades + c] and A items wait for wait_target there.
cudaError_t launch_cascade_update_persistent(const DeviceBuffers& b, const CascadeDispatch* dispatch_host, int count,
                                             cudaStream_t stream, int* queue_dev, const int* item_table_dev, int total_items,
                                             int resident_ctas, bool multi_frame = false);
int build_item_table(int map_size, int count, int group, int lag, int* out);
// Queue order of `frames` consecutive updates of the same `count` cascades in one launch: A(f0) A(f1) B(f0) A(f2) B(f1) ... with
// A(f) = the row-pass items of every cascade; slot of (frame f, cascade position c) = f * count + c.  Frames alternate between the
// halves of the scratch: A(f, c) waits for B(f-2, c) (CascadeDispatch::wait_target), B(f, c) for A(f, c) and B(f-1, c).
int build_item_table_frames(int map_size, int count, int frames, int* out);
int b_items_per_cascade(int map_size);
int persistent_group(int map_size);
int persistent_lag(int map_size);     // groups between the row pass and the column pass of a group in the queue order
cudaError_t persistent_grid_size(int map_size, int* out);
int a_items_per_cascade(int map_size);

// Compares the branch-free sqrt/div with __fsqrt_rn/__fdiv_rn on the device (debug entry point).
cudaError_t launch_selftest_math(unsigned long long* failures_dev, unsigned long long* tested_dev, cudaStream_t stream);

// De-interleaves one cascade of the row-pass scratch into [4][N][N][2] floats (debug tap).
cudaError_t launch_rowpass_export(const DeviceBuffers& b, int scratch_layer, float2* out_dev, cudaStream_t stream);
// ocean_sample.cu: batched map queries (water.gdshader:27-39,42-84); scales_dev = map_scales[num_cascades] as float4
cudaError_t launch_sample_maps(const DeviceBuffers& b, int num_cascades, const float2* points_dev, int n, const float4* scales_dev,
                               float* disp_out_dev, float* grad_out_dev, cudaStream_t stream);

// ocean_surface.cu: surface query (water.gdshader:27-39 inverted, then :72-84 at the solved source point); out_dev receives
// n ocean_surface_point records
cudaError_t launch_query_surface(const DeviceBuffers& b, int num_cascades, const float2* points_dev, int n, const float4* scales_dev,
                                 int iterations, void* out_dev, cudaStream_t stream);

// ocean_spray.cu: spray candidates (sea_spray_particle.gdshader:80-94) as a stable stream compaction; counts_dev is
// [spray_blocks(n) + 1] ints of scratch whose last element receives the number of active candidates
int spray_blocks(int n);
cudaError_t launch_extract_spray(const DeviceBuffers& b, int num_cascades, const float2* points_dev, int n, const float4* scales_dev,
                                 float3 particle_scale, int* counts_dev, void* records_dev, int max_records, cudaStream_t stream);

}  // namespace ocean
