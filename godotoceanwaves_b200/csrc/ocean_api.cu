// ocean_api.cu -- the C ABI of libocean.so (include/ocean.h) and the host-side sequencing of
// the reference's WaveGenerator (assets/water/wave_generator.gd:17-121): resource allocation,
// dirty-flag handling, push-constant rounding (assets/render_context.gd:122-135), the
// update / _process pending-cascade state machine, and the hand-off of the finished maps.
// No CPU fallback exists: every compute entry point launches the sm_100a kernels or fails.
#include "../../include/ocean.h"
#include "ocean_kernels.cuh"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <map>
#include <vector>

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define OCEAN_CUDA(expr)                                                                       \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(OCEAN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

constexpr double kG = 9.81;       // wave_generator.gd:5
constexpr double kDepth = 20.0;   // wave_generator.gd:6
constexpr int kRing = 8;          // pinned staging slots for dispatch records

}  // namespace

struct ocean_generator {
    int device = 0;
    int map_size = 0;
    int num_cascades = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;                 // snapshot hand-off: device->host copies that overlap the next update
    cudaEvent_t snap_ready = nullptr, snap_free = nullptr;
    uint2* snap_disp = nullptr;                         // [num_cascades][N][N] snapshot of the maps (lazy)
    uint2* snap_normal = nullptr;
    bool snap_busy = false;
    ocean::DeviceBuffers buf{};
    float2* twiddles = nullptr;
    float2* export_buf = nullptr;                       // rowpass export scratch (lazy)
    float2* q_points = nullptr;                         // query staging (lazy, grown on demand): points, outputs, scales
    float* q_disp = nullptr;
    float* q_grad = nullptr;
    float4* q_scales = nullptr;
    size_t q_capacity = 0;
    int* spray_counts = nullptr;                        // spray op scratch: block counts / offsets (+ total), grown on demand
    int spray_count_capacity = 0;
    void* spray_records = nullptr;                      // spray op staging for the host entry point
    size_t spray_record_capacity = 0;
    void* surface_points = nullptr;                     // surface query staging for the host entry point
    size_t surface_point_capacity = 0;
    ocean::CascadeDispatch* d_cascade = nullptr;        // [num_cascades] (two-kernel path only)
    ocean::SpectrumDispatch* d_spectrum = nullptr;      // [num_cascades]
    ocean::TableDispatch* d_tables = nullptr;           // [num_cascades]
    ocean::CascadeDispatch* h_cascade = nullptr;        // pinned [kRing][num_cascades]
    ocean::SpectrumDispatch* h_spectrum = nullptr;      // pinned [kRing][num_cascades]
    ocean::TableDispatch* h_tables = nullptr;           // pinned [kRing][num_cascades]
    // dispersion tables are keyed by (tile_length, depth): cascades with equal keys share a slot
    struct TableKey { float tile_x, tile_y, depth; };
    std::vector<TableKey> slot_key;                     // [num_cascades] key whose table the slot holds (valid if slot_valid)
    std::vector<char> slot_valid;
    std::vector<int> slot_refs;                         // cascades currently pointing at the slot
    std::vector<int> cascade_slot;                      // [num_cascades] slot of each cascade, -1 = none yet
    std::vector<int> scratch_layer_of;                  // [num_cascades] where the last update left the cascade's row pass (debug tap)
    cudaEvent_t ring_done[kRing] = {};
    int ring_next = 0;
    cudaEvent_t timer_start = nullptr, timer_stop = nullptr;
    cudaEvent_t prof[5] = {};                           // gen-start, A-start, after A(chunk 0), end, after B(chunk 0)
    int prof_chunk = 0;                                 // cascades in the profiled first chunk
    bool profiling = false;
    bool prof_valid = false, prof_had_gen = false;
    int* d_queue = nullptr;                             // [1 + 3 * num_cascades] work counter + completion counters
    std::vector<uint32_t> done_count;                   // host mirror of the completion counters (modulo 2^32)
    int resident_ctas = 0;
    std::map<int, std::pair<int*, int>> item_tables;    // cascades per launch -> (device item table, item count)
    std::map<std::pair<int, int>, std::pair<int*, int>> frame_tables;   // (cascades, frames per launch) -> same, multi-frame order
    bool persistent = true;                             // OCEAN_PIPELINE=split selects the two-kernel path
    std::vector<ocean_cascade_params> pass_parameters;  // wave_generator.gd:14
    int pass_num_cascades_remaining = 0;                // wave_generator.gd:15
    uint64_t kernel_launches = 0;
    uint64_t cascade_updates = 0;
    uint64_t device_bytes = 0;
};

namespace {

// Every entry point runs on the generator's device and hands the caller's current device back on return (a host that
// drives other CUDA work from the same thread -- a torch process, a C# engine host -- must not find its device changed).
struct DeviceScope {
    int prev = -1;
    ~DeviceScope() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    cudaError_t enter(int device) {
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) cur = -1;
        if (cur == device) return cudaSuccess;
        cudaError_t e = cudaSetDevice(device);
        if (e == cudaSuccess) prev = cur;
        return e;
    }
};
int enter_gen(ocean_generator* g, DeviceScope& scope) {
    if (!g) return fail(OCEAN_ERR_INVALID_ARGUMENT, "generator handle is NULL");
    cudaError_t e = scope.enter(g->device);
    if (e != cudaSuccess) return fail(OCEAN_ERR_CUDA, "cudaSetDevice(%d) failed: %s", g->device, cudaGetErrorString(e));
    return OCEAN_OK;
}
#define OCEAN_ENTER(gen)                 \
    DeviceScope device_scope__;          \
    int rc = enter_gen(gen, device_scope__)

template <typename T>
cudaError_t dev_alloc(ocean_generator* g, T** p, size_t count) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
    if (e == cudaSuccess) g->device_bytes += count * sizeof(T);
    return e;
}

void release(ocean_generator* g) {
    if (!g) return;
    DeviceScope scope;
    scope.enter(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    cudaFree(g->buf.disp_table);
    cudaFree(g->buf.disp_kvy);
    cudaFree(g->d_tables);
    if (g->h_tables) cudaFreeHost(g->h_tables);
    cudaFree(g->buf.spectrum);
    cudaFree(g->buf.rowpass);
    cudaFree(g->buf.displacement);
    cudaFree(g->buf.normal);
    cudaFree(g->buf.displacement_f32);
    cudaFree(g->buf.normal_f32);
    cudaFree(g->twiddles);
    cudaFree(g->export_buf);
    cudaFree(g->q_points);
    cudaFree(g->q_disp);
    cudaFree(g->q_grad);
    cudaFree(g->q_scales);
    cudaFree(g->snap_disp);
    cudaFree(g->snap_normal);
    if (g->copy_stream) { cudaStreamSynchronize(g->copy_stream); cudaStreamDestroy(g->copy_stream); }
    if (g->snap_ready) cudaEventDestroy(g->snap_ready);
    if (g->snap_free) cudaEventDestroy(g->snap_free);
    cudaFree(g->spray_counts);
    cudaFree(g->spray_records);
    cudaFree(g->surface_points);
    cudaFree(g->d_cascade);
    cudaFree(g->d_spectrum);
    cudaFree(g->d_queue);
    for (auto& kv : g->item_tables) cudaFree(kv.second.first);
    for (auto& kv : g->frame_tables) cudaFree(kv.second.first);
    if (g->h_cascade) cudaFreeHost(g->h_cascade);
    if (g->h_spectrum) cudaFreeHost(g->h_spectrum);
    for (auto& ev : g->ring_done)
        if (ev) cudaEventDestroy(ev);
    if (g->timer_start) cudaEventDestroy(g->timer_start);
    if (g->timer_stop) cudaEventDestroy(g->timer_stop);
    for (auto& ev : g->prof)
        if (ev) cudaEventDestroy(ev);
    if (g->stream) cudaStreamDestroy(g->stream);
    delete g;
}

// Push constants of wave_generator.gd:69-71 (spectrum_compute) with the binary64 -> binary32
// rounding of render_context.gd:134.
ocean::SpectrumDispatch make_spectrum_dispatch(const ocean_cascade_params& p, int cascade) {
    ocean::SpectrumDispatch d;
    const double alpha = ocean_jonswap_alpha(p.wind_speed, p.fetch_length * 1e3);
    const double omega = ocean_jonswap_peak_angular_frequency(p.wind_speed, p.fetch_length * 1e3);
    d.cascade = cascade;
    d.seed_x = p.spectrum_seed[0];
    d.seed_y = p.spectrum_seed[1];
    d.tile_x = p.tile_length[0];
    d.tile_y = p.tile_length[1];
    d.alpha = (float)alpha;
    d.peak_frequency = (float)omega;
    d.wind_speed = (float)p.wind_speed;
    d.angle = (float)(p.wind_direction * (M_PI / 180.0));   // deg_to_rad
    d.depth = (float)kDepth;
    d.swell = (float)p.swell;
    d.detail = (float)p.detail;
    d.spread = (float)p.spread;
    return d;
}

// DETMATH exp of a binary32 argument (DESIGN.md "DETMATH", same operation sequence as detmath::exp64 in
// detmath.cuh): clamp to [-110, 90], n = rint(x*log2e), two-term ln2 reduction, Taylor polynomial to r^13 in
// binary64, one rounding to binary32.  Evaluated here because exp(-foam_decay_rate) (fft_unpack.glsl:62) is
// uniform per dispatch; std::fma is the exact fused operation, so host and device agree bit for bit.
float exp_det_host(float xf) {
    double x = (double)xf;
    if (x != x) return xf;
    if (x < -110.0) x = -110.0;
    if (x > 90.0) x = 90.0;
    const double fn = std::nearbyint(x * 0x1.71547652b82fep+0);   // default rounding mode: ties to even, like rint() on the device
    double r = std::fma(-fn, 0x1.62e42ff000000p-1, x);
    r = std::fma(-fn, -0x1.718432a1b0e26p-35, r);
    static const double c[12] = {0x1.1eed8eff8d898p-29, 0x1.ae64567f544e4p-26, 0x1.27e4fb7789f5cp-22, 0x1.71de3a556c734p-19,
                                 0x1.a01a01a01a01ap-16, 0x1.a01a01a01a01ap-13, 0x1.6c16c16c16c17p-10, 0x1.1111111111111p-7,
                                 0x1.5555555555555p-5,  0x1.5555555555555p-3,  0x1.0000000000000p-1,  0.0};
    double p = 0x1.6124613a86d09p-33;
    for (int i = 0; i < 11; ++i) p = std::fma(p, r, c[i]);
    volatile double rr = r * r;                                    // a separately rounded product, never contracted
    const double e = std::fma(rr, p, r) + 1.0;
    const long long sb = ((long long)fn + 1023LL) << 52;
    double scale;
    std::memcpy(&scale, &sb, sizeof scale);
    return (float)(e * scale);
}

// Push constants of wave_generator.gd:73 (spectrum_modulate) and :85 (fft_unpack).  tile_length and DEPTH reach the
// kernels through the dispersion table of `table_slot` (assign_table_slot).
ocean::CascadeDispatch make_cascade_dispatch(const ocean_cascade_params& p, int cascade, int table_slot) {
    ocean::CascadeDispatch d;
    d.cascade = cascade;
    d.table_slot = table_slot;
    d.time = (float)p.time;
    d.whitecap = (float)p.whitecap;
    d.foam_grow_rate = (float)p.foam_grow_rate;
    d.foam_decay_factor = exp_det_host(-(float)p.foam_decay_rate);
    d.done_target = 0;
    d.wait_target = 0;
    d.col_wait_target = 0;
    d.done_slot = cascade;
    d.scratch_layer = 2 * cascade;                    // half 0 of the scratch (single updates always use it)
    return d;
}

// Points cascade `i` at the dispersion table of (tile_length, DEPTH): keeps its slot when the key is unchanged, shares a
// slot that already holds the key, otherwise claims an unreferenced slot and queues its (re)build in jobs[*n_jobs].
// There are as many slots as cascades and a cascade holds one reference, so a free slot always exists.
int assign_table_slot(ocean_generator* g, int i, const ocean_cascade_params& p, ocean::TableDispatch* jobs, int* n_jobs) {
    const ocean_generator::TableKey key{p.tile_length[0], p.tile_length[1], (float)kDepth};
    auto same = [&](const ocean_generator::TableKey& k) {
        return std::memcmp(&k, &key, sizeof key) == 0;       // bit equality: the table is a function of the bits
    };
    int cur = g->cascade_slot[i];
    if (cur >= 0 && g->slot_valid[cur] && same(g->slot_key[cur])) return cur;
    if (cur >= 0) {
        g->slot_refs[cur] -= 1;
        g->cascade_slot[i] = -1;
    }
    const int S = (int)g->slot_key.size();
    int pick = -1;
    for (int s2 = 0; s2 < S && pick < 0; ++s2)
        if (g->slot_valid[s2] && same(g->slot_key[s2])) pick = s2;          // shared (or cached) table
    if (pick < 0) {
        for (int s2 = 0; s2 < S && pick < 0; ++s2)
            if (g->slot_refs[s2] == 0) pick = s2;
        if (pick < 0) return -1;                                            // cannot happen (see above)
        g->slot_key[pick] = key;
        g->slot_valid[pick] = 1;
        ocean::TableDispatch job;
        job.slot = pick;
        job.tile_x = key.tile_x;
        job.tile_y = key.tile_y;
        job.depth = key.depth;
        jobs[(*n_jobs)++] = job;
    }
    g->slot_refs[pick] += 1;
    g->cascade_slot[i] = pick;
    return pick;
}

// Runs WaveGenerator._update (wave_generator.gd:65-85) for the cascades listed in `indices`
// (all of them in ONE batched launch sequence; cascades are independent).
int run_cascades(ocean_generator* g, const int* indices, int n) {
    if (n <= 0) return OCEAN_OK;
    const int slot = g->ring_next;
    OCEAN_CUDA(cudaEventSynchronize(g->ring_done[slot]));           // staging slot free again?
    ocean::CascadeDispatch* hc = g->h_cascade + (size_t)slot * g->num_cascades;
    ocean::SpectrumDispatch* hs = g->h_spectrum + (size_t)slot * g->num_cascades;
    ocean::TableDispatch* ht = g->h_tables + (size_t)slot * g->num_cascades;
    int n_dirty = 0, n_tables = 0;
    const uint32_t per_update = (uint32_t)ocean::a_items_per_cascade(g->map_size);
    for (int k = 0; k < n; ++k) {
        const int i = indices[k];
        const ocean_cascade_params& p = g->pass_parameters[i];
        if (p.should_generate_spectrum) hs[n_dirty++] = make_spectrum_dispatch(p, i);   // :68-72
        const int ts = assign_table_slot(g, i, p, ht, &n_tables);
        if (ts < 0) return fail(OCEAN_ERR_STATE, "no free dispersion-table slot (internal error)");
        hc[k] = make_cascade_dispatch(p, i, ts);                     // :73,85
        hc[k].done_target = g->done_count[i] + per_update;           // modulo 2^32
        g->scratch_layer_of[i] = hc[k].scratch_layer;
    }
    // From here on the device is touched.  The host-side state that must agree with it (dirty flags, the mirror of
    // the completion counters, the staging ring) is committed only after everything has been enqueued; on a failure
    // the device counters are re-synchronised from the unchanged mirror so that later launches cannot wait forever.
    bool counters_touched = false;
    auto fail_resync = [&](int code) {
        if (counters_touched) {
            cudaStreamSynchronize(g->stream);
            cudaMemcpy(g->d_queue + 1, g->done_count.data(), sizeof(uint32_t) * g->done_count.size(), cudaMemcpyHostToDevice);
        }
        return code;
    };
#define RUN_CUDA(expr)                                                                                              \
    do {                                                                                                            \
        cudaError_t e__ = (expr);                                                                                   \
        if (e__ != cudaSuccess)                                                                                     \
            return fail_resync(fail(OCEAN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__)); \
    } while (0)
    if (g->profiling) RUN_CUDA(cudaEventRecord(g->prof[0], g->stream));
    if (n_dirty) {
        RUN_CUDA(cudaMemcpyAsync(g->d_spectrum, hs, sizeof(ocean::SpectrumDispatch) * n_dirty, cudaMemcpyHostToDevice, g->stream));
        RUN_CUDA(ocean::launch_spectrum_compute(g->buf, g->d_spectrum, n_dirty, g->stream));
    }
    if (n_tables) {
        RUN_CUDA(cudaMemcpyAsync(g->d_tables, ht, sizeof(ocean::TableDispatch) * n_tables, cudaMemcpyHostToDevice, g->stream));
        RUN_CUDA(ocean::launch_dispersion_tables(g->buf, g->d_tables, n_tables, g->stream));
    }
    const bool two_kernel = !(g->persistent && !g->profiling);
    if (two_kernel)   // the persistent launch takes its dispatch records by value
        RUN_CUDA(cudaMemcpyAsync(g->d_cascade, hc, sizeof(ocean::CascadeDispatch) * n, cudaMemcpyHostToDevice, g->stream));
    RUN_CUDA(cudaEventRecord(g->ring_done[slot], g->stream));
    int launched = 0;
    if (g->profiling) RUN_CUDA(cudaEventRecord(g->prof[1], g->stream));
    if (!two_kernel) {
        // one persistent launch per <= kMaxPersistentCascades cascades (their dispatch records travel by value)
        for (int first = 0; first < n; first += ocean::kMaxPersistentCascades) {
            const int m = (n - first < ocean::kMaxPersistentCascades) ? n - first : ocean::kMaxPersistentCascades;
            auto it = g->item_tables.find(m);
            if (it == g->item_tables.end()) {
                const int group = ocean::persistent_group(g->map_size), lag = ocean::persistent_lag(g->map_size);
                const int total = ocean::build_item_table(g->map_size, m, group, lag, nullptr);
                std::vector<int> host((size_t)total);
                ocean::build_item_table(g->map_size, m, group, lag, host.data());
                int* dev = nullptr;
                RUN_CUDA(dev_alloc(g, &dev, (size_t)total));
                cudaError_t ce = cudaMemcpyAsync(dev, host.data(), sizeof(int) * (size_t)total, cudaMemcpyHostToDevice, g->stream);
                if (ce == cudaSuccess) ce = cudaStreamSynchronize(g->stream);        // host vector goes out of scope
                if (ce != cudaSuccess) {
                    cudaFree(dev);
                    RUN_CUDA(ce);
                }
                it = g->item_tables.emplace(m, std::make_pair(dev, total)).first;
            }
            counters_touched = true;
            RUN_CUDA(ocean::launch_cascade_update_persistent(g->buf, hc + first, m, g->stream, g->d_queue, it->second.first,
                                                             it->second.second, g->resident_ctas));
            launched += 1;
        }
    } else {
        RUN_CUDA(ocean::launch_cascade_update(g->buf, g->d_cascade, n, g->stream, &launched, g->profiling ? g->prof[2] : nullptr,
                                              g->profiling ? g->prof[4] : nullptr));
        // (the device-side completion counters are brought in step with the host mirror at the commit below)
    }
    if (g->profiling) {
        RUN_CUDA(cudaEventRecord(g->prof[3], g->stream));
        g->prof_valid = true;
        g->prof_had_gen = n_dirty != 0;
        const int ch = ocean::chunk_cascades(g->map_size);
        g->prof_chunk = n < ch ? n : ch;
    }
    // ---- commit ----
    for (int k = 0; k < n; ++k) {
        const int i = indices[k];
        g->pass_parameters[i].should_generate_spectrum = 0;          // :72
        g->done_count[i] += per_update;
    }
    if (two_kernel)
        RUN_CUDA(cudaMemcpyAsync(g->d_queue + 1, g->done_count.data(), sizeof(uint32_t) * g->done_count.size(), cudaMemcpyHostToDevice, g->stream));
#undef RUN_CUDA
    g->ring_next = (g->ring_next + 1) % kRing;
    g->kernel_launches += (uint64_t)launched + (n_dirty ? 1 : 0) + (n_tables ? 1 : 0);
    g->cascade_updates += (uint64_t)n;
    return OCEAN_OK;
}

int validate_params(ocean_generator* g, const ocean_cascade_params* parameters, int count) {
    if (!parameters) return fail(OCEAN_ERR_INVALID_ARGUMENT, "parameters is NULL");
    if (count <= 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "parameters.size() must be != 0 (wave_generator.gd:91)");
    if (count > g->num_cascades)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "%d cascades passed but the generator was created with %d layers", count, g->num_cascades);
    for (int i = 0; i < count; ++i) {
        const ocean_cascade_params& p = parameters[i];
        if (!(p.tile_length[0] > 0.0f) || !(p.tile_length[1] > 0.0f))
            return fail(OCEAN_ERR_INVALID_ARGUMENT, "cascade %d: tile_length must be positive", i);
        if (!(p.wind_speed > 0.0) || !(p.fetch_length > 0.0))
            return fail(OCEAN_ERR_INVALID_ARGUMENT, "cascade %d: wind_speed and fetch_length must be positive (setters clamp to 1e-4)", i);
    }
    return OCEAN_OK;
}

int check_cascade(ocean_generator* g, int cascade) {
    if (cascade < 0 || cascade >= g->num_cascades)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "cascade index %d out of range [0,%d)", cascade, g->num_cascades);
    return OCEAN_OK;
}

}  // namespace

extern "C" {

const char* ocean_last_error(void) { return g_last_error.c_str(); }
const char* ocean_version(void) { return "godotoceanwaves_b200 0.1 (sm_100a)"; }

double ocean_jonswap_alpha(double wind_speed, double fetch_length) {             // wave_generator.gd:116-117
    return 0.076 * std::pow(wind_speed * wind_speed / (fetch_length * kG), 0.22);
}
double ocean_jonswap_peak_angular_frequency(double wind_speed, double fetch_length) {   // wave_generator.gd:120-121
    return 22.0 * std::pow(kG * kG / (wind_speed * fetch_length), 1.0 / 3.0);
}

int ocean_default_cascade_params(ocean_cascade_params* out) {                    // wave_cascade_parameters.gd:7-42
    if (!out) return fail(OCEAN_ERR_INVALID_ARGUMENT, "out is NULL");
    std::memset(out, 0, sizeof *out);
    out->tile_length[0] = out->tile_length[1] = 50.0f;
    out->displacement_scale = 1.0;
    out->normal_scale = 1.0;
    out->wind_speed = 20.0;
    out->wind_direction = 0.0;
    out->fetch_length = 550.0;
    out->swell = 0.8;
    out->spread = 0.2;
    out->detail = 1.0;
    out->whitecap = 0.5;
    out->foam_amount = 5.0;
    out->should_generate_spectrum = 1;
    return OCEAN_OK;
}

int ocean_create(int device, int map_size, int num_cascades, ocean_generator** out) {
    if (!out) return fail(OCEAN_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (map_size != 128 && map_size != 256 && map_size != 512 && map_size != 1024)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "map_size %d not in {128,256,512,1024} (water.gd:38)", map_size);
    if (num_cascades < 1) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_layers >= 1 required (render_context.gd:77)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(OCEAN_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(OCEAN_ERR_INVALID_ARGUMENT, "device %d out of range [0,%d)", device, ndev);
    DeviceScope device_scope;
    OCEAN_CUDA(device_scope.enter(device));
    cudaDeviceProp prop;
    OCEAN_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(OCEAN_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);

    ocean_generator* g = new (std::nothrow) ocean_generator();
    if (!g) return fail(OCEAN_ERR_STATE, "out of host memory");
    g->device = device;
    g->map_size = map_size;
    g->num_cascades = num_cascades;
    const size_t NN = (size_t)map_size * map_size;
    const size_t C = (size_t)num_cascades;
#define CREATE_CUDA(expr)                                                                                        \
    do {                                                                                                         \
        cudaError_t e__ = (expr);                                                                                \
        if (e__ != cudaSuccess) {                                                                                \
            release(g);                                                                                          \
            return fail(OCEAN_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__));                        \
        }                                                                                                        \
    } while (0)
    CREATE_CUDA(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    CREATE_CUDA(dev_alloc(g, &g->buf.spectrum, C * NN));                  // wave_generator.gd:31
    CREATE_CUDA(dev_alloc(g, &g->buf.rowpass, ocean::kScratchHalves * C * 2 * NN));               // replaces fft_buffer, :33
    CREATE_CUDA(dev_alloc(g, &g->buf.displacement, C * NN));              // :34
    CREATE_CUDA(dev_alloc(g, &g->buf.normal, C * NN));                    // :35
    CREATE_CUDA(dev_alloc(g, &g->twiddles, (size_t)ocean::kTwiddleCount + 1));   // :32
    CREATE_CUDA(dev_alloc(g, &g->buf.disp_table, C * (size_t)(map_size / 2 + 1) * map_size));   // one slot per cascade at most
    CREATE_CUDA(dev_alloc(g, &g->buf.disp_kvy, C * (size_t)map_size));
    CREATE_CUDA(dev_alloc(g, &g->d_cascade, C));
    CREATE_CUDA(dev_alloc(g, &g->d_spectrum, C));
    CREATE_CUDA(dev_alloc(g, &g->d_tables, C));
    CREATE_CUDA(dev_alloc(g, &g->d_queue, 3 * C + 1));
    CREATE_CUDA(cudaMemsetAsync(g->d_queue, 0, sizeof(int) * (3 * C + 1), g->stream));
    g->done_count.assign(3 * C, 0u);                  // [0, C): row-pass counters (scratch half 0), [C, 2C): column pass, [2C, 3C): row pass, half 1
    g->slot_key.assign(C, ocean_generator::TableKey{0.f, 0.f, 0.f});
    g->slot_valid.assign(C, 0);
    g->slot_refs.assign(C, 0);
    g->cascade_slot.assign(C, -1);
    g->scratch_layer_of.resize(C);
    for (int i = 0; i < C; ++i) g->scratch_layer_of[i] = 2 * i;
    {
        const char* mode = std::getenv("OCEAN_PIPELINE");
        g->persistent = !(mode && std::strcmp(mode, "split") == 0);
    }
    CREATE_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g->h_cascade), sizeof(ocean::CascadeDispatch) * kRing * C, cudaHostAllocDefault));
    CREATE_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g->h_spectrum), sizeof(ocean::SpectrumDispatch) * kRing * C, cudaHostAllocDefault));
    CREATE_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g->h_tables), sizeof(ocean::TableDispatch) * kRing * C, cudaHostAllocDefault));
    for (auto& ev : g->ring_done) CREATE_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreate(&g->timer_start));
    CREATE_CUDA(cudaEventCreate(&g->timer_stop));
    for (auto& ev : g->prof) CREATE_CUDA(cudaEventCreate(&ev));
    // textures start cleared (foam state = 0)
    CREATE_CUDA(cudaMemsetAsync(g->buf.spectrum, 0, sizeof(float4) * C * NN, g->stream));
    CREATE_CUDA(cudaMemsetAsync(g->buf.rowpass, 0, sizeof(float4) * ocean::kScratchHalves * C * 2 * NN, g->stream));
    CREATE_CUDA(cudaMemsetAsync(g->buf.displacement, 0, sizeof(uint2) * C * NN, g->stream));
    CREATE_CUDA(cudaMemsetAsync(g->buf.normal, 0, sizeof(uint2) * C * NN, g->stream));
    g->buf.map_size = map_size;
    g->buf.num_cascades = num_cascades;
    g->buf.twiddles = g->twiddles;
    CREATE_CUDA(ocean::make_rowpass_tensor_map(g->buf.rowpass, map_size, num_cascades, &g->buf.rowpass_tmap));
    CREATE_CUDA(ocean::configure_kernels(map_size));
    CREATE_CUDA(ocean::persistent_grid_size(map_size, &g->resident_ctas));
    CREATE_CUDA(ocean::init_twiddles(g->twiddles, g->stream));            // fft_butterfly once, :52-54
    g->kernel_launches += 1;
    CREATE_CUDA(cudaStreamSynchronize(g->stream));
#undef CREATE_CUDA
    *out = g;
    return OCEAN_OK;
}

int ocean_destroy(ocean_generator* gen) {
    if (!gen) return fail(OCEAN_ERR_INVALID_ARGUMENT, "generator handle is NULL");
    release(gen);
    return OCEAN_OK;
}

int ocean_update(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    rc = validate_params(gen, parameters, count);
    if (rc) return rc;
    // wave_generator.gd:94-98: finish the cascades of the previous pass that were never processed
    if (gen->pass_num_cascades_remaining != 0) {
        std::vector<int> idx(gen->pass_num_cascades_remaining);
        for (int i = 0; i < gen->pass_num_cascades_remaining; ++i) idx[i] = i;
        // the reference dereferences the live Resource objects: refresh from the caller's array where it overlaps
        for (int i = 0; i < gen->pass_num_cascades_remaining && i < count; ++i) gen->pass_parameters[i] = parameters[i];
        rc = run_cascades(gen, idx.data(), (int)idx.size());
        if (rc) return rc;
        for (int i = 0; i < gen->pass_num_cascades_remaining && i < count; ++i)
            parameters[i].should_generate_spectrum = gen->pass_parameters[i].should_generate_spectrum;
        gen->pass_num_cascades_remaining = 0;
    }
    // :100-106
    for (int i = 0; i < count; ++i) {
        ocean_cascade_params& p = parameters[i];
        p.time += delta;
        p.foam_grow_rate = delta * p.foam_amount * 7.5;
        p.foam_decay_rate = delta * std::fmax(0.5, 10.0 - p.foam_amount) * 1.15;
    }
    gen->pass_parameters.assign(parameters, parameters + count);       // :108
    gen->pass_num_cascades_remaining = count;                          // :109
    return OCEAN_OK;
}

int ocean_process(ocean_generator* gen, ocean_cascade_params* parameters, int count) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (gen->pass_num_cascades_remaining == 0) return OCEAN_OK;        // :58
    if (parameters) {
        if (count != (int)gen->pass_parameters.size())
            return fail(OCEAN_ERR_INVALID_ARGUMENT, "ocean_process: count %d differs from the armed pass (%d)", count, (int)gen->pass_parameters.size());
        rc = validate_params(gen, parameters, count);
        if (rc) return rc;
    }
    gen->pass_num_cascades_remaining -= 1;                             // :59
    const int i = gen->pass_num_cascades_remaining;
    if (parameters) gen->pass_parameters[i] = parameters[i];
    rc = run_cascades(gen, &i, 1);                                     // :61-63
    if (rc) return rc;
    if (parameters) parameters[i].should_generate_spectrum = gen->pass_parameters[i].should_generate_spectrum;
    return OCEAN_OK;
}

int ocean_update_all(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count) {
    int rc = ocean_update(gen, delta, parameters, count);
    if (rc) return rc;
    std::vector<int> idx(count);
    for (int i = 0; i < count; ++i) idx[i] = i;
    rc = run_cascades(gen, idx.data(), count);
    if (rc) return rc;
    for (int i = 0; i < count; ++i) parameters[i].should_generate_spectrum = gen->pass_parameters[i].should_generate_spectrum;
    gen->pass_num_cascades_remaining = 0;
    return OCEAN_OK;
}

// ---- completion-counter protocol of a fused launch: pure host arithmetic, shared by ocean_update_frames and by
// ocean_debug_frame_protocol (tests/test_queue_protocol_cpu.py runs it against random schedules on the CPU) ----
// counters[0, C): row passes in scratch half 0, [C, 2C): column passes, [2C, 3C): row passes in half 1 -- their values when the
// launch starts (every earlier launch is complete by then).  Frame f of the launch is frame first_frame + f of the call.
// Frame `first_frame + f` runs in half (first_frame + f) & 1 of the scratch, so its row pass only waits for the column pass two
// frames back and runs beside the previous frame's column pass; its column pass waits for its own row pass and -- foam plane,
// maps -- for the previous frame's column pass.  The halves count their row passes separately (frames f, f-2, ... of the launch).
static void frame_protocol_targets(ocean::CascadeDispatch& d, const uint32_t* counters, int C, int i, int first_frame, int f,
                                   uint32_t a_per, uint32_t b_per) {
    const int half = (first_frame + f) & 1;
    d.done_slot = half ? 2 * C + i : i;
    d.done_target = counters[d.done_slot] + (uint32_t)(f / 2 + 1) * a_per;
    d.wait_target = counters[C + i] + (uint32_t)(f > 0 ? f - 1 : 0) * b_per;
    d.col_wait_target = counters[C + i] + (uint32_t)f * b_per;
    d.scratch_layer = 2 * (half * C + i);
}
// the counters once a launch of F frames starting at frame first_frame is complete
static void frame_protocol_commit(uint32_t* counters, int C, int i, int first_frame, int F, uint32_t a_per, uint32_t b_per) {
    const int first_half = first_frame & 1;                        // half of the launch's frame 0; it runs (F + 1) / 2 frames there
    counters[first_half ? 2 * C + i : i] += (uint32_t)((F + 1) / 2) * a_per;
    counters[first_half ? i : 2 * C + i] += (uint32_t)(F / 2) * a_per;
    counters[C + i] += (uint32_t)F * b_per;
}

int ocean_debug_frame_protocol(int map_size, int num_cascades, int count, int first_frame, int frames, uint32_t* counters, int32_t* records) {
    const uint32_t a_per = (uint32_t)ocean::a_items_per_cascade(map_size), b_per = (uint32_t)ocean::b_items_per_cascade(map_size);
    if (a_per == 0 || num_cascades < 1 || count < 1 || count > num_cascades || first_frame < 0 || frames < 1 || !counters || !records)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "ocean_debug_frame_protocol: bad arguments");
    for (int f = 0; f < frames; ++f)
        for (int i = 0; i < count; ++i) {
            ocean::CascadeDispatch d{};
            d.cascade = i;
            frame_protocol_targets(d, counters, num_cascades, i, first_frame, f, a_per, b_per);
            int32_t* r = records + ((size_t)f * count + i) * 6;
            r[0] = d.cascade; r[1] = d.done_slot; r[2] = (int32_t)d.done_target; r[3] = (int32_t)d.wait_target;
            r[4] = (int32_t)d.col_wait_target; r[5] = d.scratch_layer;
        }
    for (int i = 0; i < count; ++i) frame_protocol_commit(counters, num_cascades, i, first_frame, frames, a_per, b_per);
    return OCEAN_OK;
}

int ocean_update_frames(ocean_generator* gen, double delta, ocean_cascade_params* parameters, int count, int frames) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (frames < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "frames %d is negative", frames);
    if (frames == 0) return OCEAN_OK;
    const int per_launch = count > 0 ? ocean::kMaxPersistentCascades / count : 0;
    if (!gen->persistent || gen->profiling || per_launch < 2) {        // two-kernel path / huge sets: frame by frame
        for (int f = 0; f < frames; ++f)
            if ((rc = ocean_update_all(gen, delta, parameters, count))) return rc;
        return OCEAN_OK;
    }
    // frame 0 exactly as ocean_update_all: flush of a pending pass, time/rate advance, spectra and tables where needed
    if ((rc = ocean_update_all(gen, delta, parameters, count))) return rc;
    const uint32_t a_per = (uint32_t)ocean::a_items_per_cascade(gen->map_size), b_per = (uint32_t)ocean::b_items_per_cascade(gen->map_size);
    const int C = gen->num_cascades;
    std::vector<ocean::CascadeDispatch> rec;
    int done = 1;
    while (done < frames) {
        const int F = (frames - done < per_launch) ? frames - done : per_launch;
        rec.resize((size_t)F * count);
        for (int f = 0; f < F; ++f) {
            for (int i = 0; i < count; ++i) {                              // wave_generator.gd:100-106, once per frame
                ocean_cascade_params& p = parameters[i];
                p.time += delta;
                p.foam_grow_rate = delta * p.foam_amount * 7.5;
                p.foam_decay_rate = delta * std::fmax(0.5, 10.0 - p.foam_amount) * 1.15;
                ocean::CascadeDispatch d = make_cascade_dispatch(p, i, gen->cascade_slot[i]);
                frame_protocol_targets(d, gen->done_count.data(), C, i, done, f, a_per, b_per);
                gen->scratch_layer_of[i] = d.scratch_layer;
                rec[(size_t)f * count + i] = d;
            }
        }
        auto key = std::make_pair(count, F);
        auto it = gen->frame_tables.find(key);
        if (it == gen->frame_tables.end()) {
            const int total = ocean::build_item_table_frames(gen->map_size, count, F, nullptr);
            std::vector<int> host((size_t)total);
            ocean::build_item_table_frames(gen->map_size, count, F, host.data());
            int* dev = nullptr;
            OCEAN_CUDA(dev_alloc(gen, &dev, (size_t)total));
            cudaError_t ce = cudaMemcpyAsync(dev, host.data(), sizeof(int) * (size_t)total, cudaMemcpyHostToDevice, gen->stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(gen->stream);
            if (ce != cudaSuccess) {
                cudaFree(dev);
                return fail(OCEAN_ERR_CUDA, "item table upload failed: %s", cudaGetErrorString(ce));
            }
            it = gen->frame_tables.emplace(key, std::make_pair(dev, total)).first;
        }
        cudaError_t le = ocean::launch_cascade_update_persistent(gen->buf, rec.data(), F * count, gen->stream, gen->d_queue, it->second.first,
                                                                 it->second.second, gen->resident_ctas, true);
        if (le != cudaSuccess) {
            cudaStreamSynchronize(gen->stream);
            cudaMemcpy(gen->d_queue + 1, gen->done_count.data(), sizeof(uint32_t) * gen->done_count.size(), cudaMemcpyHostToDevice);
            return fail(OCEAN_ERR_CUDA, "multi-frame launch failed: %s", cudaGetErrorString(le));
        }
        for (int i = 0; i < count; ++i) frame_protocol_commit(gen->done_count.data(), C, i, done, F, a_per, b_per);
        gen->kernel_launches += 1;
        gen->cascade_updates += (uint64_t)F * count;
        done += F;
    }
    gen->pass_parameters.assign(parameters, parameters + count);
    for (int i = 0; i < count; ++i) gen->pass_parameters[i].should_generate_spectrum = 0;
    gen->pass_num_cascades_remaining = 0;
    return OCEAN_OK;
}

// ---- Water node hand-off (assets/water/water.gd) ----
int ocean_scheduler_init(ocean_scheduler* s, double updates_per_second) {
    if (!s) return fail(OCEAN_ERR_INVALID_ARGUMENT, "scheduler is NULL");
    s->updates_per_second = updates_per_second;       // water.gd:51
    s->time = 0.0;                                    // :62
    s->next_update_time = 0.0;                        // :63
    return OCEAN_OK;
}

int ocean_scheduler_set_rate(ocean_scheduler* s, double value) {                  // water.gd:52-54
    if (!s) return fail(OCEAN_ERR_INVALID_ARGUMENT, "scheduler is NULL");
    s->next_update_time = s->next_update_time - (1.0 / (s->updates_per_second + 1e-10) - 1.0 / (value + 1e-10));
    s->updates_per_second = value;
    return OCEAN_OK;
}

int ocean_scheduler_tick(ocean_scheduler* s, double delta, double* update_delta) {   // water.gd:75-82
    if (!s) {
        fail(OCEAN_ERR_INVALID_ARGUMENT, "scheduler is NULL");
        return 0;
    }
    int due = 0;
    if (s->updates_per_second == 0 || s->time >= s->next_update_time) {              // :77
        const double target_update_delta = 1.0 / (s->updates_per_second + 1e-10);    // :78
        const double ud = (s->updates_per_second == 0) ? delta : target_update_delta + (s->time - s->next_update_time);   // :79
        s->next_update_time = s->time + target_update_delta;                         // :80
        if (update_delta) *update_delta = ud;
        due = 1;                                                                     // :81 _update_water(update_delta)
    }
    s->time += delta;                                                                // :82
    return due;
}

int ocean_water_frame(ocean_generator* gen, ocean_scheduler* s, double delta, ocean_cascade_params* parameters, int count, int* did_update) {
    if (!s) return fail(OCEAN_ERR_INVALID_ARGUMENT, "scheduler is NULL");
    double ud = 0.0;
    const int due = ocean_scheduler_tick(s, delta, &ud);
    if (did_update) *did_update = due;
    if (due) {                                                                       // Water._process -> _update_water, :112-114
        const int rc = ocean_update(gen, ud, parameters, count);
        if (rc) return rc;
    }
    return ocean_process(gen, parameters, count);                                    // the child node's _process, wave_generator.gd:56-63
}

int ocean_map_scales(const ocean_cascade_params* parameters, int count, float* map_scales) {     // water.gd:102-110
    if (!parameters || !map_scales) return fail(OCEAN_ERR_INVALID_ARGUMENT, "NULL argument");
    for (int i = 0; i < count; ++i) {
        map_scales[4 * i + 0] = 1.0f / parameters[i].tile_length[0];     // Vector2.ONE / tile_length (binary32)
        map_scales[4 * i + 1] = 1.0f / parameters[i].tile_length[1];
        map_scales[4 * i + 2] = (float)parameters[i].displacement_scale;
        map_scales[4 * i + 3] = (float)parameters[i].normal_scale;
    }
    return OCEAN_OK;
}

double ocean_water_default_time(int cascade) { return 120.0 + M_PI * cascade; }                   // water.gd:32

int ocean_get_maps(ocean_generator* gen, void** displacement_dev, void** normal_dev, size_t* layer_bytes) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (displacement_dev) *displacement_dev = gen->buf.displacement;
    if (normal_dev) *normal_dev = gen->buf.normal;
    if (layer_bytes) *layer_bytes = sizeof(uint2) * (size_t)gen->map_size * gen->map_size;
    return OCEAN_OK;
}

int ocean_copy_maps_to_host_async(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (first < 0 || count < 0 || first + count > gen->num_cascades)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "layer range [%d,%d) outside [0,%d)", first, first + count, gen->num_cascades);
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    if (displacement_host)
        OCEAN_CUDA(cudaMemcpyAsync(displacement_host, gen->buf.displacement + first * layer, sizeof(uint2) * layer * count, cudaMemcpyDeviceToHost, gen->stream));
    if (normal_host)
        OCEAN_CUDA(cudaMemcpyAsync(normal_host, gen->buf.normal + first * layer, sizeof(uint2) * layer * count, cudaMemcpyDeviceToHost, gen->stream));
    return OCEAN_OK;
}

int ocean_snapshot_maps_to_host_async(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (first < 0 || count < 0 || first + count > gen->num_cascades)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "layer range [%d,%d) outside [0,%d)", first, first + count, gen->num_cascades);
    if (count == 0) return OCEAN_OK;
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    if (!gen->copy_stream) {
        OCEAN_CUDA(cudaStreamCreateWithFlags(&gen->copy_stream, cudaStreamNonBlocking));
        OCEAN_CUDA(cudaEventCreateWithFlags(&gen->snap_ready, cudaEventDisableTiming));
        OCEAN_CUDA(cudaEventCreateWithFlags(&gen->snap_free, cudaEventDisableTiming));
        OCEAN_CUDA(dev_alloc(gen, &gen->snap_disp, (size_t)gen->num_cascades * layer));
        OCEAN_CUDA(dev_alloc(gen, &gen->snap_normal, (size_t)gen->num_cascades * layer));
    }
    // the snapshot buffers are free again once the previous hand-off has left the device
    if (gen->snap_busy) OCEAN_CUDA(cudaStreamWaitEvent(gen->stream, gen->snap_free, 0));
    if (displacement_host)
        OCEAN_CUDA(cudaMemcpyAsync(gen->snap_disp + first * layer, gen->buf.displacement + first * layer, sizeof(uint2) * layer * count,
                                   cudaMemcpyDeviceToDevice, gen->stream));
    if (normal_host)
        OCEAN_CUDA(cudaMemcpyAsync(gen->snap_normal + first * layer, gen->buf.normal + first * layer, sizeof(uint2) * layer * count,
                                   cudaMemcpyDeviceToDevice, gen->stream));
    OCEAN_CUDA(cudaEventRecord(gen->snap_ready, gen->stream));
    OCEAN_CUDA(cudaStreamWaitEvent(gen->copy_stream, gen->snap_ready, 0));
    if (displacement_host)
        OCEAN_CUDA(cudaMemcpyAsync(displacement_host, gen->snap_disp + first * layer, sizeof(uint2) * layer * count, cudaMemcpyDeviceToHost,
                                   gen->copy_stream));
    if (normal_host)
        OCEAN_CUDA(cudaMemcpyAsync(normal_host, gen->snap_normal + first * layer, sizeof(uint2) * layer * count, cudaMemcpyDeviceToHost,
                                   gen->copy_stream));
    OCEAN_CUDA(cudaEventRecord(gen->snap_free, gen->copy_stream));
    gen->snap_busy = true;
    return OCEAN_OK;
}

int ocean_wait_snapshot(ocean_generator* gen) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (gen->copy_stream) OCEAN_CUDA(cudaStreamSynchronize(gen->copy_stream));
    return OCEAN_OK;
}

int ocean_copy_maps_to_host(ocean_generator* gen, int first, int count, void* displacement_host, void* normal_host) {
    int rc = ocean_copy_maps_to_host_async(gen, first, count, displacement_host, normal_host);
    if (rc) return rc;
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_synchronize(ocean_generator* gen) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return fail(OCEAN_ERR_INVALID_ARGUMENT, "ptr is NULL");
    OCEAN_CUDA(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
    return OCEAN_OK;
}
int ocean_host_free(void* ptr) {
    OCEAN_CUDA(cudaFreeHost(ptr));
    return OCEAN_OK;
}

int ocean_copy_spectrum_to_host(ocean_generator* gen, int cascade, float* host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "host is NULL");
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    OCEAN_CUDA(cudaMemcpyAsync(host, gen->buf.spectrum + cascade * layer, sizeof(float4) * layer, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_set_spectrum_amplitudes(ocean_generator* gen, int cascade, const float* amplitudes) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!amplitudes) return fail(OCEAN_ERR_INVALID_ARGUMENT, "amplitudes is NULL");
    const int N = gen->map_size;
    std::vector<float> tex((size_t)N * N * 4);
    for (int y = 0; y < N; ++y)
        for (int x = 0; x < N; ++x) {
            const int xm = (N - x) % N, ym = (N - y) % N;                          // ivec2(mod(-id0, dims)), spectrum_compute.glsl:121
            const float* a0 = amplitudes + ((size_t)y * N + x) * 2;
            const float* a1 = amplitudes + ((size_t)ym * N + xm) * 2;
            float* t = tex.data() + ((size_t)y * N + x) * 4;
            t[0] = a0[0]; t[1] = a0[1]; t[2] = a1[0]; t[3] = -a1[1];                // (h0(k), conj h0(-k))  :124
        }
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    OCEAN_CUDA(cudaMemcpy(gen->buf.spectrum + (size_t)cascade * N * N, tex.data(), sizeof(float) * tex.size(), cudaMemcpyHostToDevice));
    return OCEAN_OK;
}

int ocean_enable_f32_taps(ocean_generator* gen, int enable) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    const size_t n = (size_t)gen->num_cascades * gen->map_size * gen->map_size;
    if (enable && !gen->buf.displacement_f32) {
        OCEAN_CUDA(dev_alloc(gen, &gen->buf.displacement_f32, n));
        OCEAN_CUDA(dev_alloc(gen, &gen->buf.normal_f32, n));
        OCEAN_CUDA(cudaMemset(gen->buf.displacement_f32, 0, sizeof(float4) * n));
        OCEAN_CUDA(cudaMemset(gen->buf.normal_f32, 0, sizeof(float4) * n));
    } else if (!enable && gen->buf.displacement_f32) {
        cudaFree(gen->buf.displacement_f32);
        cudaFree(gen->buf.normal_f32);
        gen->buf.displacement_f32 = gen->buf.normal_f32 = nullptr;
        gen->device_bytes -= 2 * sizeof(float4) * n;
    }
    return OCEAN_OK;
}

int ocean_copy_f32_maps_to_host(ocean_generator* gen, int cascade, float* displacement_host, float* normal_host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!gen->buf.displacement_f32) return fail(OCEAN_ERR_STATE, "binary32 taps are disabled; call ocean_enable_f32_taps(gen, 1) first");
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    if (displacement_host)
        OCEAN_CUDA(cudaMemcpyAsync(displacement_host, gen->buf.displacement_f32 + cascade * layer, sizeof(float4) * layer, cudaMemcpyDeviceToHost, gen->stream));
    if (normal_host)
        OCEAN_CUDA(cudaMemcpyAsync(normal_host, gen->buf.normal_f32 + cascade * layer, sizeof(float4) * layer, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_copy_rowpass_to_host(ocean_generator* gen, int cascade, float* host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "host is NULL");
    // without the taps the column pass drops the scratch lines from L2 once it has consumed them (no DRAM write-back)
    if (!gen->buf.displacement_f32) return fail(OCEAN_ERR_STATE, "the row-pass scratch is only kept while the taps are on; call ocean_enable_f32_taps(gen, 1) before the update");
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    if (!gen->export_buf) OCEAN_CUDA(dev_alloc(gen, &gen->export_buf, 4 * layer));
    OCEAN_CUDA(ocean::launch_rowpass_export(gen->buf, gen->scratch_layer_of[cascade], gen->export_buf, gen->stream));
    gen->kernel_launches += 1;
    OCEAN_CUDA(cudaMemcpyAsync(host, gen->export_buf, sizeof(float2) * 4 * layer, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

float ocean_detmath_expf(float x) { return exp_det_host(x); }

int ocean_debug_work_queue(int map_size, int count, int group, int lag, int frames, int32_t* items, int capacity) {
    if (ocean::a_items_per_cascade(map_size) == 0 || count < 1 || frames < 0 || (long long)count * (frames > 0 ? frames : 1) > 0x7fff ||
        (items == nullptr && capacity > 0))
        return -fail(OCEAN_ERR_INVALID_ARGUMENT, "ocean_debug_work_queue: map_size must be 128/256/512/1024, 1 <= count * frames <= 32767");
    if (group <= 0) group = ocean::persistent_group(map_size);
    if (lag <= 0) lag = ocean::persistent_lag(map_size);
    auto build = [&](int* out) {
        return frames > 0 ? ocean::build_item_table_frames(map_size, count, frames, out) : ocean::build_item_table(map_size, count, group, lag, out);
    };
    const int total = build(nullptr);
    if (items && capacity > 0) {
        std::vector<int> all((size_t)total);
        build(all.data());
        for (int i = 0; i < total && i < capacity; ++i) items[i] = all[(size_t)i];
    }
    return total;
}

// ---- map queries (SURVEY 8f row f2) ----
namespace {
int upload_scales(ocean_generator* gen, int num_cascades, const float* map_scales_host) {
    if (num_cascades < 1 || num_cascades > gen->num_cascades)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_cascades %d outside [1, %d]", num_cascades, gen->num_cascades);
    if (!map_scales_host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "map_scales is NULL");
    if (!gen->q_scales) OCEAN_CUDA(dev_alloc(gen, &gen->q_scales, (size_t)gen->num_cascades));
    OCEAN_CUDA(cudaMemcpyAsync(gen->q_scales, map_scales_host, sizeof(float4) * (size_t)num_cascades, cudaMemcpyHostToDevice, gen->stream));
    return OCEAN_OK;
}
// Grows the query staging (points and the map query's outputs; the host entry points of every query op share it) to n points.
int reserve_query_points(ocean_generator* gen, size_t n) {
    if (n <= gen->q_capacity) return OCEAN_OK;
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    cudaFree(gen->q_points); cudaFree(gen->q_disp); cudaFree(gen->q_grad);
    gen->q_points = nullptr; gen->q_disp = gen->q_grad = nullptr; gen->q_capacity = 0;
    OCEAN_CUDA(dev_alloc(gen, &gen->q_points, n));
    OCEAN_CUDA(dev_alloc(gen, &gen->q_disp, 3 * n));
    OCEAN_CUDA(dev_alloc(gen, &gen->q_grad, 3 * n));
    gen->q_capacity = n;
    return OCEAN_OK;
}
}  // namespace

int ocean_sample_maps_device(ocean_generator* gen, int num_points, const float* points_xz_dev, int num_cascades, const float* map_scales_host,
                             float* displacement_dev, float* gradient_foam_dev) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (num_points < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_points %d is negative", num_points);
    if (num_points == 0) return OCEAN_OK;
    if (!points_xz_dev || !displacement_dev || !gradient_foam_dev) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a device buffer is NULL");
    if ((rc = upload_scales(gen, num_cascades, map_scales_host))) return rc;
    OCEAN_CUDA(ocean::launch_sample_maps(gen->buf, num_cascades, reinterpret_cast<const float2*>(points_xz_dev), num_points, gen->q_scales,
                                         displacement_dev, gradient_foam_dev, gen->stream));
    gen->kernel_launches += 1;
    return OCEAN_OK;
}

int ocean_sample_maps(ocean_generator* gen, int num_points, const float* points_xz_host, int num_cascades, const float* map_scales_host,
                      float* displacement_host, float* gradient_foam_host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (num_points < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_points %d is negative", num_points);
    if (num_points == 0) return OCEAN_OK;
    if (!points_xz_host || !displacement_host || !gradient_foam_host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a host buffer is NULL");
    const size_t n = (size_t)num_points;
    if ((rc = reserve_query_points(gen, n))) return rc;
    OCEAN_CUDA(cudaMemcpyAsync(gen->q_points, points_xz_host, sizeof(float2) * n, cudaMemcpyHostToDevice, gen->stream));
    if ((rc = ocean_sample_maps_device(gen, num_points, reinterpret_cast<const float*>(gen->q_points), num_cascades, map_scales_host,
                                       gen->q_disp, gen->q_grad)))
        return rc;
    OCEAN_CUDA(cudaMemcpyAsync(displacement_host, gen->q_disp, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaMemcpyAsync(gradient_foam_host, gen->q_grad, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

// ---- spray candidates (SURVEY 8f row f3) ----
static_assert(sizeof(ocean_spray_record) == 32, "ocean_spray_record layout");

int ocean_spray_grid(int num_particles, const float* emission_transform, float* points_xz_host) {
    if (num_particles < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_particles %d is negative", num_particles);
    if (num_particles == 0) return OCEAN_OK;
    if (!points_xz_host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "points_xz is NULL");
    static const float identity[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    const float* E = emission_transform ? emission_transform : identity;
    // sea_spray_particle.gdshader:47,52-54, binary32 with every operation rounded on its own (volatile defeats contraction)
    const unsigned t = (unsigned)std::sqrt((float)num_particles);
    if (t < 2) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_particles %d gives a grid side below 2 (division by t - 1)", num_particles);
    const float tm1 = (float)t - 1.0f;
    for (unsigned i = 0; i < (unsigned)num_particles; ++i) {
        volatile float cx = (float)(i / t) / tm1, cz = (float)(i % t) / tm1;
        cx = cx - 0.5f; cz = cz - 0.5f;
        cx = cx * 10.0f; cz = cz * 10.0f;
        for (int k = 0; k < 2; ++k) {
            const float* row = E + 4 * (k == 0 ? 0 : 2);
            volatile float a = row[0] * cx, b0 = row[1] * 0.0f, c = row[2] * cz;
            volatile float sum = a + b0;
            sum = sum + c;
            sum = sum + row[3];
            points_xz_host[2 * (size_t)i + k] = sum;
        }
    }
    return OCEAN_OK;
}

int ocean_extract_spray_device(ocean_generator* gen, int num_candidates, const float* points_xz_dev, int num_cascades,
                               const float* map_scales_host, const float* particle_scale, int max_records,
                               ocean_spray_record* records_dev, int* num_active_dev) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (num_candidates < 0 || max_records < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "negative count");
    if (!num_active_dev) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_active is NULL");
    if (num_candidates == 0) {
        OCEAN_CUDA(cudaMemsetAsync(num_active_dev, 0, sizeof(int), gen->stream));
        return OCEAN_OK;
    }
    if (!points_xz_dev || !particle_scale || (max_records > 0 && !records_dev)) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a buffer is NULL");
    if ((rc = upload_scales(gen, num_cascades, map_scales_host))) return rc;
    const int blocks = ocean::spray_blocks(num_candidates);
    if (blocks + 1 > gen->spray_count_capacity) {
        OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
        cudaFree(gen->spray_counts);
        gen->spray_counts = nullptr;
        gen->spray_count_capacity = 0;
        OCEAN_CUDA(dev_alloc(gen, &gen->spray_counts, (size_t)blocks + 1));
        gen->spray_count_capacity = blocks + 1;
    }
    OCEAN_CUDA(ocean::launch_extract_spray(gen->buf, num_cascades, reinterpret_cast<const float2*>(points_xz_dev), num_candidates, gen->q_scales,
                                           make_float3(particle_scale[0], particle_scale[1], particle_scale[2]), gen->spray_counts, records_dev,
                                           max_records, gen->stream));
    gen->kernel_launches += 3;
    OCEAN_CUDA(cudaMemcpyAsync(num_active_dev, gen->spray_counts + blocks, sizeof(int), cudaMemcpyDeviceToDevice, gen->stream));
    return OCEAN_OK;
}

int ocean_extract_spray(ocean_generator* gen, int num_candidates, const float* points_xz_host, int num_cascades,
                        const float* map_scales_host, const float* particle_scale, int max_records,
                        ocean_spray_record* records_host, int* num_active) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (num_candidates < 0 || max_records < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "negative count");
    if (!num_active) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_active is NULL");
    *num_active = 0;
    if (num_candidates == 0) return OCEAN_OK;
    if (!points_xz_host || (max_records > 0 && !records_host)) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a host buffer is NULL");
    const size_t n = (size_t)num_candidates;
    if ((rc = reserve_query_points(gen, n))) return rc;    // the candidate staging buffer is shared with the map-query op
    const size_t rec_bytes = ((size_t)max_records + 1) * sizeof(ocean_spray_record);    // + one slot for the count
    if (rec_bytes > gen->spray_record_capacity) {
        OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
        cudaFree(gen->spray_records);
        gen->spray_records = nullptr;
        gen->spray_record_capacity = 0;
        OCEAN_CUDA(cudaMalloc(&gen->spray_records, rec_bytes));
        gen->device_bytes += rec_bytes;
        gen->spray_record_capacity = rec_bytes;
    }
    ocean_spray_record* recs = static_cast<ocean_spray_record*>(gen->spray_records);
    int* count_dev = reinterpret_cast<int*>(recs + max_records);
    OCEAN_CUDA(cudaMemcpyAsync(gen->q_points, points_xz_host, sizeof(float2) * n, cudaMemcpyHostToDevice, gen->stream));
    if ((rc = ocean_extract_spray_device(gen, num_candidates, reinterpret_cast<const float*>(gen->q_points), num_cascades, map_scales_host,
                                         particle_scale, max_records, recs, count_dev)))
        return rc;
    int count = 0;
    OCEAN_CUDA(cudaMemcpyAsync(&count, count_dev, sizeof(int), cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    const int kept = count < max_records ? count : max_records;
    if (kept > 0) OCEAN_CUDA(cudaMemcpy(records_host, recs, sizeof(ocean_spray_record) * (size_t)kept, cudaMemcpyDeviceToHost));
    *num_active = count;
    return OCEAN_OK;
}

// ---- surface query: the map query above a world position, horizontal displacement inverted ----
static_assert(sizeof(ocean_surface_point) == 32, "ocean_surface_point layout");

namespace {
int check_surface_args(int num_points, int iterations) {
    if (num_points < 0) return fail(OCEAN_ERR_INVALID_ARGUMENT, "num_points %d is negative", num_points);
    if (iterations < 0 || iterations > OCEAN_SURFACE_MAX_ITERATIONS)
        return fail(OCEAN_ERR_INVALID_ARGUMENT, "iterations %d outside [0, %d]", iterations, OCEAN_SURFACE_MAX_ITERATIONS);
    return OCEAN_OK;
}
}  // namespace

int ocean_query_surface_device(ocean_generator* gen, int num_points, const float* points_xz_dev, int num_cascades, const float* map_scales_host,
                               int iterations, ocean_surface_point* out_dev) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_surface_args(num_points, iterations))) return rc;
    if (num_points == 0) return OCEAN_OK;
    if (!points_xz_dev || !out_dev) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a device buffer is NULL");
    if ((rc = upload_scales(gen, num_cascades, map_scales_host))) return rc;
    OCEAN_CUDA(ocean::launch_query_surface(gen->buf, num_cascades, reinterpret_cast<const float2*>(points_xz_dev), num_points, gen->q_scales,
                                           iterations, out_dev, gen->stream));
    gen->kernel_launches += 1;
    return OCEAN_OK;
}

int ocean_query_surface(ocean_generator* gen, int num_points, const float* points_xz_host, int num_cascades, const float* map_scales_host,
                        int iterations, ocean_surface_point* out_host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_surface_args(num_points, iterations))) return rc;
    if (num_points == 0) return OCEAN_OK;
    if (!points_xz_host || !out_host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "a host buffer is NULL");
    const size_t n = (size_t)num_points;
    if ((rc = reserve_query_points(gen, n))) return rc;
    const size_t out_bytes = n * sizeof(ocean_surface_point);
    if (out_bytes > gen->surface_point_capacity) {
        OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
        cudaFree(gen->surface_points);
        gen->device_bytes -= gen->surface_point_capacity;
        gen->surface_points = nullptr;
        gen->surface_point_capacity = 0;
        OCEAN_CUDA(cudaMalloc(&gen->surface_points, out_bytes));
        gen->device_bytes += out_bytes;
        gen->surface_point_capacity = out_bytes;
    }
    ocean_surface_point* out_dev = static_cast<ocean_surface_point*>(gen->surface_points);
    OCEAN_CUDA(cudaMemcpyAsync(gen->q_points, points_xz_host, sizeof(float2) * n, cudaMemcpyHostToDevice, gen->stream));
    if ((rc = ocean_query_surface_device(gen, num_points, reinterpret_cast<const float*>(gen->q_points), num_cascades, map_scales_host,
                                         iterations, out_dev)))
        return rc;
    OCEAN_CUDA(cudaMemcpyAsync(out_host, out_dev, out_bytes, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_copy_twiddles_to_host(ocean_generator* gen, float* host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (!host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "host is NULL");
    OCEAN_CUDA(cudaMemcpyAsync(host, gen->twiddles, sizeof(float2) * (gen->map_size - 1), cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_get_foam_state(ocean_generator* gen, int cascade, uint16_t* host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "host is NULL");
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    const uint16_t* src = reinterpret_cast<const uint16_t*>(gen->buf.normal + cascade * layer) + 3;
    OCEAN_CUDA(cudaMemcpy2DAsync(host, sizeof(uint16_t), src, sizeof(uint2), sizeof(uint16_t), layer, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_set_foam_state(ocean_generator* gen, int cascade, const uint16_t* host) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if ((rc = check_cascade(gen, cascade))) return rc;
    if (!host) return fail(OCEAN_ERR_INVALID_ARGUMENT, "host is NULL");
    const size_t layer = (size_t)gen->map_size * gen->map_size;
    uint16_t* dst = reinterpret_cast<uint16_t*>(gen->buf.normal + cascade * layer) + 3;
    OCEAN_CUDA(cudaMemcpy2DAsync(dst, sizeof(uint2), host, sizeof(uint16_t), sizeof(uint16_t), layer, cudaMemcpyHostToDevice, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    return OCEAN_OK;
}

int ocean_timer_start(ocean_generator* gen) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    OCEAN_CUDA(cudaEventRecord(gen->timer_start, gen->stream));
    return OCEAN_OK;
}

int ocean_timer_stop(ocean_generator* gen, float* elapsed_ms) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (!elapsed_ms) return fail(OCEAN_ERR_INVALID_ARGUMENT, "elapsed_ms is NULL");
    OCEAN_CUDA(cudaEventRecord(gen->timer_stop, gen->stream));
    OCEAN_CUDA(cudaEventSynchronize(gen->timer_stop));
    OCEAN_CUDA(cudaEventElapsedTime(elapsed_ms, gen->timer_start, gen->timer_stop));
    return OCEAN_OK;
}

int ocean_set_profiling(ocean_generator* gen, int enable) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    gen->profiling = enable != 0;
    gen->prof_valid = false;
    return OCEAN_OK;
}

int ocean_get_last_kernel_times(ocean_generator* gen, float* spectrum_ms, float* rowpass_ms, float* colpass_ms, int* chunk_cascades) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (!gen->prof_valid) return fail(OCEAN_ERR_STATE, "no profiled launch yet; call ocean_set_profiling(gen, 1) and run an update");
    OCEAN_CUDA(cudaEventSynchronize(gen->prof[3]));
    float t = 0.f;
    if (spectrum_ms) { OCEAN_CUDA(cudaEventElapsedTime(&t, gen->prof[0], gen->prof[1])); *spectrum_ms = gen->prof_had_gen ? t : 0.f; }
    if (rowpass_ms) OCEAN_CUDA(cudaEventElapsedTime(rowpass_ms, gen->prof[1], gen->prof[2]));
    if (colpass_ms) OCEAN_CUDA(cudaEventElapsedTime(colpass_ms, gen->prof[2], gen->prof[4]));
    if (chunk_cascades) *chunk_cascades = gen->prof_chunk;
    return OCEAN_OK;
}

int ocean_selftest_math(ocean_generator* gen, uint64_t* failures, uint64_t* tested) {
    OCEAN_ENTER(gen);
    if (rc) return rc;
    if (!failures || !tested) return fail(OCEAN_ERR_INVALID_ARGUMENT, "NULL argument");
    unsigned long long* d = nullptr;
    OCEAN_CUDA(cudaMalloc(reinterpret_cast<void**>(&d), 2 * sizeof(unsigned long long)));
    OCEAN_CUDA(cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), gen->stream));
    OCEAN_CUDA(ocean::launch_selftest_math(d, d + 1, gen->stream));
    gen->kernel_launches += 1;
    unsigned long long h[2] = {0, 0};
    OCEAN_CUDA(cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, gen->stream));
    OCEAN_CUDA(cudaStreamSynchronize(gen->stream));
    cudaFree(d);
    *failures = h[0];
    *tested = h[1];
    return OCEAN_OK;
}

int ocean_get_info(ocean_generator* gen, ocean_info* out) {
    if (!gen || !out) return fail(OCEAN_ERR_INVALID_ARGUMENT, "NULL argument");
    out->device = gen->device;
    out->map_size = gen->map_size;
    out->num_cascades = gen->num_cascades;
    out->pending_cascades = gen->pass_num_cascades_remaining;
    out->kernel_launches = gen->kernel_launches;
    out->cascade_updates = gen->cascade_updates;
    out->device_bytes = gen->device_bytes;
    return OCEAN_OK;
}

}  // extern "C"
