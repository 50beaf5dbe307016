// OceanNative.cs -- P/Invoke binding of libocean.so (include/ocean.h) and a WaveGenerator-shaped host class.
//
// NOT COMPILED IN THIS REPOSITORY'S CI: the build image has no dotnet/mono/csc.  The ABI is exercised through
// the Python ctypes mirror (godotoceanwaves_b200/native.py) and tests/test_abi_cpu.py instead; this file shows the
// binding a Godot C# project would add.  Convention follows the one in-tree P/Invoke precedent of the reference,
// addons/imgui-godot/ImGuiGodot/Internal/Viewports.cs:157-165 ([LibraryImport], cdecl, unsafe partial).
//
// Replaces: assets/water/wave_generator.gd (WaveGenerator node) and, below it, every RenderingContext call of
// assets/render_context.gd:35-135 that the generator makes.  The two RGBA16F layered maps are handed to Godot with
// RenderingDevice.TextureUpdate(rid, layer, bytes), which the reference's textures already allow
// (TEXTURE_USAGE_CAN_UPDATE_BIT, wave_generator.gd:34-35).
using System;
using System.Runtime.InteropServices;

namespace OceanB200
{
    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct OceanCascadeParams            // struct ocean_cascade_params <- wave_cascade_parameters.gd:2-42
    {
        public fixed float tile_length[2];
        public double displacement_scale, normal_scale;
        public double wind_speed, wind_direction, fetch_length, swell, spread, detail, whitecap, foam_amount;
        public fixed int spectrum_seed[2];
        public int should_generate_spectrum;
        public double time, foam_grow_rate, foam_decay_rate;
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct OceanScheduler                                    // struct ocean_scheduler <- water.gd:51,62-63
    {
        public double updates_per_second, time, next_update_time;
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct OceanSprayRecord                           // struct ocean_spray_record <- sea_spray_particle.gdshader:80-94
    {
        public uint index;
        public float start_x, start_z, scale_factor;
        public fixed float particle_scale[3];
        public float foam;
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct OceanSurfacePoint                          // struct ocean_surface_point (32 B) <- water.gdshader:31-37 inverted
    {
        public float height;                                        // surface height above the query point
        public float source_x, source_z;                            // undisplaced position whose vertex lands over the query point
        public float residual;                                      // |source + D.xz(source) - q|, metres
        public fixed float gradient_foam[3];                        // ocean_sample_maps' gradient/foam at the source point
        public float jacobian;                                      // <= 0: folded surface
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct OceanInfo
    {
        public int device, map_size, num_cascades, pending_cascades;
        public ulong kernel_launches, cascade_updates, device_bytes;
    }

    internal static unsafe partial class Native
    {
        private const string Lib = "ocean";           // libocean.so next to the Godot binary / in LD_LIBRARY_PATH

        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_default_cascade_params(OceanCascadeParams* p);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_create(int device, int map_size, int num_cascades, IntPtr* handle);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_destroy(IntPtr handle);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_update(IntPtr handle, double delta, OceanCascadeParams* parameters, int count);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_process(IntPtr handle, OceanCascadeParams* parameters, int count);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_update_all(IntPtr handle, double delta, OceanCascadeParams* parameters, int count);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_get_maps(IntPtr handle, IntPtr* displacement_dev, IntPtr* normal_dev, nuint* layer_bytes);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_copy_maps_to_host(IntPtr handle, int first, int count, void* displacement, void* normal);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_copy_maps_to_host_async(IntPtr handle, int first, int count, void* displacement, void* normal);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_synchronize(IntPtr handle);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_host_alloc(void** ptr, nuint bytes);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_host_free(void* ptr);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_get_foam_state(IntPtr handle, int cascade, ushort* host);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_set_foam_state(IntPtr handle, int cascade, ushort* host);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial double ocean_jonswap_alpha(double wind_speed, double fetch_length);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial double ocean_jonswap_peak_angular_frequency(double wind_speed, double fetch_length);
        // map queries (water.gdshader:27-39,42-84): points [n][2] world x,z; map_scales [c][4]; outputs [n][3]
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_sample_maps(IntPtr handle, int num_points, float* points_xz, int num_cascades, float* map_scales,
                                                      float* displacement, float* gradient_foam);
        // surface query: the map query above world x,z with the horizontal displacement inverted; iterations in [0, 32], 8 = default.
        // The _device form takes device pointers for points and records and is asynchronous on the generator's stream.
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_query_surface(IntPtr handle, int num_points, float* points_xz, int num_cascades, float* map_scales,
                                                        int iterations, OceanSurfacePoint* points_out);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_query_surface_device(IntPtr handle, int num_points, float* points_xz_dev, int num_cascades,
                                                               float* map_scales, int iterations, OceanSurfacePoint* points_out_dev);
        // fused frames, overlapped hand-off, Water scheduler, spray candidates (include/ocean.h)
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_update_frames(IntPtr handle, double delta, OceanCascadeParams* parameters, int count, int frames);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_snapshot_maps_to_host_async(IntPtr handle, int first, int count, void* displacement, void* normal);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_wait_snapshot(IntPtr handle);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_scheduler_init(OceanScheduler* s, double updates_per_second);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_scheduler_set_rate(OceanScheduler* s, double updates_per_second);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_scheduler_tick(OceanScheduler* s, double delta, double* update_delta);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_water_frame(IntPtr handle, OceanScheduler* s, double delta, OceanCascadeParams* parameters, int count, int* did_update);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_map_scales(OceanCascadeParams* parameters, int count, float* map_scales);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial double ocean_water_default_time(int cascade);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_spray_grid(int num_particles, float* emission_transform, float* points_xz);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_extract_spray(IntPtr handle, int num_candidates, float* points_xz, int num_cascades, float* map_scales,
                                                        float* particle_scale, int max_records, OceanSprayRecord* records, int* num_active);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial int ocean_get_info(IntPtr handle, OceanInfo* info);
        [LibraryImport(Lib)] [UnmanagedCallConv(CallConvs = new[] { typeof(System.Runtime.CompilerServices.CallConvCdecl) })]
        internal static partial IntPtr ocean_last_error();
    }

    public sealed class OceanException : Exception { public OceanException(string m) : base(m) { } }

    /// <summary>Same surface as the reference's WaveGenerator (assets/water/wave_generator.gd): MapSize, InitGpu,
    /// Update, Process, the two maps and the static JONSWAP helpers.</summary>
    public sealed unsafe class WaveGenerator : IDisposable
    {
        public const double G = 9.81, Depth = 20.0;               // wave_generator.gd:5-6
        public int MapSize;                                         // wave_generator.gd:8
        private IntPtr _handle;
        private int _layers;
        private byte* _dispHost, _normHost;                         // pinned staging for texture_update

        private static void Check(int status)
        {
            if (status != 0) throw new OceanException(Marshal.PtrToStringAnsi(Native.ocean_last_error()) ?? "libocean error");
        }

        public void InitGpu(int numCascades, int device = 0)        // wave_generator.gd:17-54
        {
            Dispose();
            IntPtr h;
            Check(Native.ocean_create(device, MapSize, numCascades, &h));
            _handle = h; _layers = numCascades;
            nuint bytes = (nuint)numCascades * (nuint)MapSize * (nuint)MapSize * 8;
            void* d, n;
            Check(Native.ocean_host_alloc(&d, bytes)); Check(Native.ocean_host_alloc(&n, bytes));
            _dispHost = (byte*)d; _normHost = (byte*)n;
        }

        public void Update(double delta, Span<OceanCascadeParams> parameters)   // wave_generator.gd:90-109
        {
            if (parameters.Length == 0) throw new ArgumentException("parameters.size() != 0");
            if (_handle == IntPtr.Zero) InitGpu(Math.Max(2, parameters.Length));
            fixed (OceanCascadeParams* p = parameters) Check(Native.ocean_update(_handle, delta, p, parameters.Length));
        }

        public void Process(Span<OceanCascadeParams> parameters)                 // wave_generator.gd:56-63 (_process)
        {
            fixed (OceanCascadeParams* p = parameters) Check(Native.ocean_process(_handle, p, parameters.Length));
        }

        /// <summary>Copies layer `cascade` of both maps to pinned host memory; the caller passes the spans to
        /// RenderingDevice.TextureUpdate(displacementRid, cascade, bytes) / (normalRid, cascade, bytes).</summary>
        public (IntPtr displacement, IntPtr normal, int bytes) FetchLayer(int cascade)
        {
            int layer = MapSize * MapSize * 8;
            Check(Native.ocean_copy_maps_to_host(_handle, cascade, 1, _dispHost + (long)cascade * layer, _normHost + (long)cascade * layer));
            return ((IntPtr)(_dispHost + (long)cascade * layer), (IntPtr)(_normHost + (long)cascade * layer), layer);
        }

        internal IntPtr Handle => _handle;
        internal byte* DisplacementHost => _dispHost;
        internal byte* NormalHost => _normHost;

        public static double JONSWAPAlpha(double windSpeed = 20.0, double fetchLength = 550e3) => Native.ocean_jonswap_alpha(windSpeed, fetchLength);
        public static double JONSWAPPeakAngularFrequency(double windSpeed = 20.0, double fetchLength = 550e3) => Native.ocean_jonswap_peak_angular_frequency(windSpeed, fetchLength);

        public void Dispose()                                       // NOTIFICATION_PREDELETE, wave_generator.gd:111-113
        {
            if (_handle != IntPtr.Zero) { Native.ocean_destroy(_handle); _handle = IntPtr.Zero; }
            if (_dispHost != null) { Native.ocean_host_free(_dispHost); _dispHost = null; }
            if (_normHost != null) { Native.ocean_host_free(_normHost); _normHost = null; }
        }
    }

    /// <summary>The wave side of the reference's Water node (assets/water/water.gd): owns the generator, runs the fixed-rate
    /// update accumulator (:75-82, in the library: ocean_scheduler_tick), gives every cascade its start time (:32), builds
    /// map_scales (:102-110) and hands finished layers to Godot.  In a Godot C# project this class derives from MeshInstance3D
    /// and _Process(delta) calls Frame(delta); the TextureUpdate calls are the only engine API it needs.</summary>
    public sealed unsafe class Water : IDisposable
    {
        public readonly WaveGenerator Generator = new WaveGenerator();
        private OceanScheduler _sched;
        private OceanCascadeParams[] _parameters = Array.Empty<OceanCascadeParams>();

        public Water(int mapSize = 1024, double updatesPerSecond = 50.0)           // water.gd:38,51
        {
            Generator.MapSize = mapSize;
            fixed (OceanScheduler* s = &_sched) Native.ocean_scheduler_init(s, updatesPerSecond);
        }

        public double UpdatesPerSecond                                             // water.gd:51-54
        {
            get => _sched.updates_per_second;
            set { fixed (OceanScheduler* s = &_sched) Native.ocean_scheduler_set_rate(s, value); }
        }

        public void SetParameters(OceanCascadeParams[] value)                      // water.gd:22-35,84-100
        {
            for (int i = 0; i < value.Length; ++i)
            {
                value[i].time = Native.ocean_water_default_time(i);                // :32
                value[i].should_generate_spectrum = 1;                             // :86-87
            }
            _parameters = value;
            Generator.InitGpu(Math.Max(2, value.Length));                          // :91
        }

        public float[] MapScales()                                                 // water.gd:102-110
        {
            var scales = new float[4 * _parameters.Length];
            fixed (OceanCascadeParams* p = _parameters) fixed (float* o = scales) Native.ocean_map_scales(p, _parameters.Length, o);
            return scales;
        }

        /// <summary>One rendered frame: Water._process (:75-82) + the child generator's _process (wave_generator.gd:56-63).
        /// `upload(rid-selector, layer, pointer, bytes)` is RenderingDevice.TextureUpdate on the displacement / normal array.</summary>
        public bool Frame(double delta, Action<bool, int, IntPtr, int> upload)
        {
            int did = 0;
            fixed (OceanScheduler* s = &_sched) fixed (OceanCascadeParams* p = _parameters)
            {
                int before = PendingCascades();
                int rc = Native.ocean_water_frame(Generator.Handle, s, delta, p, _parameters.Length, &did);
                if (rc != 0) throw new OceanException(Marshal.PtrToStringAnsi(Native.ocean_last_error()) ?? "libocean error");
                // the cascade that was just processed is the one to re-upload (highest pending index first, wave_generator.gd:59)
                int after = PendingCascades();
                if (after < before || did != 0)
                {
                    int layer = after;
                    var (d, n, bytes) = Generator.FetchLayer(layer);
                    upload(true, layer, d, bytes);
                    upload(false, layer, n, bytes);
                }
            }
            return did != 0;
        }

        private int PendingCascades()
        {
            OceanInfo info;
            Native.ocean_get_info(Generator.Handle, &info);
            return info.pending_cascades;
        }

        public void Dispose() => Generator.Dispose();                              // water.gd:116-119
    }
}
