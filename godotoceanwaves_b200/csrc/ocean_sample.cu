// ocean_sample.cu -- batched map queries: the sampling contract of the reference's water shader as a CUDA op
// (SURVEY 8f row f2; what buoyancy / gameplay code and the spray emitter need from the generator's outputs).
//
// Reference: assets/shaders/spatial/water.gdshader
//   vertex()   :27-39   displacement(UV) = sum_i texture(displacements, vec3(UV*scales_i.xy, i)).xyz * scales_i.z
//   cubic_weights / texture_bicubic :42-70
//   fragment() :72-84   gradient/foam(UV) = sum_i mix(texture_bicubic(normals, c_i), texture(normals, c_i),
//                                                       min(1, ppm_i*0.1)).xyw * vec3(scales_i.ww, 1)
// with map_scales[i] = (1/tile_length.x, 1/tile_length.y, displacement_scale, normal_scale), water.gd:102-110.
//
// Numeric policy (oracle/sampling.py is the specification): binary32, round to nearest, the shader's operation order,
// no contraction (-fmad=false); texture() = exact-weight bilinear filter with REPEAT addressing on the RGBA16F texels.
// One thread per query point; the texel gathers are 8 B reads served by L2 (the maps of a frame are L2-resident for
// N <= 1024 x 8 cascades = 128 MiB only partly -- the op is sector-bound, see DESIGN.md).
#include "ocean_kernels.cuh"
#include "ocean_texture.cuh"

namespace ocean {

namespace {

__global__ void __launch_bounds__(256) k_sample_maps(const uint2* __restrict__ displacement, const uint2* __restrict__ normal, int N, int C,
                                                     const float2* __restrict__ points, int n, const float4* __restrict__ scales,
                                                     float* __restrict__ disp_out, float* __restrict__ grad_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 p = points[i];
    float dx = 0.0f, dy = 0.0f, dz = 0.0f, gx = 0.0f, gy = 0.0f, gf = 0.0f;
    for (int c = 0; c < C; ++c) {
        const float4 s = __ldg(&scales[c]);
        const float u = p.x * s.x, v = p.y * s.y;
        const size_t layer = (size_t)c * N * N;
        const float4 d = texture_bilinear(displacement + layer, N, u, v);                         // :34-35
        dx = dx + d.x * s.z;
        dy = dy + d.y * s.z;
        dz = dz + d.z * s.z;
        const float4 m = normal_sample(normal + layer, N, s, u, v);                               // :80-83
        gx = gx + m.x * s.w;
        gy = gy + m.y * s.w;
        gf = gf + m.w * 1.0f;
    }
    disp_out[3 * (size_t)i + 0] = dx;
    disp_out[3 * (size_t)i + 1] = dy;
    disp_out[3 * (size_t)i + 2] = dz;
    grad_out[3 * (size_t)i + 0] = gx;
    grad_out[3 * (size_t)i + 1] = gy;
    grad_out[3 * (size_t)i + 2] = gf;
}

}  // namespace

cudaError_t launch_sample_maps(const DeviceBuffers& b, int num_cascades, const float2* points_dev, int n, const float4* scales_dev,
                               float* disp_out_dev, float* grad_out_dev, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    k_sample_maps<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(b.displacement, b.normal, b.map_size, num_cascades, points_dev, n, scales_dev,
                                                                  disp_out_dev, grad_out_dev);
    return cudaGetLastError();
}

}  // namespace ocean
