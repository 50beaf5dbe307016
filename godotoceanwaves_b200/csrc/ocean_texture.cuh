// ocean_texture.cuh -- texture() of the reference's spatial shaders on the generator's RGBA16F maps: exact-weight bilinear
// filter with REPEAT addressing, binary32, round to nearest, no contraction (oracle/sampling.py is the specification).
// Shared by the map-query op (ocean_sample.cu), the spray-candidate op (ocean_spray.cu) and the surface query
// (ocean_surface.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace ocean {
namespace {

__device__ __forceinline__ float4 texel(const uint2* __restrict__ layer, int N, int x, int y) {
    const uint2 t = __ldg(&layer[(size_t)y * N + x]);
    const __half2 lo = *reinterpret_cast<const __half2*>(&t.x), hi = *reinterpret_cast<const __half2*>(&t.y);
    const float2 a = __half22float2(lo), b = __half22float2(hi);
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float mixf(float a, float b, float t) { return a * (1.0f - t) + b * t; }   // GLSL mix
__device__ __forceinline__ float4 mix4(const float4 a, const float4 b, float t) {
    return make_float4(mixf(a.x, b.x, t), mixf(a.y, b.y, t), mixf(a.z, b.z, t), mixf(a.w, b.w, t));
}

// The four texels texture() filters at (u, v) and their weights (oracle/surface.py texel_quad).
struct TexelQuad {
    float4 t00, t10, t01, t11;
    float fx, fy;
};
// N is a power of two (128..1024), so the REPEAT wrap is a mask.
__device__ __forceinline__ TexelQuad texel_quad(const uint2* __restrict__ layer, int N, float u, float v) {
    const float n = (float)N;
    const float x = u * n - 0.5f, y = v * n - 0.5f;
    const float x0 = floorf(x), y0 = floorf(y);
    TexelQuad q;
    q.fx = x - x0;
    q.fy = y - y0;
    const int ix0 = (int)(long long)x0 & (N - 1), iy0 = (int)(long long)y0 & (N - 1);
    const int ix1 = (ix0 + 1) & (N - 1), iy1 = (iy0 + 1) & (N - 1);
    q.t00 = texel(layer, N, ix0, iy0);
    q.t10 = texel(layer, N, ix1, iy0);
    q.t01 = texel(layer, N, ix0, iy1);
    q.t11 = texel(layer, N, ix1, iy1);
    return q;
}

// texture(): bilinear, REPEAT.
__device__ __forceinline__ float4 texture_bilinear(const uint2* __restrict__ layer, int N, float u, float v) {
    const TexelQuad q = texel_quad(layer, N, u, v);
    return mix4(mix4(q.t00, q.t10, q.fx), mix4(q.t01, q.t11, q.fx), q.fy);
}

// water.gdshader:42-51
__device__ __forceinline__ void cubic_weights(float a, float (&w)[4]) {
    const float a2 = a * a, a3 = a2 * a;
    w[0] = (-a3 + a2 * 3.0f - a * 3.0f + 1.0f) / 6.0f;
    w[1] = (a3 * 3.0f - a2 * 6.0f + 4.0f) / 6.0f;
    w[2] = (-a3 * 3.0f + a2 * 3.0f + a * 3.0f + 1.0f) / 6.0f;
    w[3] = a3 / 6.0f;
}

// water.gdshader:55-70
__device__ __forceinline__ float4 texture_bicubic(const uint2* __restrict__ layer, int N, float u, float v) {
    const float dims = (float)N, dims_inv = 1.0f / dims;
    const float ux = u * dims + 0.5f, vy = v * dims + 0.5f;
    const float flx = floorf(ux), fly = floorf(vy);
    float wx[4], wy[4];
    cubic_weights(ux - flx, wx);
    cubic_weights(vy - fly, wy);
    const float gx = wx[0] + wx[1], gy = wx[2] + wx[3], gz = wy[0] + wy[1], gw = wy[2] + wy[3];
    const float hx = (wx[1] / gx + -1.5f + flx) * dims_inv;
    const float hy = (wx[3] / gy + 0.5f + flx) * dims_inv;
    const float hz = (wy[1] / gz + -1.5f + fly) * dims_inv;
    const float hw = (wy[3] / gw + 0.5f + fly) * dims_inv;
    const float wxx = gx / (gx + gy), wyy = gz / (gz + gw);
    return mix4(mix4(texture_bilinear(layer, N, hy, hw), texture_bilinear(layer, N, hx, hw), wxx),
                mix4(texture_bilinear(layer, N, hy, hz), texture_bilinear(layer, N, hx, hz), wxx), wyy);
}

// water.gdshader:80,83: the normal-map read of one cascade, bicubic blended towards bilinear by the texel density
// ppm = map_size * min(scales.x, scales.y); the caller sums .xyw * vec3(scales.ww, 1).
__device__ __forceinline__ float4 normal_sample(const uint2* __restrict__ layer, int N, float4 s, float u, float v) {
    const float ppm = (float)N * fminf(s.x, s.y);
    const float t = fminf(1.0f, ppm * 0.1f);
    return mix4(texture_bicubic(layer, N, u, v), texture_bilinear(layer, N, u, v), t);
}

}  // namespace
}  // namespace ocean
