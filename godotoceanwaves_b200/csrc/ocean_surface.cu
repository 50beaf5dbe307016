// ocean_surface.cu -- the surface query: water height, normal and foam ABOVE a world position, with the choppy horizontal
// displacement of the water shader inverted (include/ocean.h, ocean_query_surface).
//
// Reference: assets/shaders/spatial/water.gdshader
//   vertex() :27-39   VERTEX += displacement(VERTEX.xz): a texel's displacement moves its vertex sideways as well as up, so
//                     the surface point above q comes from the undisplaced p with p + D.xz(p) = q; its height is D.y(p)
//   fragment() :72-84 the gradient/foam read at p (the sample op's normal read)
// Solver (oracle/surface.py is the specification and fixes every operation's order): p_0 = q, then K damped Newton steps
// on the exact Jacobian of the bilinear interpolant, which reads the same four texels per cascade as D does -- the step
// falls back to the fixed-point step r where det J <= 0.05 (folds, NaN) and is clamped to twice the residual's length.
// No early exit: the iteration count is fixed, results are deterministic and bit-identical to the specification.
//
// One thread per point; p, D and J stay in registers.  Texel gathers per point: 4 C per step (8 B each, shared between D
// and J), then 4 C (displacement + Jacobian) + 20 C (normal: bilinear + four-tap bicubic) for the final evaluation at p_K,
// i.e. 4 C (K + 1) + 20 C in all.  Numeric policy as ocean_sample.cu: binary32, round to nearest, -fmad=false.
#include "ocean_kernels.cuh"
#include "ocean_texture.cuh"

namespace ocean {

namespace {

struct DisplacementJacobian {
    float dx, dy, dz;             // D = sum_i texture(displacements, p * s_i.xy, i).xyz * s_i.z
    float jxx, jxz, jzx, jzz;     // dDx/dx, dDx/dz, dDz/dx, dDz/dz of the bilinear interpolant
};

__device__ __forceinline__ DisplacementJacobian displacement_jacobian(const uint2* __restrict__ displacement, int N, int C,
                                                                      const float4* __restrict__ scales, float px, float pz) {
    DisplacementJacobian r{0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    const float n = (float)N;
    for (int c = 0; c < C; ++c) {
        const float4 s = __ldg(&scales[c]);
        const TexelQuad t = texel_quad(displacement + (size_t)c * N * N, N, px * s.x, pz * s.y);
        const float4 d = mix4(mix4(t.t00, t.t10, t.fx), mix4(t.t01, t.t11, t.fx), t.fy);     // texture_bilinear
        r.dx = r.dx + d.x * s.z;
        r.dy = r.dy + d.y * s.z;
        r.dz = r.dz + d.z * s.z;
        const float gx = (s.x * n) * s.z, gz = (s.y * n) * s.z;                                // d(texel coordinate)/dx * scale
        const float exx = mixf(t.t10.x - t.t00.x, t.t11.x - t.t01.x, t.fy), exz = mixf(t.t10.z - t.t00.z, t.t11.z - t.t01.z, t.fy);
        const float ezx = mixf(t.t01.x - t.t00.x, t.t11.x - t.t10.x, t.fx), ezz = mixf(t.t01.z - t.t00.z, t.t11.z - t.t10.z, t.fx);
        r.jxx = r.jxx + exx * gx;
        r.jzx = r.jzx + exz * gx;
        r.jxz = r.jxz + ezx * gz;
        r.jzz = r.jzz + ezz * gz;
    }
    return r;
}

struct SurfacePoint {       // == ocean_surface_point (include/ocean.h), 32 bytes
    float height, source_x, source_z, residual;
    float gradient_foam[3];
    float jacobian;
};

__global__ void __launch_bounds__(256) k_query_surface(const uint2* __restrict__ displacement, const uint2* __restrict__ normal, int N, int C,
                                                       const float2* __restrict__ points, int n, const float4* __restrict__ scales,
                                                       int iterations, SurfacePoint* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 q = points[i];
    float px = q.x, pz = q.y;
    for (int k = 0; k < iterations; ++k) {
        const DisplacementJacobian J = displacement_jacobian(displacement, N, C, scales, px, pz);
        const float rx = (px + J.dx) - q.x, rz = (pz + J.dz) - q.y;
        const float a = 1.0f + J.jxx, d = 1.0f + J.jzz;
        const float det = a * d - J.jxz * J.jzx;
        float sx = rx, sz = rz;                                                                // fixed-point step
        if (det > 0.05f) {                                                                     // Newton step J^-1 r
            sx = __fdiv_rn(d * rx - J.jxz * rz, det);
            sz = __fdiv_rn(a * rz - J.jzx * rx, det);
        }
        const float rn = __fsqrt_rn(rx * rx + rz * rz), sn = __fsqrt_rn(sx * sx + sz * sz);
        const float lim = 2.0f * rn;
        if (sn > lim) {
            const float f = __fdiv_rn(lim, sn);
            sx = sx * f;
            sz = sz * f;
        }
        px = px - sx;
        pz = pz - sz;
    }
    const DisplacementJacobian J = displacement_jacobian(displacement, N, C, scales, px, pz);
    const float rx = (px + J.dx) - q.x, rz = (pz + J.dz) - q.y;
    const float a = 1.0f + J.jxx, d = 1.0f + J.jzz;
    float gx = 0.0f, gy = 0.0f, gf = 0.0f;
    for (int c = 0; c < C; ++c) {                                                              // the sample op's normal read at p
        const float4 s = __ldg(&scales[c]);
        const float4 m = normal_sample(normal + (size_t)c * N * N, N, s, px * s.x, pz * s.y);
        gx = gx + m.x * s.w;
        gy = gy + m.y * s.w;
        gf = gf + m.w * 1.0f;
    }
    SurfacePoint r;
    r.height = J.dy;
    r.source_x = px;
    r.source_z = pz;
    r.residual = __fsqrt_rn(rx * rx + rz * rz);
    r.gradient_foam[0] = gx;
    r.gradient_foam[1] = gy;
    r.gradient_foam[2] = gf;
    r.jacobian = a * d - J.jxz * J.jzx;
    out[i] = r;
}

}  // namespace

cudaError_t launch_query_surface(const DeviceBuffers& b, int num_cascades, const float2* points_dev, int n, const float4* scales_dev,
                                 int iterations, void* out_dev, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    k_query_surface<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(b.displacement, b.normal, b.map_size, num_cascades, points_dev, n,
                                                                    scales_dev, iterations, static_cast<SurfacePoint*>(out_dev));
    return cudaGetLastError();
}

}  // namespace ocean
