"""CPU specification of the surface query: the water height, normal and foam ABOVE a world position, with the choppy
horizontal displacement of the water shader inverted (include/ocean.h, ocean_query_surface).

TEST INFRASTRUCTURE ONLY -- the product path (godotoceanwaves_b200/csrc) never imports or calls this module.

The water shader moves every vertex sideways as well as up (water.gdshader:31-37, VERTEX += displacement), so the surface
point above q comes from the undisplaced position p that solves
    p + D.xz(p) = q,   D(p) = sum_i texture(displacements, p * scales_i.xy, i).xyz * scales_i.z,
and its height is D.y(p).  Solver: a fixed number K of damped Newton steps from p_0 = q on the exact Jacobian of the
bilinear interpolant (the derivative reads the same four texels as D, so it costs no extra gathers):

  per cascade i (u = p.x*s.x, v = p.z*s.y; texel quad t00, t10, t01, t11 and weights fx, fy exactly as
  sampling.texture_bilinear picks them):
      d   = mix(mix(t00, t10, fx), mix(t01, t11, fx), fy)            (== sampling.texture_bilinear)
      Dx  = Dx + d.x * s.z;   Dz = Dz + d.z * s.z                      (cascade order, as sampling.sample_maps sums)
      gx  = (s.x * N) * s.z;  gz = (s.y * N) * s.z
      ex  = mix(t10 - t00, t11 - t01, fy);   ez = mix(t01 - t00, t11 - t10, fx)
      Jxx = Jxx + ex.x * gx;  Jzx = Jzx + ex.z * gx;  Jxz = Jxz + ez.x * gz;  Jzz = Jzz + ez.z * gz
  then (every operation binary32, round to nearest, in this order, no contraction):
      rx = (p.x + Dx) - q.x;  rz = (p.z + Dz) - q.z
      a = 1 + Jxx;  d = 1 + Jzz;  det = a*d - Jxz*Jzx
      det > 0.05 (false for NaN):  sx = (d*rx - Jxz*rz) / det;  sz = (a*rz - Jzx*rx) / det      Newton step J^-1 r
      otherwise:                   sx = rx;  sz = rz                                            fixed-point step
      rn = sqrt(rx*rx + rz*rz);  sn = sqrt(sx*sx + sz*sz);  lim = 2 * rn                        (sqrt, / correctly rounded)
      sn > lim:                    f = lim / sn;  sx = sx * f;  sz = sz * f                     step clamp
      p.x = p.x - sx;  p.z = p.z - sz
No early exit: every point runs exactly K steps, so results are deterministic and comparable bit for bit.

The final evaluation at p_K is sampling.sample_maps(p_K) (height = displacement.y, gradient_foam) together with D.xz and the
Jacobian of the same texel quads: residual = sqrt(rx*rx + rz*rz) and jacobian = det as written above, at p_K.  Where the
surface folds over itself (det <= 0, the foam regions) q can have zero or several preimages; the result then is wherever
K steps ended, and the residual and the jacobian say so.

Convergence of this binary32 specification on the C oracle's demo cascades (2 updates, 2e4 random points in +-300 m), share
of residuals <= 1 mm:  128^2 x 3: 99.82 % at K = 8, 99.89 % at K = 12;  256^2 x 4: 98.78 % / 99.54 %;  512^2 x 4: 98.46 % /
99.48 %;  K = 0 (the map query at q): 0 %.
"""
from __future__ import annotations

import numpy as np

from . import sampling

F = np.float32

SURFACE_POINT = np.dtype([("height", np.float32), ("source_x", np.float32), ("source_z", np.float32), ("residual", np.float32),
                          ("gradient_foam", np.float32, 3), ("jacobian", np.float32)])    # struct ocean_surface_point, 32 B

DET_MIN = F(0.05)


def texel_quad(tex: np.ndarray, u: np.ndarray, v: np.ndarray):
    """The four texels and weights sampling.texture_bilinear filters: (t00, t10, t01, t11) float32 [n][4], (fx, fy) [n][1]."""
    N = tex.shape[0]
    n = F(N)
    x = u * n - F(0.5)
    y = v * n - F(0.5)
    x0 = np.floor(x)
    y0 = np.floor(y)
    fx = (x - x0)[:, None]
    fy = (y - y0)[:, None]
    ix0 = np.mod(x0.astype(np.int64), N)
    iy0 = np.mod(y0.astype(np.int64), N)
    ix1 = np.mod(ix0 + 1, N)
    iy1 = np.mod(iy0 + 1, N)
    t00, t10 = tex[iy0, ix0].astype(np.float32), tex[iy0, ix1].astype(np.float32)
    t01, t11 = tex[iy1, ix0].astype(np.float32), tex[iy1, ix1].astype(np.float32)
    return (t00, t10, t01, t11), (fx, fy)


def displacement_jacobian(displacement: np.ndarray, px: np.ndarray, pz: np.ndarray, sc: np.ndarray):
    """D.xz at p and the four entries of dD.xz/dxz (Jxx = dDx/dx, Jxz = dDx/dz, Jzx = dDz/dx, Jzz = dDz/dz), float32 [n]."""
    C, N = displacement.shape[0], displacement.shape[1]
    z = np.zeros(px.shape, np.float32)
    Dx, Dz, Jxx, Jxz, Jzx, Jzz = z, z, z, z, z, z
    for i in range(C):
        (t00, t10, t01, t11), (fx, fy) = texel_quad(displacement[i], px * sc[i, 0], pz * sc[i, 1])
        d = sampling._mix(sampling._mix(t00, t10, fx), sampling._mix(t01, t11, fx), fy)
        Dx = Dx + d[:, 0] * sc[i, 2]
        Dz = Dz + d[:, 2] * sc[i, 2]
        gx = (sc[i, 0] * F(N)) * sc[i, 2]
        gz = (sc[i, 1] * F(N)) * sc[i, 2]
        ex = sampling._mix(t10 - t00, t11 - t01, fy)
        ez = sampling._mix(t01 - t00, t11 - t10, fx)
        Jxx = Jxx + ex[:, 0] * gx
        Jzx = Jzx + ex[:, 2] * gx
        Jxz = Jxz + ez[:, 0] * gz
        Jzz = Jzz + ez[:, 2] * gz
    return Dx, Dz, Jxx, Jxz, Jzx, Jzz


def _residual_det(px, pz, qx, qz, Dx, Dz, Jxx, Jxz, Jzx, Jzz):
    rx = (px + Dx) - qx
    rz = (pz + Dz) - qz
    a = F(1.0) + Jxx
    d = F(1.0) + Jzz
    det = a * d - Jxz * Jzx
    return rx, rz, a, d, det


def query_surface(displacement: np.ndarray, normal: np.ndarray, points_xz: np.ndarray, map_scales: np.ndarray, iterations: int):
    """displacement, normal: [C][N][N][4] float16; points_xz: [n][2] world x, z of the query points q; map_scales: [C][4]
    float32 (sampling.sample_maps' meaning); iterations: K >= 0.  Returns a SURFACE_POINT array [n]."""
    pts = np.ascontiguousarray(points_xz, np.float32).reshape(-1, 2)
    sc = np.ascontiguousarray(map_scales, np.float32).reshape(-1, 4)
    displacement = displacement[:sc.shape[0]]
    normal = normal[:sc.shape[0]]
    qx, qz = pts[:, 0].copy(), pts[:, 1].copy()
    px, pz = qx.copy(), qz.copy()
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for _ in range(int(iterations)):
            Dx, Dz, Jxx, Jxz, Jzx, Jzz = displacement_jacobian(displacement, px, pz, sc)
            rx, rz, a, d, det = _residual_det(px, pz, qx, qz, Dx, Dz, Jxx, Jxz, Jzx, Jzz)
            newton = det > DET_MIN
            safe = np.where(newton, det, F(1.0))
            sx = np.where(newton, (d * rx - Jxz * rz) / safe, rx)
            sz = np.where(newton, (a * rz - Jzx * rx) / safe, rz)
            rn = np.sqrt(rx * rx + rz * rz)
            sn = np.sqrt(sx * sx + sz * sz)
            lim = F(2.0) * rn
            clamp = sn > lim
            f = np.where(clamp, lim / np.where(clamp, sn, F(1.0)), F(1.0))
            sx = np.where(clamp, sx * f, sx)
            sz = np.where(clamp, sz * f, sz)
            px = px - sx
            pz = pz - sz
        Dx, Dz, Jxx, Jxz, Jzx, Jzz = displacement_jacobian(displacement, px, pz, sc)
        rx, rz, _, _, det = _residual_det(px, pz, qx, qz, Dx, Dz, Jxx, Jxz, Jzx, Jzz)
        # height and gradient/foam are the map query at the source point; its displacement.xz is Dx, Dz above, bit for bit
        disp, grad = sampling.sample_maps(displacement, normal, np.stack([px, pz], 1), sc)
        out = np.empty(pts.shape[0], SURFACE_POINT)
        out["height"] = disp[:, 1]
        out["source_x"] = px
        out["source_z"] = pz
        out["residual"] = np.sqrt(rx * rx + rz * rz)
        out["gradient_foam"] = grad
        out["jacobian"] = det
    return out
