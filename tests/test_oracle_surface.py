"""CPU checks of the surface-query specification (oracle/surface.py): the water surface above a world position, with the
horizontal displacement of water.gdshader:31-37 inverted by damped Newton steps."""
import numpy as np
import pytest

from conftest import demo_params
from oracle import sampling as sp
from oracle import surface as su

F = np.float32


def _oracle_maps(N, C, frames=2):
    from oracle import pyoracle as po
    g = po.OracleWaveGenerator(N)
    g.init_gpu(max(2, C))
    params = [demo_params(po.CascadeParams, c) for c in range(C)]
    for _ in range(frames):
        g.update_all(1.0 / 50.0, params)
    scales = np.array([[F(1) / F(p.tile_length[0]), F(1) / F(p.tile_length[1]), p.displacement_scale, p.normal_scale] for p in params], F)
    return g.displacement_half()[:C].copy(), g.normal_half()[:C].copy(), scales


def test_constant_displacement_is_inverted_in_one_step():
    N = 128
    c = np.array([[1.5, -0.75, 2.25, 0.0], [-0.5, 0.25, 0.125, 0.0]], np.float16)
    disp = np.broadcast_to(c[:, None, None, :], (2, N, N, 4)).copy()
    rng = np.random.default_rng(1)
    nrm = rng.standard_normal((2, N, N, 4)).astype(np.float16)
    scales = np.array([[1 / 64.0, 1 / 64.0, 1.0, 1.0], [1 / 32.0, 1 / 32.0, 0.5, 0.25]], F)   # dyadic: every step below is exact
    q = (rng.integers(-64 * 300, 64 * 300, (3000, 2)) / 64.0).astype(F)
    cx = F(1.5) + F(-0.5) * F(0.5)
    cy = F(-0.75) + F(0.25) * F(0.5)
    cz = F(2.25) + F(0.125) * F(0.5)
    for K in (1, 3):
        r = su.query_surface(disp, nrm, q, scales, K)
        assert np.array_equal(r["source_x"], q[:, 0] - cx) and np.array_equal(r["source_z"], q[:, 1] - cz)
        assert np.all(r["height"] == cy)
        assert np.all(r["residual"] == 0.0) and np.all(r["jacobian"] == 1.0)
    _, grad = sp.sample_maps(disp, nrm, np.stack([r["source_x"], r["source_z"]], 1), scales)
    assert np.array_equal(r["gradient_foam"].view(np.uint32), grad.view(np.uint32))


def test_zero_iterations_is_the_map_query():
    N, C = 128, 3
    rng = np.random.default_rng(2)
    disp = rng.standard_normal((C, N, N, 4)).astype(np.float16)
    nrm = rng.standard_normal((C, N, N, 4)).astype(np.float16)
    q = rng.uniform(-300.0, 300.0, (4000, 2)).astype(F)
    scales = np.array([[1 / 88.0, 1 / 88.0, 1.0, 1.0], [1 / 57.0, 1 / 57.0, 0.75, 1.0], [1 / 16.0, 1 / 16.0, 0.0, 0.25]], F)
    r = su.query_surface(disp, nrm, q, scales, 0)
    d, g = sp.sample_maps(disp, nrm, q, scales)
    assert np.array_equal(r["source_x"].view(np.uint32), q[:, 0].view(np.uint32))
    assert np.array_equal(r["source_z"].view(np.uint32), q[:, 1].view(np.uint32))
    assert np.array_equal(r["height"].view(np.uint32), d[:, 1].view(np.uint32))
    assert np.array_equal(r["gradient_foam"].view(np.uint32), g.view(np.uint32))
    rx, rz = (q[:, 0] + d[:, 0]) - q[:, 0], (q[:, 1] + d[:, 2]) - q[:, 1]
    assert np.array_equal(r["residual"], np.sqrt(rx * rx + rz * rz))
    # the spec's own D.xz (texel quads) is the map query's displacement, bit for bit
    Dx, Dz, *_ = su.displacement_jacobian(disp, q[:, 0], q[:, 1], scales)
    assert np.array_equal(Dx.view(np.uint32), d[:, 0].view(np.uint32)) and np.array_equal(Dz.view(np.uint32), d[:, 2].view(np.uint32))


def test_jacobian_is_the_derivative_of_the_bilinear_filter():
    N, C = 128, 2
    rng = np.random.default_rng(3)
    disp = rng.standard_normal((C, N, N, 4)).astype(np.float16)
    scales = np.array([[1 / 88.0, 1 / 88.0, 1.0, 1.0], [1 / 57.0, 1 / 57.0, 0.75, 1.0]], F)
    p = rng.uniform(-300.0, 300.0, (2000, 2)).astype(F)
    _, _, Jxx, Jxz, Jzx, Jzz = su.displacement_jacobian(disp, p[:, 0], p[:, 1], scales)
    # central differences of the float64 interpolant, away from texel edges (where the derivative jumps)
    h = 1e-4

    def D64(x, z):
        out = np.zeros((len(x), 3))
        for i in range(C):
            gx = x * float(scales[i, 0]) * N - 0.5
            gy = z * float(scales[i, 1]) * N - 0.5
            x0, y0 = np.floor(gx), np.floor(gy)
            fx, fy = (gx - x0)[:, None], (gy - y0)[:, None]
            t = disp[i].astype(np.float64)
            ix0, iy0 = np.mod(x0.astype(np.int64), N), np.mod(y0.astype(np.int64), N)
            ix1, iy1 = np.mod(ix0 + 1, N), np.mod(iy0 + 1, N)
            d = (t[iy0, ix0] * (1 - fx) + t[iy0, ix1] * fx) * (1 - fy) + (t[iy1, ix0] * (1 - fx) + t[iy1, ix1] * fx) * fy
            out += d[:, :3] * float(scales[i, 2])
        return out

    x, z = p[:, 0].astype(np.float64), p[:, 1].astype(np.float64)
    ddx = (D64(x + h, z) - D64(x - h, z)) / (2 * h)
    ddz = (D64(x, z + h) - D64(x, z - h)) / (2 * h)
    inner = np.ones(len(p), bool)
    for i in range(C):
        for c in (x, z):
            f = np.mod(c * float(scales[i, 0]) * N - 0.5, 1.0)
            inner &= (f > 0.01) & (f < 0.99)
    assert inner.sum() > 1000
    for got, ref in ((Jxx, ddx[:, 0]), (Jzx, ddx[:, 2]), (Jxz, ddz[:, 0]), (Jzz, ddz[:, 2])):
        assert np.allclose(got[inner], ref[inner], rtol=1e-3, atol=1e-3)


@pytest.fixture(scope="module")
def demo_128x3():
    disp, nrm, scales = _oracle_maps(128, 3)
    q = np.random.default_rng(4).uniform(-300.0, 300.0, (20000, 2)).astype(F)
    return disp, nrm, scales, q, su.query_surface(disp, nrm, q, scales, 8)


def test_newton_converges_on_oracle_maps(demo_128x3):
    disp, nrm, scales, q, r = demo_128x3
    # binary32 measurement of this specification on these maps: 99.82 % within 1 mm at K = 8 (99.89 % at K = 12), against
    # 0.00 % for the map query at q itself (K = 0), whose median error is over a metre
    assert np.mean(r["residual"] <= 1e-3) >= 0.995
    r0 = su.query_surface(disp, nrm, q, scales, 0)
    assert np.median(r0["residual"]) > 0.5
    # the final evaluation is the map query at the returned source point, bit for bit
    d, g = sp.sample_maps(disp, nrm, np.stack([r["source_x"], r["source_z"]], 1), scales)
    assert np.array_equal(r["height"].view(np.uint32), d[:, 1].view(np.uint32))
    assert np.array_equal(r["gradient_foam"].view(np.uint32), g.view(np.uint32))


def test_converged_points_agree_with_a_float64_evaluation(demo_128x3):
    ndi = pytest.importorskip("scipy.ndimage")
    disp, nrm, scales, q, r = demo_128x3
    ok = r["residual"] <= 1e-3
    px, pz = r["source_x"][ok].astype(np.float64), r["source_z"][ok].astype(np.float64)
    N = disp.shape[1]
    D = np.zeros((ok.sum(), 3))
    for i in range(disp.shape[0]):
        x = px * float(scales[i, 0]) * N - 0.5
        y = pz * float(scales[i, 1]) * N - 0.5
        for ch in range(3):
            D[:, ch] += ndi.map_coordinates(disp[i, :, :, ch].astype(np.float64), [y, x], order=1, mode="grid-wrap") * float(scales[i, 2])
    miss = np.hypot(px + D[:, 0] - q[ok, 0], pz + D[:, 2] - q[ok, 1])
    assert miss.max() <= 2e-3
    assert np.abs(D[:, 1] - r["height"][ok]).max() <= 1e-3


def test_surface_point_layout():
    assert su.SURFACE_POINT.itemsize == 32
    assert [su.SURFACE_POINT.fields[k][1] for k in ("height", "source_x", "source_z", "residual", "gradient_foam", "jacobian")] == \
        [0, 4, 8, 12, 16, 28]
    import godotoceanwaves_b200 as gow
    assert gow.WaveGenerator.SURFACE_POINT == su.SURFACE_POINT
