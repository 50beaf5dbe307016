"""GPU parity of the surface query (ocean_query_surface; water.gdshader:31-37 inverted, then :72-84 at the source point)
against its numpy specification oracle/surface.py, on the generator's own RGBA16F maps.  Bar: bit-identical records."""
import numpy as np
import pytest

from conftest import demo_params
from oracle import surface as su
from godotoceanwaves_b200.native import check

pytestmark = pytest.mark.gpu


def _gen(N, C, frames=2):
    import godotoceanwaves_b200 as gow
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(max(2, C))
    params = [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]
    for _ in range(frames):
        g.update_all(1.0 / 50.0, params)
    return gow, g, params


def _points(n, seed, span):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-span, span, (n, 2)).astype(np.float32)
    # texel centres, texel edges, the origin, whole tiles away: the corner points of test_gpu_sampling.py
    pts[:8] = np.array([[0, 0], [0.34375, 0.34375], [88.0, -88.0], [-0.0, 57.0], [1e-30, -1e-30], [16.0, 16.0], [-1234.5, 987.25],
                        [4096.0, -4096.0]], np.float32)
    return pts


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("N,C", [(128, 3), (256, 4), (512, 2), (1024, 8)])
def test_query_surface_bit_exact(N, C):
    gow, g, params = _gen(N, C)
    d16, n16 = g.maps_to_host(0, C)
    scales = gow.WaveGenerator.map_scales(params)
    pts = _points(20000, 23 + N, 300.0)
    for K in (0, 1, 8):
        before = g.info().kernel_launches
        rec = g.query_surface(pts, scales, K)
        assert g.info().kernel_launches == before + 1
        ref = su.query_surface(d16, n16, pts, scales, K)
        assert rec.dtype == ref.dtype and rec.shape == (len(pts),)
        assert np.array_equal(_bits(rec), _bits(ref)), (N, C, K)
    # fewer cascades than layers: the first ones only
    rec = g.query_surface(pts[:1000], scales[:1], 8)
    assert np.array_equal(_bits(rec), _bits(su.query_surface(d16[:1], n16[:1], pts[:1000], scales[:1], 8)))
    g.free()


def test_query_surface_is_the_map_query_at_the_source():
    gow, g, params = _gen(256, 4)
    scales = gow.WaveGenerator.map_scales(params)
    pts = _points(20000, 5, 300.0)
    rec = g.query_surface(pts, scales)
    assert np.mean(rec["residual"] <= 1e-3) >= 0.98
    src = np.stack([rec["source_x"], rec["source_z"]], 1)
    d, gr = g.sample(src, scales)
    assert np.array_equal(_bits(rec["height"]), _bits(d[:, 1]))
    assert np.array_equal(_bits(rec["gradient_foam"]), _bits(gr))
    # the residual is the distance between the displaced source and the query point, as the map query sees it
    rx, rz = (src[:, 0] + d[:, 0]) - pts[:, 0], (src[:, 1] + d[:, 2]) - pts[:, 1]
    assert np.array_equal(_bits(rec["residual"]), _bits(np.sqrt(rx * rx + rz * rz)))
    g.free()


def test_query_surface_device_entry_point():
    import torch
    gow, g, params = _gen(256, 4)
    scales = gow.WaveGenerator.map_scales(params)
    pts = _points(20000, 6, 300.0)
    host = g.query_surface(pts, scales, 8)
    pts_dev = torch.from_numpy(pts).cuda()
    out_dev = torch.zeros((len(pts), 8), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    lib = gow.load_library()
    check(lib.ocean_query_surface_device(g.context, len(pts), pts_dev.data_ptr(), len(scales), scales.ctypes.data, 8, out_dev.data_ptr()))
    g.synchronize()
    dev = out_dev.cpu().numpy().view(gow.WaveGenerator.SURFACE_POINT).reshape(-1)
    assert np.array_equal(_bits(dev), _bits(host))
    g.free()


def test_query_surface_arguments():
    gow, g, params = _gen(128, 2, frames=1)
    scales = gow.WaveGenerator.map_scales(params)
    pts = np.zeros((4, 2), np.float32)
    rec = g.query_surface(np.zeros((0, 2), np.float32), scales)           # empty batch
    assert rec.shape == (0,) and rec.dtype == gow.WaveGenerator.SURFACE_POINT
    for bad in (-1, 33):
        with pytest.raises(gow.OceanError):
            g.query_surface(pts, scales, bad)
    assert len(g.query_surface(pts, scales, 32)) == 4
    with pytest.raises(gow.OceanError):
        g.query_surface(pts, np.zeros((3, 4), np.float32))                 # more cascades than layers
    with pytest.raises(gow.OceanError):
        g.query_surface(pts, np.zeros((0, 4), np.float32))
    lib = gow.load_library()
    out = np.empty(4, gow.WaveGenerator.SURFACE_POINT)
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface(g.context, -1, pts.ctypes.data, 2, scales.ctypes.data, 8, out.ctypes.data))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface(g.context, 4, None, 2, scales.ctypes.data, 8, out.ctypes.data))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface(g.context, 4, pts.ctypes.data, 2, scales.ctypes.data, 8, None))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface(g.context, 4, pts.ctypes.data, 2, None, 8, out.ctypes.data))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface_device(g.context, 4, None, 2, scales.ctypes.data, 8, None))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_query_surface_device(None, 4, pts.ctypes.data, 2, scales.ctypes.data, 8, out.ctypes.data))
    g.free()
