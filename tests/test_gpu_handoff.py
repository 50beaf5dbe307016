"""GPU tests of the host hand-off of the maps and of the device entry points of the map and spray queries.

ocean_snapshot_maps_to_host_async copies the maps on the device (compute stream) and sends the copy to the host on a second
stream while the next update runs, into buffers the caller alternates; ocean_wait_snapshot waits for the last hand-off.  Every
host buffer must end up holding the maps of the step it was requested for.  The device entry points must give exactly what
the host entry points give."""
import ctypes as Ct

import numpy as np
import pytest

from conftest import demo_params
from godotoceanwaves_b200.native import check

pytestmark = pytest.mark.gpu


def _gow():
    import godotoceanwaves_b200 as gow
    return gow


def _generator(N, C):
    gow = _gow()
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(C)
    return g, [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]


def _host_alloc(lib, nbytes):
    p = Ct.c_void_p()
    check(lib.ocean_host_alloc(Ct.byref(p), nbytes))
    return p


def _read(ptr, count, N):
    """`count` RGBA16F layers from a host buffer, as uint16 [count][N][N][4]."""
    n = count * N * N * 4
    return np.ctypeslib.as_array((Ct.c_uint16 * n).from_address(ptr.value)).reshape(count, N, N, 4).copy()


def test_snapshot_double_buffering():
    """bench.py's end-to-end loop at 256x256 x 4: update_all, then a snapshot into one of two alternating pinned buffer pairs,
    six steps, one wait at the end.  A second generator fed the same parameters gives the maps of every step through the
    synchronous copy."""
    gow = _gow()
    lib = gow.load_library()
    N, C = 256, 4
    delta = 1.0 / 50.0
    a, pa = _generator(N, C)
    b, pb = _generator(N, C)
    layer_bytes = N * N * 8
    host = [(_host_alloc(lib, C * layer_bytes), _host_alloc(lib, C * layer_bytes)) for _ in range(2)]
    ref = []
    for i in range(6):
        a.update_all(delta, pa)
        check(lib.ocean_snapshot_maps_to_host_async(a.context, 0, C, host[i & 1][0], host[i & 1][1]))
        b.update_all(delta, pb)
        d, n = b.maps_to_host()
        ref.append((d.view(np.uint16), n.view(np.uint16)))
    check(lib.ocean_wait_snapshot(a.context))
    for k, step in ((0, 4), (1, 5)):                      # steps 5 and 6
        assert np.array_equal(_read(host[k][0], C, N), ref[step][0]), f"displacement, step {step + 1}"
        assert np.array_equal(_read(host[k][1], C, N), ref[step][1]), f"normal, step {step + 1}"
    assert not np.array_equal(ref[4][1], ref[5][1])      # the two steps differ, so a stale buffer would show

    # a partial range: layers [1, 3) land at the start of the host buffers
    a.update_all(delta, pa)
    b.update_all(delta, pb)
    check(lib.ocean_snapshot_maps_to_host_async(a.context, 1, 2, host[0][0], host[0][1]))
    check(lib.ocean_wait_snapshot(a.context))
    d7, n7 = b.maps_to_host(1, 2)
    assert np.array_equal(_read(host[0][0], 2, N), d7.view(np.uint16))
    assert np.array_equal(_read(host[0][1], 2, N), n7.view(np.uint16))

    # one NULL host pointer: the other map is handed off, the buffer of the skipped one is left alone
    untouched = _read(host[1][1], C, N)
    a.update_all(delta, pa)
    b.update_all(delta, pb)
    check(lib.ocean_snapshot_maps_to_host_async(a.context, 0, C, host[1][0], None))
    a.update_all(delta, pa)                               # the next update runs beside the hand-off
    check(lib.ocean_wait_snapshot(a.context))
    d8, n8 = b.maps_to_host()
    assert np.array_equal(_read(host[1][0], C, N), d8.view(np.uint16))
    assert np.array_equal(_read(host[1][1], C, N), untouched)
    b.update_all(delta, pb)
    check(lib.ocean_snapshot_maps_to_host_async(a.context, 0, C, None, host[0][1]))
    check(lib.ocean_wait_snapshot(a.context))
    _, n9 = b.maps_to_host()
    assert np.array_equal(_read(host[0][1], C, N), n9.view(np.uint16))

    # argument errors: ranges outside the layers; an empty range is a no-op
    for first, count in ((-1, 1), (0, -1), (0, C + 1), (C, 1), (3, 2)):
        with pytest.raises(gow.OceanError):
            check(lib.ocean_snapshot_maps_to_host_async(a.context, first, count, host[0][0], host[0][1]))
    check(lib.ocean_snapshot_maps_to_host_async(a.context, C, 0, host[0][0], host[0][1]))
    check(lib.ocean_wait_snapshot(a.context))
    assert np.array_equal(_read(host[0][1], C, N), n9.view(np.uint16))
    for d, n in host:
        check(lib.ocean_host_free(d))
        check(lib.ocean_host_free(n))
    a.free(); b.free()


def test_copy_maps_to_host_async():
    gow = _gow()
    lib = gow.load_library()
    N, C = 256, 4
    g, p = _generator(N, C)
    for _ in range(3):
        g.update_all(0.02, p)
    d_ref, n_ref = g.maps_to_host()
    d = np.full((C, N, N, 4), 0x7e00, np.uint16)
    n = np.full((C, N, N, 4), 0x7e00, np.uint16)
    check(lib.ocean_copy_maps_to_host_async(g.context, 0, C, d.ctypes.data, n.ctypes.data))
    check(lib.ocean_synchronize(g.context))
    assert np.array_equal(d, d_ref.view(np.uint16)) and np.array_equal(n, n_ref.view(np.uint16))
    d2 = np.zeros((2, N, N, 4), np.uint16)
    check(lib.ocean_copy_maps_to_host_async(g.context, 2, 2, d2.ctypes.data, None))
    check(lib.ocean_synchronize(g.context))
    assert np.array_equal(d2, d_ref[2:].view(np.uint16))
    with pytest.raises(gow.OceanError):
        check(lib.ocean_copy_maps_to_host_async(g.context, 3, 2, d2.ctypes.data, None))
    g.free()


def test_sample_maps_device_entry_point():
    import torch
    gow = _gow()
    g, p = _generator(256, 4)
    for _ in range(2):
        g.update_all(0.02, p)
    scales = gow.WaveGenerator.map_scales(p)
    rng = np.random.default_rng(3)
    pts = rng.uniform(-300.0, 300.0, (20000, 2)).astype(np.float32)
    pts[:4] = np.array([[0, 0], [88.0, -88.0], [-0.0, 57.0], [4096.0, -4096.0]], np.float32)
    d_host, g_host = g.sample(pts, scales)
    pts_dev = torch.from_numpy(pts).cuda()
    d_dev = torch.full((len(pts), 3), float("nan"), dtype=torch.float32, device="cuda")
    g_dev = torch.full((len(pts), 3), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    lib = gow.load_library()
    check(lib.ocean_sample_maps_device(g.context, len(pts), pts_dev.data_ptr(), len(scales), scales.ctypes.data, d_dev.data_ptr(),
                                       g_dev.data_ptr()))
    g.synchronize()
    assert np.array_equal(d_dev.cpu().numpy().view(np.uint32), d_host.view(np.uint32))
    assert np.array_equal(g_dev.cpu().numpy().view(np.uint32), g_host.view(np.uint32))
    # fewer cascades than layers
    d1, g1 = g.sample(pts, scales[:1])
    check(lib.ocean_sample_maps_device(g.context, len(pts), pts_dev.data_ptr(), 1, scales.ctypes.data, d_dev.data_ptr(), g_dev.data_ptr()))
    g.synchronize()
    assert np.array_equal(d_dev.cpu().numpy().view(np.uint32), d1.view(np.uint32))
    assert np.array_equal(g_dev.cpu().numpy().view(np.uint32), g1.view(np.uint32))
    g.free()


def test_extract_spray_device_entry_point():
    import torch
    gow = _gow()
    N, C = 128, 3
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(C)
    p = [demo_params(gow.WaveCascadeParameters, c, whitecap=0.9, foam_amount=10.0) for c in range(C)]
    for _ in range(25):                                   # a foamy sea (test_gpu_spray.py)
        g.update_all(1.0 / 50.0, p)
    scales = gow.WaveGenerator.map_scales(p)
    pts = gow.WaveGenerator.spray_grid(10000)
    ps = np.array([0.6, 1.4, 0.6], np.float32)
    ref, count = g.extract_spray(pts, scales, ps)
    assert 7 < count < len(pts)
    lib = gow.load_library()
    rec_size = gow.WaveGenerator.SPRAY_RECORD.itemsize
    pts_dev = torch.from_numpy(pts).cuda()
    active = torch.full((1,), -1, dtype=torch.int32, device="cuda")

    def run(n, max_records):
        recs = torch.full((max(max_records, 1) * rec_size,), 0xAB, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        check(lib.ocean_extract_spray_device(g.context, n, pts_dev.data_ptr(), len(scales), scales.ctypes.data, ps.ctypes.data, max_records,
                                             recs.data_ptr(), active.data_ptr()))
        g.synchronize()
        return recs.cpu().numpy(), int(active.item())

    recs, num = run(len(pts), len(pts))
    assert num == count
    assert recs[:count * rec_size].tobytes() == ref.tobytes()
    assert np.all(recs[count * rec_size:] == 0xAB)         # nothing written past the active records
    recs, num = run(len(pts), 7)                          # max_records cuts the records, not the count
    assert num == count and recs.tobytes() == ref[:7].tobytes()
    active.fill_(12345)
    recs, num = run(0, 4)                                 # no candidates: the count is written, nothing else
    assert num == 0 and np.all(recs == 0xAB)
    g.free()
