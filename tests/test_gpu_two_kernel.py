"""GPU parity of the two-kernel update path against the CPU oracle and the float64 model.

The library runs an update either as one persistent work-queue launch (the default) or as the launch pairs
k_modulate_rowfft + k_colfft_unpack, issued in L2-sized chunks of chunk_cascades(N) cascades.  The two-kernel path is
taken whenever profiling is on (ocean_set_profiling: CUDA events between the two kernels) or OCEAN_PIPELINE=split was set
when the generator was created.  Its column pass reads the row-pass scratch with plain loads instead of TMA panels, its
completion counters are brought in step by the host after the launches, and ocean_update_frames runs it frame by frame.
Every test here holds it to the same bars as the persistent path: bit-identical binary32 maps and RGBA16F textures."""
import math

import numpy as np
import pytest

from conftest import EDGE_CASES, demo_params
from oracle import pyoracle as po
from test_oracle_numpy_model_large import assert_foam_sign_matches_model, assert_matches_model, model_frame

pytestmark = pytest.mark.gpu

OCEAN_ERR_STATE = 4          # include/ocean.h
SWITCHES = ("split_env", "profiling")


def _gow():
    import godotoceanwaves_b200 as gow
    return gow


def _chunk_cascades(N):
    """ocean_kernels.cu chunk_cascades: the row-pass scratch of a chunk (32 B per texel) fits in 48 MiB of L2."""
    return max(1, (48 << 20) // (N * N * 32))


def _pair(cls_gpu, n, **over):
    return ([demo_params(cls_gpu, c, **over) for c in range(n)],
            [demo_params(po.CascadeParams, c, **over) for c in range(n)])


def _bits_equal(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _same_values(a, b):
    """element-wise ==: bit-identical up to the sign of exact zeros (the unit-twiddle butterflies skip the multiplication
    by (1, 0), which can only change the sign of a zero)"""
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(autouse=True)
def _modes():
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)
    yield
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)


def _generator(N, layers, switch, monkeypatch):
    """A generator on the two-kernel path, selected by `switch`: OCEAN_PIPELINE=split (read when the generator is created) or
    profiling; any other `switch` leaves it on the persistent path."""
    gow = _gow()
    if switch == "split_env":
        monkeypatch.setenv("OCEAN_PIPELINE", "split")
    g = gow.WaveGenerator()
    g.map_size = N
    g.init_gpu(layers)
    monkeypatch.delenv("OCEAN_PIPELINE", raising=False)
    if switch == "profiling":
        g.set_profiling(True)
    return g


def _launches_are_two_kernel(g, update, C, N, extra):
    """Runs `update` and checks the launch count of the two-kernel path: one launch pair per chunk, plus `extra` spectrum and
    dispersion-table launches (a persistent update would count one launch instead of the pairs)."""
    before = g.info().kernel_launches
    update()
    assert g.info().kernel_launches - before == 2 * math.ceil(C / _chunk_cascades(N)) + extra


# ---- 1. every stage, every size, taps on ----
@pytest.mark.parametrize("switch", SWITCHES)
@pytest.mark.parametrize("N,C", [(128, 1), (256, 4), (512, 2), (1024, 1)])
def test_single_frame_all_stages(N, C, switch, monkeypatch):
    gow = _gow()
    pg, pcpu = _pair(gow.WaveCascadeParameters, C)
    g = _generator(N, max(2, C), switch, monkeypatch)
    g.enable_f32_taps(True)
    o = po.OracleWaveGenerator(N)
    _launches_are_two_kernel(g, lambda: g.update_all(1.0 / 50.0, pg), C, N, 2)
    o.update_all(1.0 / 50.0, pcpu)
    disp16, norm16 = g.maps_to_host(0, C)
    for c in range(C):
        assert pg[c].time == pcpu[c].time and not pg[c].should_generate_spectrum
        assert _bits_equal(g.spectrum_to_host(c), o.spectrum[c]), f"spectrum cascade {c}"
        rp = g.rowpass_to_host(c)
        assert _same_values(rp, np.ascontiguousarray(np.swapaxes(o.fft_buffer[c, 0], 1, 2))), f"row pass cascade {c}"
        d32, n32 = g.f32_maps_to_host(c)
        assert _bits_equal(d32, o.displacement_f32[c]), f"binary32 displacement cascade {c}"
        assert _bits_equal(n32, o.normal_f32[c]), f"binary32 normal cascade {c}"
        assert _bits_equal(disp16[c], o.displacement_half()[c]), f"displacement texture {c}"
        assert _bits_equal(norm16[c], o.normal_half()[c]), f"normal texture {c}"
    g.free()


# ---- 2. taps off: k_colfft_unpack<N, false>, the instance the profiled bench steps run ----
@pytest.mark.parametrize("switch", SWITCHES)
@pytest.mark.parametrize("N,C", [(128, 3), (256, 4), (512, 2), (1024, 1)])
def test_textures_without_taps(N, C, switch, monkeypatch):
    gow = _gow()
    pg, pcpu = _pair(gow.WaveCascadeParameters, C)
    g = _generator(N, max(2, C), switch, monkeypatch)
    o = po.OracleWaveGenerator(N)
    o.keep_f32 = False
    for delta in (0.02, 0.017):
        g.update_all(delta, pg)
        o.update_all(delta, pcpu)
    d16, n16 = g.maps_to_host(0, C)
    assert _bits_equal(d16.view(np.uint16), o.displacement_map[:C])
    assert _bits_equal(n16.view(np.uint16), o.normal_map[:C])
    g.free()


# ---- 3. chunk boundaries: the second chunk's dispatch records and grid ----
@pytest.mark.parametrize("switch", SWITCHES)
@pytest.mark.parametrize("N,C,pick", [(256, 25, (0, 1, 22, 23, 24)), (512, 7, (0, 4, 5, 6)), (1024, 2, (0, 1))])
def test_chunk_boundaries(N, C, pick, switch, monkeypatch):
    """More cascades than one L2-sized chunk (24 at 256x256, 6 at 512x512, 1 at 1024x1024): cascades on both sides of the
    chunk boundary against the oracle over two updates."""
    gow = _gow()
    assert _chunk_cascades(N) < C
    pg = [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]
    pcpu = [demo_params(po.CascadeParams, c) for c in pick]
    g = _generator(N, C, switch, monkeypatch)
    o = po.OracleWaveGenerator(N)
    o.keep_f32 = False
    for extra in (2, 0):                                    # spectra and tables on the first update only
        _launches_are_two_kernel(g, lambda: g.update_all(0.02, pg), C, N, extra)
        o.update_all(0.02, pcpu)
    if switch == "profiling":
        assert g.last_kernel_times()[3] == _chunk_cascades(N)
    d16, n16 = g.maps_to_host(0, C)
    for k, c in enumerate(pick):
        assert _bits_equal(d16[c].view(np.uint16), o.displacement_map[k]), c
        assert _bits_equal(n16[c].view(np.uint16), o.normal_map[k]), c
    g.free()


# ---- 4. the foam loop across the paths, as bench.py switches them ----
def _oracle_frames(o, pcpu, delta, frames):
    for _ in range(frames):
        o.update_all(delta, pcpu)


@pytest.mark.parametrize("C,queue,taps", [(3, None, True), (3, None, False), (7, ("2", "2"), False)],
                         ids=["128x3_taps", "128x3", "128x7_group2_lag2"])
def test_foam_loop_across_paths(C, queue, taps, monkeypatch):
    """About 30 frames of one 128x128 generator switching between the persistent launch, the profiled two-kernel path, the fused
    multi-frame launch, the profiled frame-by-frame fallback of ocean_update_frames and update()/_process() while profiled.
    The foam plane carries the state across every switch; the maps are compared with the oracle bit for bit at three checkpoints
    and at the end; with the taps on, the binary32 maps and the row-pass scratch of the half the last update used as well.
    update_frames(4) ends in scratch half 1, so the two-kernel update after it writes half 0 while the counters of half 1 are
    ahead.  With OCEAN_QUEUE_GROUP=2 / OCEAN_QUEUE_LAG=2 the persistent launches after a switch wait on the counters that the
    host copied back after the two-kernel launches."""
    gow = _gow()
    if queue:
        monkeypatch.setenv("OCEAN_QUEUE_GROUP", queue[0])
        monkeypatch.setenv("OCEAN_QUEUE_LAG", queue[1])
    N = 128
    pg, pcpu = _pair(gow.WaveCascadeParameters, C)
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(C)
    if taps:
        g.enable_f32_taps(True)
    o = po.OracleWaveGenerator(N)
    o.keep_f32 = taps
    delta = 1.0 / 50.0
    rng = np.random.default_rng(11)

    def checkpoint(tag):
        d16, n16 = g.maps_to_host(0, C)
        for c in range(C):
            assert [p.time for p in pg] == [p.time for p in pcpu], tag
            assert _bits_equal(d16[c].view(np.uint16), o.displacement_map[c]), (tag, c)
            assert _bits_equal(n16[c].view(np.uint16), o.normal_map[c]), (tag, "foam state", c)
            if taps:
                d32, n32 = g.f32_maps_to_host(c)
                assert _bits_equal(d32, o.displacement_f32[c]) and _bits_equal(n32, o.normal_f32[c]), (tag, c)
                assert _same_values(g.rowpass_to_host(c), np.ascontiguousarray(np.swapaxes(o.fft_buffer[c, 0], 1, 2))), (tag, c)

    for _ in range(4):                                      # persistent
        g.update_all(delta, pg)
    _oracle_frames(o, pcpu, delta, 4)
    g.set_profiling(True)                                   # two-kernel
    for _ in range(4):
        g.update_all(delta, pg)
    _oracle_frames(o, pcpu, delta, 4)
    g.set_profiling(False)
    checkpoint("after the profiled updates")
    g.update_frames(delta, pg, 4)                           # fused persistent launch, ends in scratch half 1
    _oracle_frames(o, pcpu, delta, 4)
    checkpoint("after the fused launch")
    g.set_profiling(True)
    g.update_all(delta, pg)                                 # two-kernel, half 0
    _oracle_frames(o, pcpu, delta, 1)
    g.update_frames(delta, pg, 3)                           # profiled: frame by frame
    _oracle_frames(o, pcpu, delta, 3)
    checkpoint("after the profiled update_frames")
    for f in range(6):                                      # update() / _process() interleaving, profiled
        g.update(delta, pg)
        o.update(delta, pcpu)
        for _ in range(int(rng.integers(0, C + 1))):
            g._process(0.0)
            o.process()
        assert g.pass_num_cascades_remaining == o.pass_num_cascades_remaining
        if f == 2:                                          # a dirty spectrum in the middle
            pg[1].wind_speed = 7.5
            pcpu[1].wind_speed = 7.5
            pcpu[1].should_generate_spectrum = True
    g.set_profiling(False)                                  # back to persistent
    g.update_all(delta, pg)
    o.update_all(delta, pcpu)
    g.update_frames(delta, pg, 3)
    _oracle_frames(o, pcpu, delta, 3)
    g.update_all(delta, pg)
    o.update_all(delta, pcpu)
    checkpoint("end")
    assert o.normal_half()[0][..., 3].max() > 0
    g.free()


# ---- 5. parameter corners through the two-kernel path ----
@pytest.mark.parametrize("name", sorted(EDGE_CASES))
def test_edge_case_parameters(name, monkeypatch):
    """EDGE_CASES through three updates at 128x128 (test_gpu_parity.py's check); detail_damped_zeros and calm reach the exact
    fix-up of the column pass's division, which k_colfft_unpack contains too."""
    gow = _gow()
    N = 128
    pg, pcpu = _pair(gow.WaveCascadeParameters, 2, **EDGE_CASES[name])
    g = _generator(N, 2, "split_env", monkeypatch)
    o = po.OracleWaveGenerator(N)
    for delta in (0.02, 0.0, 0.031):
        g.update_all(delta, pg)
        o.update_all(delta, pcpu)
    d16, n16 = g.maps_to_host(0, 2)
    for c in range(2):
        assert _same_values(d16[c].astype(np.float32), o.displacement_half()[c].astype(np.float32)), (name, c)
        assert _same_values(n16[c].astype(np.float32), o.normal_half()[c].astype(np.float32)), (name, c)
    g.free()


# ---- 6. ocean_get_last_kernel_times ----
def test_last_kernel_times_structure():
    import ctypes as Ct
    gow = _gow()
    lib = gow.load_library()
    N, C = 256, 4
    pg = [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(C)
    a, b, c_, n = Ct.c_float(), Ct.c_float(), Ct.c_float(), Ct.c_int()

    def status():
        return lib.ocean_get_last_kernel_times(g.context, Ct.byref(a), Ct.byref(b), Ct.byref(c_), Ct.byref(n))

    assert status() == OCEAN_ERR_STATE                       # nothing profiled yet
    g.update_all(0.02, pg)
    assert status() == OCEAN_ERR_STATE                       # a persistent launch is not profiled
    g.set_profiling(True)
    assert status() == OCEAN_ERR_STATE                       # switching profiling on forgets earlier launches
    pg[2].wind_speed = 12.0                                  # one dirty spectrum
    g.update_all(0.02, pg)
    spec, row, col, chunk = g.last_kernel_times()
    assert chunk == min(C, _chunk_cascades(N))
    assert spec > 0 and math.isfinite(spec)
    assert row > 0 and col > 0 and math.isfinite(row) and math.isfinite(col)
    g.update_all(0.02, pg)                                   # no dirty spectrum
    spec, row, col, chunk = g.last_kernel_times()
    assert spec == 0 and row > 0 and col > 0 and chunk == min(C, _chunk_cascades(N))
    g.update(0.02, pg)                                       # _process: one cascade per launch sequence
    g._process(0.0)
    assert g.last_kernel_times()[3] == 1
    g.set_profiling(False)
    assert status() == OCEAN_ERR_STATE
    g.free()


# ---- float64 model at 512x512 and 1024x1024, both paths ----
@pytest.mark.parametrize("pipeline", ["persistent", "split_env"])
@pytest.mark.parametrize("N", [512, 1024])
def test_maps_match_float64_model(N, pipeline, monkeypatch):
    """The binary32 maps of demo cascades 0 and 2 against oracle/numpy_model.py at the bars of
    test_oracle_numpy_model_large.py, and the first-frame foam sign against the float64 Jacobian.  The maps are bit-identical
    to the oracle's, so the distances equal those measured on the CPU; a failure here with the parity tests passing would mean
    that the oracle and the kernels share a mistake."""
    gow = _gow()
    C = 3
    pg = [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]
    g = _generator(N, C, pipeline, monkeypatch)
    g.enable_f32_taps(True)
    g.update_all(1.0 / 50.0, pg)
    for c in (0, 2):
        d32, n32 = g.f32_maps_to_host(c)
        sp = g.spectrum_to_host(c)
        model = model_frame(N, pg[c], sp)
        assert_matches_model(sp, d32, n32, model)
        assert_foam_sign_matches_model(n32, model[4], pg[c].whitecap)
        del model
    g.free()
