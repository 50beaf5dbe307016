"""The C oracle against the independent float64 model (oracle/numpy_model.py) at 512x512 and 1024x1024, the map sizes whose
FFT plans (16*16*2, 16*16*4) test_oracle_pins.py does not reach.  Same check and bars as test_full_frame_matches_numpy_model:
spectrum within 2e-6 of max|h0|, the three displacement and the three normal channels within 5e-6 of each field's maximum,
first-frame foam within 1e-5 absolute; the RGBA16F textures are the RTNE rounding of the binary32 maps.  The largest distance
measured is 1.3e-6 relative (normal x at 1024x1024, demo cascade 0), about 4x below the bar.

The helpers here are shared with tests/test_gpu_two_kernel.py, which holds the CUDA maps to the same model."""
import numpy as np
import pytest

from conftest import EDGE_CASES, demo_params
from oracle import numpy_model as nm
from oracle import pyoracle as po

SPECTRUM_TOL = 2e-6     # of max|h0|
FIELD_TOL = 5e-6        # of max|field|
FOAM_TOL = 1e-5         # absolute

# Foam-sign band.  On the first frame (foam_prev = 0, foam_grow_rate > 0) foam > 0 holds exactly where the binary32 Jacobian is
# below whitecap.  On texels with 0 < foam < 1, foam / foam_grow_rate = whitecap - J, so the foam plane gives the oracle's
# Jacobian back: its largest distance to the float64 Jacobian over the six cases below is 9.5e-7 (1024x1024, demo cascade 0).
# JACOBIAN_BAND is four times that, the margin of the field bars.  Texels with |J - whitecap| < JACOBIAN_BAND are excluded from
# the mask comparison: 1, 0, 4, 2, 6 and 5 texels in the six cases (of 2^18 or 2^20 each); none of them actually differs.
JACOBIAN_BAND = 4e-6
MAX_BAND_TEXELS = 16

CASES = {
    "512_c0": (512, 0, {}),
    "512_c2": (512, 2, {}),
    "1024_c0": (1024, 0, {}),
    "1024_c2": (1024, 2, {}),
    "1024_anisotropic_tile": (1024, 0, EDGE_CASES["anisotropic_tile"]),
    "1024_late_time": (1024, 0, EDGE_CASES["late_time"]),
}


@pytest.fixture(autouse=True)
def _modes():
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)
    yield
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)


def model_frame(N, p, spectrum):
    """float64 model of one update of the cascade with parameters p (time and foam rates as the update left them) from the
    binary32 spectrum texture [N][N][4] the update used.  Returns (h0, conj h0(-k), displacement, normal, jacobian)."""
    pc = po.pc_spectrum_compute(p, 0)
    tl = (pc.tile_length[0], pc.tile_length[1])
    h0, h0m = nm.spectrum(N, p.spectrum_seed, tl, pc.alpha, pc.peak_frequency, pc.wind_speed, pc.angle, pc.depth,
                          pc.swell, pc.detail, pc.spread)
    sp = spectrum.astype(np.float64)
    layers = nm.modulate(sp[..., 0] + 1j * sp[..., 1], sp[..., 2] + 1j * sp[..., 3], N, tl, po.DEPTH, float(np.float32(p.time)))
    disp, normal, jac = nm.unpack(nm.ifft_maps(layers), 0.0, float(np.float32(p.whitecap)), float(np.float32(p.foam_grow_rate)),
                                  float(np.float32(p.foam_decay_rate)))
    return h0, h0m, disp, normal, jac


def assert_matches_model(spectrum, d32, n32, model):
    """The bars of test_full_frame_matches_numpy_model; returns the largest relative field distance."""
    h0, h0m, disp, normal, _ = model
    sp = spectrum.astype(np.float64)
    scale = np.max(np.abs(h0))
    assert np.max(np.abs(sp[..., 0] + 1j * sp[..., 1] - h0)) <= SPECTRUM_TOL * scale
    assert np.max(np.abs(sp[..., 2] + 1j * sp[..., 3] - h0m)) <= SPECTRUM_TOL * scale
    worst = 0.0
    for got, ref, name in ((d32, disp, "displacement"), (n32, normal, "normal")):
        for ch in range(3):
            rel = float(np.max(np.abs(got[..., ch] - ref[..., ch])) / np.max(np.abs(ref[..., ch])))
            assert rel <= FIELD_TOL, (name, ch, rel)
            worst = max(worst, rel)
    assert np.max(np.abs(n32[..., 3] - normal[..., 3])) <= FOAM_TOL
    return worst


def assert_foam_sign_matches_model(n32, jacobian, whitecap):
    """First frame: foam > 0 exactly where the float64 Jacobian is below whitecap, outside the band |J - whitecap| < JACOBIAN_BAND."""
    wc = float(np.float32(whitecap))
    keep = np.abs(jacobian - wc) >= JACOBIAN_BAND
    assert int((~keep).sum()) <= MAX_BAND_TEXELS
    foaming = n32[..., 3] > 0
    assert foaming.any() and not foaming.all()
    bad = keep & (foaming != (jacobian < wc))
    assert not bad.any(), (int(bad.sum()), np.argwhere(bad)[:4].tolist())


@pytest.fixture(scope="module", params=sorted(CASES))
def oracle_case(request):
    """One update of the case's cascade through the oracle and the model.  Module scope: pytest runs both checks of a case
    before it builds the next one, so only one case (a few hundred MB at 1024x1024) is alive at a time."""
    N, c, over = CASES[request.param]
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)
    p = demo_params(po.CascadeParams, c, **over)
    g = po.OracleWaveGenerator(N)
    g.init_gpu(1)
    g.update_all(1.0 / 50.0, [p])
    return p, g, model_frame(N, p, g.spectrum[0])


def test_large_frame_matches_numpy_model(oracle_case):
    p, g, model = oracle_case
    d, n = g.displacement_f32[0], g.normal_f32[0]
    assert_matches_model(g.spectrum[0], d, n, model)
    assert np.array_equal(g.displacement_half()[0], d.astype(np.float16))
    assert np.array_equal(g.normal_half()[0], n.astype(np.float16))


def test_large_frame_foam_sign_matches_float64_jacobian(oracle_case):
    p, g, model = oracle_case
    assert p.foam_grow_rate > 0
    assert_foam_sign_matches_model(g.normal_f32[0], model[4], p.whitecap)
