"""Pins the oracle to the reference itself.

oracle/_ref/libocean_ref.so is the reference's OWN six compute shaders (assets/shaders/compute/*.glsl, text unmodified
apart from the lexical plumbing listed in oracle/ref/glsl2cpp.py) compiled for the CPU and driven like
assets/water/wave_generator.gd drives them (oracle/pyref.py).  tools/make_golden.py ran every scenario below through those
shaders and stored a SHA-256 of each resource at every checkpoint in tests/golden/ref_pins/states.json.  These tests run
the same scenarios through oracle/ocean_oracle.c -- the C restatement every GPU parity test compares the CUDA path
against -- and assert that it reproduces the shaders' outputs BIT FOR BIT: the butterfly table, the spectrum texture,
both halves of the FFT buffer and both RGBA16F maps, for the BASELINE configs that a CPU finishes in seconds, the
parameter corners, the update/_process interleaving, random parameter draws and every numeric-policy mode.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import EDGE_CASES, ROOT, demo_params
from oracle import pyoracle as po
from oracle import pyref as pr

PINS_PATH = os.path.join(ROOT, "tests", "golden", "ref_pins", "states.json")
RESOURCES = ("butterfly", "spectrum", "fft_buffer", "displacement_map", "normal_map")

MODES = [("detmath_fma", po.MATH_DET, po.CONTRACT_FMA), ("detmath_strict", po.MATH_DET, po.CONTRACT_STRICT),
         ("libm_strict", po.MATH_LIBM, po.CONTRACT_STRICT), ("libm_fma", po.MATH_LIBM, po.CONTRACT_FMA)]
BASELINE_CONFIGS = [(128, 1, 1), (256, 4, 2)]
BASELINE_IDS = ["cfg1_128x1", "cfg2_256x4"]

# the two pipelines a scenario can run on: the C oracle, and the reference's shaders (what the pins were recorded from)
ORACLE = (po.OracleWaveGenerator, po.set_modes)
REFERENCE = (pr.RefWaveGenerator, pr.set_modes)


def state(g) -> dict:
    """SHA-256 of the bytes of every resource the shaders write."""
    return {r: hashlib.sha256(np.ascontiguousarray(getattr(g, r)).tobytes()).hexdigest() for r in RESOURCES}


def baseline_config(impl, N, C, frames, mode):
    """BASELINE.json configs[0] and configs[1]: the state after each update."""
    Gen, set_modes = impl
    set_modes(mode[1], mode[2])
    g, p = Gen(N), [demo_params(po.CascadeParams, c) for c in range(C)]
    states = []
    for _ in range(frames):
        g.update_all(1.0 / 50.0, p)
        states.append(state(g))
    return {"states": states, "times": [q.time for q in p]}


def parameter_corner(impl, name, contract):
    Gen, set_modes = impl
    set_modes(po.MATH_DET, contract)
    g, p = Gen(128), [demo_params(po.CascadeParams, c, **EDGE_CASES[name]) for c in range(2)]
    for delta in (0.02, 0.0, 0.031):
        g.update_all(delta, p)
    return {"states": [state(g)]}


def foam_loop(impl):
    """update()/_process() interleaving (wave_generator.gd:56-63,90-109) and the foam state carried through RGBA16F
    (fft_unpack.glsl:59-67) over 10 frames of the three demo cascades.  Returns the pin and the generator."""
    Gen, set_modes = impl
    set_modes(po.MATH_DET, po.CONTRACT_FMA)
    N, C = 128, 3
    g, p = Gen(N), [demo_params(po.CascadeParams, c) for c in range(C)]
    rng = np.random.default_rng(11)
    for f in range(10):
        g.update(1.0 / 50.0 + float(rng.uniform(0, 0.004)), p)
        for _ in range(int(rng.integers(0, C + 1))):
            g.process()
        if f == 4:                                   # a parameter change mid-run regenerates one spectrum
            p[1].wind_speed = 12.5
            p[1].should_generate_spectrum = True
    g.update(0.02, p)
    while g.pass_num_cascades_remaining:
        g.process()
    return {"states": [state(g)]}, g


def random_parameters(impl, kw, contract, delta):
    """One random draw over the @export_range space of wave_cascade_parameters.gd (and beyond): two updates at 128x128."""
    Gen, set_modes = impl
    set_modes(po.MATH_DET, contract)
    g, p = Gen(128), [po.CascadeParams(**kw)]
    for _ in range(2):
        g.update_all(delta, p)
    return {"states": [state(g)]}


def random_draw_kwargs(draw: dict) -> dict:
    """CascadeParams keyword arguments of a stored random draw (JSON keeps the tuples as lists)."""
    return {k: tuple(v) if isinstance(v, list) else v for k, v in draw["params"].items()}


@pytest.fixture(scope="module")
def pins():
    with open(PINS_PATH) as f:
        return json.load(f)


@pytest.fixture(autouse=True)
def _restore_modes():
    yield
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)


def _assert_same_states(got, want, what):
    assert len(got["states"]) == len(want["states"]), what
    for i, (g, w) in enumerate(zip(got["states"], want["states"])):
        for r in RESOURCES:
            assert g[r] == w[r], f"{what} checkpoint {i}: {r} differs from the reference shaders'"


@pytest.mark.skipif(not pr.available(), reason="needs the reference's shaders compiled for the CPU (oracle/_ref)")
def test_reference_shaders_compiled():
    L = pr.lib()
    for s in pr.SHADERS:
        assert L.ref_has_shader(s.encode())
    import ctypes as C
    xyz = (C.c_int * 3)()
    assert L.ref_local_size(b"fft_compute", xyz) == 0 and tuple(xyz) == (1024, 1, 1)       # fft_compute.glsl:12
    assert L.ref_local_size(b"fft_unpack", xyz) == 0 and tuple(xyz) == (16, 16, 2)         # fft_unpack.glsl:11


@pytest.mark.parametrize("mode", MODES, ids=[m[0] for m in MODES])
@pytest.mark.parametrize("N,C,frames", BASELINE_CONFIGS, ids=BASELINE_IDS)
def test_oracle_reproduces_reference_shaders(N, C, frames, mode, pins):
    """BASELINE.json configs[0] and configs[1]: every resource bit-identical after each update."""
    key = f"baseline/{N}x{C}x{frames}/{mode[0]}"
    got, want = baseline_config(ORACLE, N, C, frames, mode), pins[key]
    _assert_same_states(got, want, key)
    assert got["times"] == want["times"]


@pytest.mark.parametrize("name", sorted(EDGE_CASES))
def test_oracle_reproduces_reference_shaders_on_parameter_corners(name, pins):
    for contract in (po.CONTRACT_FMA, po.CONTRACT_STRICT):
        key = f"corner/{name}/contract{contract}"
        _assert_same_states(parameter_corner(ORACLE, name, contract), pins[key], key)


def test_foam_recurrence_and_scheduling_against_reference_shaders(pins):
    got, o = foam_loop(ORACLE)
    _assert_same_states(got, pins["foam_loop"], "foam loop")
    assert o.normal_half()[0][..., 3].max() > 0


def test_half_conversion_of_the_oracle_equals_the_compilers():
    """RGBA16F stores: the oracle's hand-written RTNE float->half against _Float16 (what the reference build uses)."""
    L = po.lib()
    rng = np.random.default_rng(5)
    vals = np.concatenate([rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-9, 6, 20000).astype(np.float32),
                           np.array([0.0, -0.0, 65504.0, 65519.9, 65520.0, 1e-8, 5.96e-8, 2.98e-8, 2.9802325e-8, 6.1e-5, np.inf, -np.inf], np.float32)])
    got = np.array([L.oracle_float_to_half(float(v)) for v in vals], np.uint16)
    with np.errstate(over="ignore"):
        ref = vals.astype(np.float16).view(np.uint16)
    assert np.array_equal(got, ref)


def test_oracle_reproduces_reference_shaders_on_random_parameters(pins):
    """Random draws over the whole @export_range space of wave_cascade_parameters.gd (and beyond), two updates each at
    128x128 -- every resource bit-identical between the C oracle and the compiled reference shaders.  The draws are
    hypothesis's (derandomized, 12 examples, boundary values included), stored with the pins by tools/make_golden.py."""
    draws = pins["random"]
    assert len(draws) >= 12
    for d in draws:
        kw = random_draw_kwargs(d)
        # NaN payloads aside (log(0) at u1 == 0 is reachable in principle), the bytes must agree
        _assert_same_states(random_parameters(ORACLE, kw, d["contract"], d["delta"]), d, f"{kw} contract={d['contract']}")
