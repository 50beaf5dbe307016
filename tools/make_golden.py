"""Writes tests/golden/*.json: golden vectors PRODUCED BY THE REFERENCE'S OWN SHADERS.

The generator is oracle/pyref.RefWaveGenerator: the six GLSL compute shaders of /root/reference compiled for the CPU
(oracle/ref/, output oracle/_ref/libocean_ref.so) and sequenced as assets/water/wave_generator.gd sequences them, in
the numeric-policy configuration the CUDA kernels reproduce (DETMATH transcendentals, FMA contraction of
x*y +/- z*w -- see oracle/ref/glsl_shim.hpp).  This script therefore only runs where /root/reference is present (this
container); the vectors travel as small JSON files and are checked
  * against the C oracle and against oracle/_ref on the CPU (-m "not gpu"),
  * against the CUDA path on the B200 (-m gpu).

Stored per case: CRC-32 of the full arrays (little-endian bytes) and a strided subsample as hex strings for debugging.
The map-query vectors (SURVEY 8f row f2) are oracle/sampling.py's (the numpy specification of the water shader's
sampling contract) evaluated on the reference-produced maps.

It also writes tests/golden/ref_pins/states.json: the scenarios of tests/test_ref_pins_oracle.py run through the same
shaders in every numeric-policy mode, stored as a SHA-256 of each resource at every checkpoint, which the C oracle must
reproduce bit for bit.

  python tools/make_golden.py            # rewrites tests/golden/
"""
import json
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import demo_params          # noqa: E402
from oracle import pyoracle as po         # noqa: E402
from oracle import pyref as pr            # noqa: E402
from oracle import sampling as sp         # noqa: E402

CASES = [dict(name="cfg1_128x1", N=128, C=1, frames=2), dict(name="demo_128x3", N=128, C=3, frames=3),
         dict(name="cfg2_256x4", N=256, C=4, frames=2)]


def crc(a) -> int:
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def sub(a, step):
    """every step-th texel of every layer as a hex string of the raw little-endian bytes"""
    return np.ascontiguousarray(a[:, ::step, ::step]).tobytes().hex()


def query_points(n, seed):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-300.0, 300.0, (n, 2)).astype(np.float32)
    pts[:4] = np.array([[0, 0], [88.0, -88.0], [-1234.5, 987.25], [0.34375, 0.34375]], np.float32)
    return pts


def run_case(case):
    N, C, frames = case["N"], case["C"], case["frames"]
    pr.set_modes(po.MATH_DET, po.CONTRACT_FMA)
    gen = pr.RefWaveGenerator(N)
    gen.init_gpu(max(2, C))
    params = [demo_params(po.CascadeParams, c) for c in range(C)]
    out = dict(case)
    out["generator"] = "oracle/_ref: /root/reference/assets/shaders/compute/*.glsl compiled for the CPU (DETMATH, FMA contraction)"
    out["frames_crc"] = []
    for f in range(frames):
        gen.update_all(1.0 / 50.0, params)
        out["frames_crc"].append({"displacement": crc(gen.displacement_map[:C]), "normal": crc(gen.normal_map[:C])})
    out["spectrum_crc"] = crc(gen.spectrum[:C])
    step = N // 8
    out["subsample_step"] = step
    out["spectrum_sub"] = sub(gen.spectrum[:C], step)
    out["displacement_sub"] = sub(gen.displacement_map[:C], step)
    out["normal_sub"] = sub(gen.normal_map[:C], step)
    # map-query op on the final maps
    pts = query_points(256, 7 + N)
    scales = np.array([[np.float32(1.0) / np.float32(p.tile_length[0]), np.float32(1.0) / np.float32(p.tile_length[1]),
                        p.displacement_scale, p.normal_scale] for p in params], np.float32)
    d, g = sp.sample_maps(gen.displacement_map[:C].view(np.float16), gen.normal_map[:C].view(np.float16), pts, scales)
    out["query"] = {"points_seed": 7 + N, "n": 256, "displacement_crc": crc(d), "gradient_foam_crc": crc(g),
                    "displacement_head": d[:4].tobytes().hex(), "gradient_foam_head": g[:4].tobytes().hex()}
    return out


def random_draws():
    """The draws hypothesis makes, derandomized (12 examples, boundary values included), over the whole @export_range
    space of wave_cascade_parameters.gd and beyond."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st

    pos = dict(allow_nan=False, allow_infinity=False)
    params = st.fixed_dictionaries(dict(
        tile_length=st.tuples(st.floats(0.5, 4000.0, width=32, **pos), st.floats(0.5, 4000.0, width=32, **pos)),
        wind_speed=st.floats(0.0001, 60.0, **pos), wind_direction=st.floats(-360.0, 720.0, **pos),
        fetch_length=st.floats(0.0001, 2000.0, **pos), swell=st.floats(0.0, 2.0, **pos), spread=st.floats(0.0, 1.0, **pos),
        detail=st.floats(0.0, 1.0, **pos), whitecap=st.floats(0.0, 2.0, **pos), foam_amount=st.floats(0.0, 10.0, **pos),
        spectrum_seed=st.tuples(st.integers(-2**31, 2**31 - 1), st.integers(-2**31, 2**31 - 1)),
        time=st.floats(0.0, 50000.0, **pos)))
    draws = []

    @settings(max_examples=12, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.too_slow])
    @given(kw=params, contract=st.sampled_from([po.CONTRACT_FMA, po.CONTRACT_STRICT]), delta=st.floats(0.0, 0.1, **pos))
    def collect(kw, contract, delta):
        draws.append(dict(params=kw, contract=contract, delta=delta))

    collect()
    return draws


def ref_pins():
    import test_ref_pins_oracle as t
    ref = t.REFERENCE
    out = {"generator": "oracle/_ref: the reference's compute shaders compiled for the CPU"}
    for N, C, frames in t.BASELINE_CONFIGS:
        for mode in t.MODES:
            out[f"baseline/{N}x{C}x{frames}/{mode[0]}"] = t.baseline_config(ref, N, C, frames, mode)
    for name in sorted(t.EDGE_CASES):
        for contract in (po.CONTRACT_FMA, po.CONTRACT_STRICT):
            out[f"corner/{name}/contract{contract}"] = t.parameter_corner(ref, name, contract)
    out["foam_loop"] = t.foam_loop(ref)[0]
    out["random"] = []
    for d in random_draws():
        d.update(t.random_parameters(ref, t.random_draw_kwargs(d), d["contract"], d["delta"]))
        out["random"].append(d)
    return out


if __name__ == "__main__":
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    for case in CASES:
        res = run_case(case)
        path = os.path.join(ROOT, "tests", "golden", case["name"] + ".json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print("wrote", os.path.relpath(path, ROOT), res["frames_crc"][-1], res["query"]["displacement_crc"])
    path = os.path.join(ROOT, "tests", "golden", "ref_pins", "states.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(ref_pins(), f, indent=1)
    print("wrote", os.path.relpath(path, ROOT))
