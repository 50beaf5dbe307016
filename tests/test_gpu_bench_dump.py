"""bench.py --dump-outputs writes the maps of the LAST TIMED step: bit for bit the oracle's maps after the updates bench.py
runs before it (one that creates the spectra, the warm-up, then exactly --steps timed ones)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    import bench
    N, C, warmup, steps = 128, 2, 3, 2
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                          "--map-size", str(N), "--cascades-per-set", str(C), "--sets", "1", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    d = np.load(tmp_path / "displacement_map.npy")
    n = np.load(tmp_path / "normal_map.npy")
    assert d.dtype == n.dtype == np.float32 and d.shape == n.shape == (C, N, N, 4)
    po.set_modes(po.MATH_DET, po.CONTRACT_FMA)
    o = po.OracleWaveGenerator(N)
    o.keep_f32 = False
    params = [bench.synth_params(po.CascadeParams, c) for c in range(C)]
    for _ in range(1 + warmup + steps):
        o.update_all(1.0 / 50.0, params)
    assert np.array_equal(d.view(np.uint32), o.displacement_half()[:C].astype(np.float32).view(np.uint32))
    assert np.array_equal(n.view(np.uint32), o.normal_half()[:C].astype(np.float32).view(np.uint32))
