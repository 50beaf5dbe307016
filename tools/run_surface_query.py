"""Times the surface query (ocean_query_surface_device) on device-resident random points, with the map query
(ocean_sample_maps_device) on the same points beside it (GPU).  Prints one JSON object per (maps, op, K) and, with --out,
appends them to that file.

Workloads: 2^20 points uniform in +-300 m on the demo cascades at 256^2 x 4 (4 MiB of maps, L2-resident) and at 1024^2 x 8
(128 MiB of maps, more than the 126 MB L2), K = 0, 4, 8 Newton steps.  Each number is the device time (the generator's CUDA
event timer) of a window of back-to-back calls after warm-up, three windows per row; every call includes the 16 B/cascade
upload of map_scales the device entry points make.  Texel gathers per point (8 B each): sample op 24 C, surface query
4 C (K + 1) + 20 C.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import godotoceanwaves_b200 as gow  # noqa: E402
from conftest import demo_params  # noqa: E402
from godotoceanwaves_b200.native import check  # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    except Exception:
        power, clock = "not measured", "not measured"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_calls(g, call, min_window_ms=200.0):
    for _ in range(5):
        call()
    g.synchronize()
    g.timer_start()
    for _ in range(5):
        call()
    probe = g.timer_stop() / 5
    reps = int(min(5000, max(10, min_window_ms / max(probe, 1e-3))))
    times = []
    for _ in range(3):
        g.timer_start()
        for _ in range(reps):
            call()
        times.append(g.timer_stop() / reps)
    return reps, sorted(times)


def run(N, C, n, ks, ident, sink):
    g = gow.WaveGenerator(); g.map_size = N; g.init_gpu(max(2, C))
    params = [demo_params(gow.WaveCascadeParameters, c) for c in range(C)]
    for _ in range(2):
        g.update_all(1.0 / 50.0, params)
    scales = gow.WaveGenerator.map_scales(params)
    lib = gow.load_library()
    pts = torch.from_numpy(np.random.default_rng(1).uniform(-300.0, 300.0, (n, 2)).astype(np.float32)).cuda()
    rec = torch.empty((n, 8), dtype=torch.float32, device="cuda")
    disp = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    grad = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    rows = [("sample_maps", None, 24 * C,
             lambda: check(lib.ocean_sample_maps_device(g.context, n, pts.data_ptr(), C, scales.ctypes.data, disp.data_ptr(), grad.data_ptr())))]
    for K in ks:
        rows.append(("query_surface", K, 4 * C * (K + 1) + 20 * C,
                     lambda K=K: check(lib.ocean_query_surface_device(g.context, n, pts.data_ptr(), C, scales.ctypes.data, K, rec.data_ptr()))))
    for op, K, gathers, call in rows:
        reps, ms = time_calls(g, call)
        med = ms[1]
        out = dict(ident, op=op, iterations=K, map_size=N, cascades=C, map_mib=2 * C * N * N * 8 / 2**20, points=n, calls_per_window=reps,
                   us_per_call=1e3 * med, us_per_call_windows=[1e3 * t for t in ms], mpoints_per_s=n / (med * 1e-3) / 1e6,
                   gathers_per_point=gathers, ggathers_per_s=gathers * n / (med * 1e-3) / 1e9)
        if op == "query_surface":
            r = rec.cpu().numpy().view(gow.WaveGenerator.SURFACE_POINT).reshape(-1)
            out["share_residual_le_1mm"] = float(np.mean(r["residual"] <= 1e-3))
        line = json.dumps(out)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
    g.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=2**20)
    ap.add_argument("--out", help="append the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures on the GPU only")
    ident = gpu_identity()
    sink = open(a.out, "a") if a.out else None
    for N, C in ((256, 4), (1024, 8)):
        run(N, C, a.points, (0, 4, 8), ident, sink)
    if sink:
        sink.close()


if __name__ == "__main__":
    main()
