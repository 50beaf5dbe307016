#!/usr/bin/env python
"""bench.py -- throughput of the wave-generation hot path (spectrum propagation -> 4 packed N x N
inverse FFTs -> displacement/normal/foam maps) on B200, per the driver contract.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      (CPU arm: the oracle on the host cores)

One "step" = one batched update of every cascade resident on a GPU (default workload: BASELINE.json
configs[1], 256x256 x 4 cascades, batched as --sets independent 4-cascade sets per GPU so that the
working set, 40 B/texel algorithmic + 64 B/texel scratch, exceeds the 126 MB L2).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_BYTES_PER_TEXEL = 40.0       # SURVEY 8d: read h0 16 + read foam texel 8 + write 2 x RGBA16F 16
METRIC = "ifft_cascades_per_sec"
UNIT = "cascades/s"
DUMP_BYTES = 32 * 2**20           # --dump-outputs budget: one 1024x1024 cascade (both maps as float32) fits it

DEMO_SETS = [   # main.tscn:43-83 + wave_cascade_parameters.gd defaults (SURVEY appendix B)
    dict(tile_length=(88.0, 88.0), displacement_scale=1.0, normal_scale=1.0, wind_speed=10.0, wind_direction=20.0,
         fetch_length=150.0, swell=0.8, spread=0.2, detail=1.0, whitecap=0.5, foam_amount=8.0),
    dict(tile_length=(57.0, 57.0), displacement_scale=0.75, normal_scale=1.0, wind_speed=5.0, wind_direction=15.0,
         fetch_length=150.0, swell=0.8, spread=0.4, detail=1.0, whitecap=0.5, foam_amount=0.0),
    dict(tile_length=(16.0, 16.0), displacement_scale=0.0, normal_scale=0.25, wind_speed=20.0, wind_direction=20.0,
         fetch_length=550.0, swell=0.8, spread=0.4, detail=1.0, whitecap=0.25, foam_amount=3.0),
    dict(tile_length=(50.0, 50.0), displacement_scale=1.0, normal_scale=1.0, wind_speed=20.0, wind_direction=0.0,
         fetch_length=550.0, swell=0.8, spread=0.2, detail=1.0, whitecap=0.5, foam_amount=5.0),
]


def synth_params(cls, global_index: int):
    """Synthetic workload of SURVEY 8d: demo parameter sets cycled, fixed integer seeds, time0 = 120 + pi*c."""
    kw = dict(DEMO_SETS[global_index % len(DEMO_SETS)])
    kw.update(spectrum_seed=(1234 + 17 * global_index, -5678 + 31 * global_index),
              time=120.0 + math.pi * (global_index % 8))
    return cls(**kw)


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the newest committed ncu capture (profiles/*traffic*.json)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*traffic*.json")))
    if not files:
        return None, None
    try:
        with open(files[-1]) as f:
            t = json.load(f)
        return float(t["dram_bytes_per_launch"]), os.path.relpath(files[-1], ROOT)
    except Exception:
        return None, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.002)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


_RESULT_OUT = sys.stdout        # replaced in main(): the real stdout, kept apart from library chatter


def host_threads() -> tuple[int, str]:
    """Threads the CPU arm uses: one per PHYSICAL core this process may run on (affinity mask, SMT siblings counted
    once), capped by the cgroup CPU quota when the container has one."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                cores.add(f.read().strip())
        except OSError:
            cores.add(str(c))
    n = max(1, len(cores))
    how = f"{n} physical cores of {len(cpus)} logical CPUs in the affinity mask"
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            q = max(1, int(float(quota) / float(period)))
            if q < n:
                n, how = q, how + f", capped by the cgroup quota of {q} CPUs"
    except (OSError, ValueError):
        pass
    return n, how


def cpu_arm(map_size: int, cascades: int, steps: int, warmup: int, budget_s=None, kind=None):
    """The reference's CPU implementation of the path on the host cores, on the GPU arm's own workload (`cascades`
    cascade updates per step).  kind "reference" = oracle/_ref, the reference's six GLSL compute shaders compiled for the
    CPU (OpenMP over workgroups inside every dispatch); kind "port" = the C oracle, one OpenMP thread per cascade.
    Every step is timed on its own; the value is cascades / MEDIAN step time after `warmup` untimed steps.
    Returns a dict for the JSON line."""
    from oracle import pyoracle as po
    from oracle import pyref as pr
    if kind is None:
        kind = "reference" if pr.available() else "port"
    threads, how = host_threads()
    params = [synth_params(po.CascadeParams, c) for c in range(cascades)]
    if kind == "reference":
        pr.set_modes(po.MATH_DET, po.CONTRACT_FMA)
        pr.lib().ref_set_num_threads(threads)
        gen = pr.RefWaveGenerator(map_size)
        gen.init_gpu(cascades)
        step = lambda: gen.update_all(1.0 / 50.0, params)
        what = "oracle/_ref (the reference's GLSL compute shaders compiled for the CPU, OpenMP over workgroups)"
    else:
        po.set_modes(po.MATH_DET, po.CONTRACT_FMA)
        po.lib().oracle_set_num_threads(threads)
        gen = po.OracleWaveGenerator(map_size)
        gen.keep_f32 = False
        gen.init_gpu(cascades)
        step = lambda: gen.update_all_batched(1.0 / 50.0, params)
        what = "C oracle port (oracle/ocean_oracle.c, one OpenMP thread per cascade)"
    t_begin = time.perf_counter()
    for _ in range(max(1, warmup)):          # the first step also generates the spectra (not steady state)
        step()
    times = []
    while len(times) < steps:
        t = time.perf_counter()
        step()
        times.append(time.perf_counter() - t)
        if budget_s is not None and len(times) >= 3 and time.perf_counter() - t_begin >= budget_s:
            break
    ts = sorted(times)
    med = ts[len(ts) // 2]
    return {"value": cascades / med, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{len(times)} steady-state steps of {cascades} cascades at {map_size}x{map_size} after {max(1, warmup)} warm-up steps: {what}; "
                      f"threads = {how}; OMP_PROC_BIND=close OMP_PLACES=cores OMP_WAIT_POLICY=passive",
            "seconds_per_step": {"median": med, "min": ts[0], "max": ts[-1], "spread": (ts[-1] - ts[0]) / med},
            "steps": len(times)}


def workload_config(args, world: int) -> dict:
    """The `config` object of both arms (the reference arm runs the same per-GPU workload on the host cores)."""
    N = args.map_size
    C = args.sets * args.cascades_per_set
    return {"workload": f"{N}x{N} x {args.cascades_per_set} cascades, full pipeline incl. foam, {args.sets} independent sets per GPU per step",
            "map_size": N, "cascades_per_set": args.cascades_per_set, "sets_per_gpu": args.sets,
            "cascades_per_step_per_gpu": C, "parallelism": f"cascade-sharded x{world}, no data-path collective",
            "l2": (lambda mib: f"working set {mib:.0f} MiB per step " + ("> 126 MB L2 (inputs larger than L2)" if mib * 2**20 > 126e6
                                                                         else "fits the 126 MB L2 (NOT an HBM-bound measurement)"))(
                (ALGO_BYTES_PER_TEXEL + 64) * C * N * N / 2**20)}


def sample_outputs(gen, C: int, N: int) -> dict:
    """What the last update_all() handed its caller: both RGBA16F maps, widened to float32 (exact), of every resident
    cascade when they fit DUMP_BYTES, else of a fixed seeded choice of cascades (in ascending order)."""
    import numpy as np
    k = max(1, min(C, DUMP_BYTES // (2 * N * N * 4 * 4)))
    pick = np.sort(np.random.default_rng(0).choice(C, size=k, replace=False))
    out = {"displacement_map": np.empty((k, N, N, 4), np.float32), "normal_map": np.empty((k, N, N, 4), np.float32)}
    for j, c in enumerate(pick):
        d, n = gen.maps_to_host(int(c), 1)
        out["displacement_map"][j] = d[0]
        out["normal_map"][j] = n[0]
    return out


def run_reference(args, rank: int):
    if rank != 0:
        return
    C = args.sets * args.cascades_per_set
    # exactly --steps timed steps after --warmup (>= 3) untimed ones, each step the GPU arm's whole per-GPU workload; the time
    # budget only guards against a host far slower than expected (the line then reports the steps it did time)
    cb = cpu_arm(args.map_size, C, args.steps, args.warmup, budget_s=args.reference_seconds)
    cps = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": cps, "unit": UNIT, "n_gpus": args.gpus, "steps": cb["steps"],
        "warmup": args.warmup, "ms_per_step": cb["seconds_per_step"]["median"] * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "mtexels_per_sec": cps * args.map_size * args.map_size / 1e6,
        "cpu_baseline": cb,
        "e2e": {"value": cps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference project itself (Godot + Vulkan/lavapipe) cannot run in this image; its compute shaders can: "
                "this arm runs them, compiled for the CPU, on the host cores",
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


def bind_to_gpu_numa_node(index: int):
    """Pins this rank to the CPUs next to its GPU (NVML's ideal CPU affinity for the device), so that the pinned host
    buffers it allocates afterwards are local to the GPU's PCIe root and the ranks do not all land on one memory controller."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        return {"bound": True, "cpus_before": before, "cpus_after": len(after), "first_cpu": after[0], "last_cpu": after[-1]}
    except Exception as e:                       # no NVML / not permitted: run unbound and say so
        return {"bound": False, "why": str(e)[:120]}


def preflight_sharding_check(world: int, local_rank: int, dist):
    """SURVEY 8e: cascade-sharded over the GPUs of this job == one GPU, bit for bit.  Every rank runs its shard of a small
    workload through the sharded path and, on its own GPU, the whole workload through a single generator; rank 0 gathers the
    CRCs.  Costs well under a second; the result travels in the JSON line."""
    import zlib
    import numpy as np
    import godotoceanwaves_b200 as gow
    from godotoceanwaves_b200.sharding import ShardedWaveGenerator, owned_cascades
    N, C, frames = 128, 16, 3
    rank = int(os.environ.get("RANK", "0"))
    params = [synth_params(gow.WaveCascadeParameters, c) for c in range(C)]
    sh = ShardedWaveGenerator(N, rank=rank, world=world, device=local_rank)
    for _ in range(frames):
        sh.update_all(1.0 / 50.0, params)
    d, n = sh.local_maps_to_host()
    mine = {c: (zlib.crc32(d[k].tobytes()), zlib.crc32(n[k].tobytes())) for k, c in enumerate(owned_cascades(C, rank, world))}
    sh.free()
    ref_params = [synth_params(gow.WaveCascadeParameters, c) for c in range(C)]
    ref = gow.WaveGenerator(device=local_rank); ref.map_size = N; ref.init_gpu(C)
    for _ in range(frames):
        ref.update_all(1.0 / 50.0, ref_params)
    rd, rn = ref.maps_to_host()
    ref.free()
    ok = all(mine[c] == (zlib.crc32(rd[c].tobytes()), zlib.crc32(rn[c].tobytes())) for c in mine)
    if world > 1:
        flags = [None] * world
        dist.all_gather_object(flags, (ok, len(mine)))
        ok = all(f[0] for f in flags)
        covered = sum(f[1] for f in flags)
    else:
        covered = len(mine)
    if not ok or covered != C:
        raise SystemExit(f"sharding pre-flight FAILED on rank {rank}: sharded maps differ from the single-GPU maps")
    return {"ok": True, "what": f"{C} cascades of {N}x{N}, {frames} updates: round-robin over {world} GPU(s) == one GPU, CRC-32 of both RGBA16F maps per cascade"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--map-size", type=int, default=256)
    ap.add_argument("--cascades-per-set", type=int, default=4)
    ap.add_argument("--sets", type=int, default=32, help="independent cascade sets resident per GPU")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="CPU-baseline sample budget inside the native arm")
    ap.add_argument("--reference-seconds", type=float, default=240.0, help="time budget of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the maps of the last timed step (rank 0's cascades, a seeded sample of them beyond 32 MiB) "
                         "as DIR/<name>.npy in float32")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4-strong"],
                    help="cfg2: BASELINE configs[1], weak scaling (default, the driver's contract); cfg4-strong: BASELINE configs[3], "
                         "1024x1024 x 8 cascades split over the GPUs (8/4/2/1 per GPU), strong scaling")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    # the CPU arm's OpenMP runtime: threads pinned to cores, sleeping (not spinning) between parallel regions -- must be in
    # the environment before the first OpenMP library is loaded
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")

    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner at every debug
    # level above NONE), so file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved stdout.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import godotoceanwaves_b200 as gow
    from godotoceanwaves_b200 import build as native_build

    native_build.build_native()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback for the native arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    numa = bind_to_gpu_numa_node(local_rank)              # before any pinned allocation: host buffers land next to the GPU
    strong = args.workload == "cfg4-strong"
    if strong:
        args.map_size, args.cascades_per_set, args.sets = 1024, 8, 1
        if 8 % world:
            raise SystemExit("cfg4-strong splits 8 cascades: --gpus must be 1, 2, 4 or 8")
    N = args.map_size
    total_cascades = (args.sets * args.cascades_per_set) if strong else world * args.sets * args.cascades_per_set
    C = total_cascades // world                            # cascades resident on this GPU
    texels_per_step = C * N * N
    sharding_check = preflight_sharding_check(world, local_rank, dist if world > 1 else None)
    # cascade-parallel split (SURVEY 8e): the global batch of world*C cascades is dealt round-robin over the
    # ranks, every rank keeps its C cascades resident; no data-path collective.
    from godotoceanwaves_b200.sharding import ShardedWaveGenerator
    all_params = [synth_params(gow.WaveCascadeParameters, c) for c in range(total_cascades)]
    shard = ShardedWaveGenerator(N, rank=rank, world=world, device=local_rank)
    shard.update_all(1.0 / 50.0, all_params)      # creates the local generator and the spectra
    gen = shard.gen
    params = [all_params[i] for i in shard.owned]
    assert len(params) == C
    delta = 1.0 / 50.0

    # ---- warm-up (first step also generates the spectra) ----
    for _ in range(args.warmup):
        gen.update_all(delta, params)
    gen.synchronize()

    # ---- device-timed region: inputs resident in HBM, CUDA events on the launching stream ----
    sampler = ClockSampler(local_rank)
    launches0 = gen.info().kernel_launches
    barrier()
    sampler.start()
    gen.timer_start()
    for _ in range(args.steps):
        gen.update_all(delta, params)
    ms = gen.timer_stop()
    # read before the untimed updates below advance the state
    outputs = sample_outputs(gen, C, N) if args.dump_outputs and rank == 0 else None
    if len(sampler.samples) < 5:
        # the timed region is only tens of milliseconds and the submitting thread rarely yields the GIL: keep the
        # same workload running (untimed) for ~0.5 s so that NVML sees the clocks under this load
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            gen.update_all(delta, params)
            time.sleep(0.0005)
        gen.synchronize()
    clocks = sampler.stop()
    barrier()
    launches = gen.info().kernel_launches - launches0
    ms = max_over_ranks(ms)
    value = total_cascades * args.steps / (ms * 1e-3)

    # ---- per-kernel times (CUDA events between the two kernels), averaged over a few steps ----
    gen.set_profiling(True)
    ka = kb = 0.0
    reps = min(args.steps, 20)
    for _ in range(reps):
        gen.update_all(delta, params)
        _, a, b, kchunk = gen.last_kernel_times()
        ka += a
        kb += b
    gen.set_profiling(False)
    ka, kb = ka / reps, kb / reps

    # ---- end to end through the public API with host buffers: params H2D + both maps D2H every step ----
    lib = gow.load_library()
    import ctypes as Ct
    map_bytes = C * N * N * 8
    hd, hn = Ct.c_void_p(), Ct.c_void_p()
    gow.native.check(lib.ocean_host_alloc(Ct.byref(hd), map_bytes))
    gow.native.check(lib.ocean_host_alloc(Ct.byref(hn), map_bytes))
    e2e_steps = max(3, min(args.steps, 20))
    hd2, hn2 = Ct.c_void_p(), Ct.c_void_p()
    gow.native.check(lib.ocean_host_alloc(Ct.byref(hd2), map_bytes))
    gow.native.check(lib.ocean_host_alloc(Ct.byref(hn2), map_bytes))
    host = [(hd, hn), (hd2, hn2)]
    for i in range(2):
        gen.update_all(delta, params)
        gow.native.check(lib.ocean_snapshot_maps_to_host_async(gen.context, 0, C, host[i][0], host[i][1]))
    gow.native.check(lib.ocean_wait_snapshot(gen.context))
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        gen.update_all(delta, params)                                          # marshals + uploads dispatch records
        # the maps of this step are snapshotted on the device and cross PCIe on a second stream while the next update runs;
        # the host buffer they land in was last used two steps ago (the snapshot call waits for the previous hand-off)
        gow.native.check(lib.ocean_snapshot_maps_to_host_async(gen.context, 0, C, host[i & 1][0], host[i & 1][1]))
    gow.native.check(lib.ocean_wait_snapshot(gen.context))                      # every step's result is on the host
    gen.synchronize()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = total_cascades * e2e_steps / e2e_s
    # host -> device per step: the dispatch records travel BY VALUE as kernel parameters of the one launch (a 256-record table
    # of 32 B records is always sent whole, plus the queue descriptor and the 128 B tensor map)
    h2d_bytes = 256 * 32 + 128 + 96
    d2h_bytes = 2 * map_bytes
    probe = np.frombuffer((Ct.c_uint16 * 4).from_address(hd.value), np.float16)
    assert np.all(np.isfinite(probe.astype(np.float32)))
    for a, b in host:
        gow.native.check(lib.ocean_host_free(a))
        gow.native.check(lib.ocean_host_free(b))
    gen.free()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    peak_gbs, peak_src = measured_peaks()
    traffic, traffic_src = ncu_traffic()
    if not (N == 256 and C == 128):
        traffic, traffic_src = None, None          # the capture is of the default workload only
    step_s = ms * 1e-3 / args.steps
    achieved = ALGO_BYTES_PER_TEXEL * texels_per_step / step_s / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "mtexels_per_sec": value * N * N / 1e6,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "traffic_kind": "static: dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu --set full capture, not measured in this run",
                     "peak_source": peak_src,
                     "kernel": "k_update_persistent (one launch per step: time propagation + row IFFT items and column IFFT + map items)",
                     "algorithmic_bytes_per_step": ALGO_BYTES_PER_TEXEL * texels_per_step,
                     "kernel_ms": {"k_modulate_rowfft": ka, "k_colfft_unpack": kb, "cascades_per_launch": kchunk}},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": e2e_s * 1e3 / e2e_steps, "steps": e2e_steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "sharding_check": sharding_check,
        "host_binding": numa,
    }
    if strong:
        line["config"]["workload"] = f"BASELINE configs[3]: 1024x1024 x 8 cascades batched across {world} GPU(s), {C} per GPU (strong scaling)"
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_arm(N, C, 10, 3, budget_s=args.cpu_seconds)
    print(json.dumps(line), file=_RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
