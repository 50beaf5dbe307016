"""Builds libocean.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libocean.so")
SOURCES = ["ocean_kernels.cu", "ocean_sample.cu", "ocean_spray.cu", "ocean_surface.cu", "ocean_api.cu"]
HEADERS = ["ocean_kernels.cuh", "ocean_texture.cuh", "detmath.cuh", "fft_core.cuh", os.path.join("..", "..", "include", "ocean.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                      # no implicit contraction: every FMA in the kernels is explicit
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libocean.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_native(force: bool = False, verbose: bool = False, out: str | None = None, defines=()) -> str:
    """Compile csrc/*.cu into godotoceanwaves_b200/libocean.so. No-op when up to date.
    `out`/`defines` build a tuning variant next to it (loaded with OCEAN_LIB=...)."""
    if out is None and not force and not is_stale():
        return LIB_PATH
    target = out or LIB_PATH
    # several ranks of one job may get here together: one builds (into a temporary file, renamed into place), the others
    # wait on the lock and then find the library up to date
    import fcntl
    with open(target + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if out is None and not force and not is_stale():
                return LIB_PATH
            tmp = f"{target}.tmp{os.getpid()}"
            cmd = [_nvcc(), *NVCC_FLAGS, *[f"-D{d}" for d in defines], "-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
            if os.path.exists("/usr/bin/g++"):
                cmd[1:1] = ["-ccbin", "/usr/bin/g++"]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + res.stdout)
            os.replace(tmp, target)
            if verbose:
                print(res.stdout)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return target


if __name__ == "__main__":
    import sys
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
