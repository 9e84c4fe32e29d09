"""Build the sm_100a shared library in-tree (nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
# one translation unit per stage (csrc/sfm_host.h); the .cpp files are host only and go straight to the host compiler
TUS = ["sfm_api.cu", "sfm_ransac.cu", "sfm_two_view.cu", "sfm_model_select.cu", "sfm_front_end.cu", "sfm_nccl.cpp",
       "sfm_sampler.cpp"]
OBJ_DIR = os.path.join(HERE, "..", "build", "sfm_b200")
SO = os.path.join(HERE, "libsfm_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = [*ARCH, "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libsfm_b200.so")


def sources():
    d = os.path.join(HERE, "csrc")
    return [os.path.join(d, f) for f in sorted(os.listdir(d))] + [
        os.path.join(HERE, "..", "include", "sfm_b200.h")
    ]


def is_stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(s) > t for s in sources() if os.path.exists(s))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every translation unit to an object in parallel (any newer source rebuilds all), then link once."""
    if not force and not is_stale():
        return SO
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs = [os.path.join(OBJ_DIR, os.path.splitext(tu)[0] + ".o") for tu in TUS]

    def compile_one(tu, obj):
        cmd = [nvcc, *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-c", "-o", obj,
               os.path.join(HERE, "csrc", tu)]
        return cmd, subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)

    with ThreadPoolExecutor(max_workers=len(TUS)) as pool:
        results = list(pool.map(compile_one, TUS, objs))
    for cmd, res in results:  # in a fixed order, so that -v output and errors do not interleave
        sys.stdout.write(res.stdout)
        if res.returncode:
            raise subprocess.CalledProcessError(res.returncode, cmd, res.stdout)
    subprocess.check_call([nvcc, *ARCH, "-shared", "-o", SO + ".tmp", *objs])
    os.replace(SO + ".tmp", SO)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
