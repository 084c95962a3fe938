"""In-tree build of libchaos_b200.so for sm_100a (nvcc cross-compiles without a GPU).

The kernels live in four translation units:
  * tu_parity.cu     -fmad=false : parity env kinds, IEEE two-rounding arithmetic
  * tu_northstar.cu  (fmad on)   : RK4 x S kinds + FMA-peak micro-kernel
  * tu_rl_ops.cu     -fmad=false : SB3 plumbing around the step (GAE, VecNormalize, metrics, ...)
  * tu_policy.cu     -fmad=false : MlpPolicy fused into the hr_sync / pmsm_sync rollout
plus chaos_b200.cu, the C-ABI host side.  The CUDA runtime is linked statically so the
library does not depend on which libcudart PyTorch bundles.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libchaos_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _sources():
    deps = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    deps.append(os.path.join(HERE, "..", "include", "chaos_b200.h"))
    return deps


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _sources())


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    units = [
        ("tu_parity.cu", ["-fmad=false"]),
        ("tu_northstar.cu", []),
        ("tu_rl_ops.cu", ["-fmad=false"]),
        ("tu_policy.cu", ["-fmad=false"]),
        ("chaos_b200.cu", []),
    ]
    def compile_unit(unit):
        src, extra = unit
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
        return obj

    # the translation units are independent: compile them side by side (55 s -> the longest unit)
    with ThreadPoolExecutor(max_workers=len(units)) as pool:
        objs = list(pool.map(compile_unit, units))
    cmd = [nvcc, *ARCH, "-shared", "-cudart", "static", "-o", LIB, *objs]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
