"""Builds libtriro_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Replaces the reference's two-stage build: `nvcc -optix-ir` of shaders.cu at install time
(setup.py:27-39) plus the JIT compile of base.cpp/binding.cpp/ray.cpp at first import
(triro/backend/ops.py:24-45).  Here there is one ahead-of-time build and no OptiX SDK.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.normpath(os.path.join(HERE, "..", "..", "csrc"))
INCLUDE = os.path.normpath(os.path.join(HERE, "..", "..", "..", "include"))
LIB_PATH = os.path.join(HERE, "libtriro_b200.so")
UNITS = ["rt_build.cu", "rt_trace.cu", "rt_compact.cu", "rt_host.cu", "rt_closest.cu", "rt_winding.cu", "rt_pseudonormal.cu", "rt_distgrad.cu", "rt_scene.cu", "rt_scene_point.cu", "rt_scene_grad.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (looked at $NVCC, /usr/local/cuda/bin/nvcc, PATH)")


def sources() -> list[str]:
    out = [os.path.join(CSRC, u) for u in UNITS]
    out += [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".h"))]
    out.append(os.path.join(INCLUDE, "raymesh_b200.h"))
    return out


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force: bool = False, verbose: bool = False, variant: str | None = None, extra: list[str] | None = None) -> str:
    """Compile every translation unit (in parallel) and link the shared library.
    `variant` + `extra` nvcc flags build an experiment library next to it (libtriro_b200_<variant>.so, selected with
    TRIRO_B200_LIB); the product is the plain build."""
    lib_path = LIB_PATH if variant is None else os.path.join(HERE, f"libtriro_b200_{variant}.so")
    if variant is None and not force and not is_stale():
        return LIB_PATH
    nvcc = nvcc_path()
    objdir = os.path.join(CSRC, "build" if variant is None else f"build_{variant}")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(unit: str) -> str:
        obj = os.path.join(objdir, unit.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *NVCC_FLAGS, *os.environ.get("TRIRO_NVCC_EXTRA", "").split(), *(extra or []), "-I", INCLUDE, "-c",
               os.path.join(CSRC, unit), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {unit}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(compile_one, UNITS))
    tmp = lib_path + ".tmp"
    r = subprocess.run([nvcc, *ARCH, "-shared", "-o", tmp, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib_path)
    return lib_path


if __name__ == "__main__":
    import sys

    var = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant=var[0] if var else None,
                extra=[a for a in sys.argv[1:] if a.startswith("-D")]))
