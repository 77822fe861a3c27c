"""Build ``libdiffus_b200.so`` in-tree with nvcc for sm_100a (no torch, no pybind: a plain C-ABI library)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libdiffus_b200.so")
# (source, extra flags, object): render_kernels.cu is compiled once per volume layout (its 100+ kernel instantiations
# are most of the build time) plus once for the dispatching entry points and the echo-only kernels
SOURCES = [("render_kernels.cu", ["-DDIFFUS_LAYOUT_SLICE=1"], "render_kernels_brick.o"),
           ("render_kernels.cu", ["-DDIFFUS_LAYOUT_SLICE=0"], "render_kernels_linear.o"),
           ("render_kernels.cu", ["-DDIFFUS_LAYOUT_SLICE=2"], "render_kernels_quad.o"),
           ("render_kernels.cu", ["-DDIFFUS_LAYOUT_SLICE=3"], "render_kernels_texture.o"),
           ("aux_kernels.cu", [], "aux_kernels.o"), ("render_kernels.cu", [], "render_kernels.o"),
           ("api.cu", [], "api.o"), ("mlp_kernels.cu", [], "mlp_kernels.o"),
           ("mlp_pwl_kernels.cu", [], "mlp_pwl_kernels.o"),
           ("splat_kernels.cu", [], "splat_kernels.o"), ("preprocess_kernels.cu", [], "preprocess_kernels.o"),
           ("train_kernels.cu", [], "train_kernels.o"), ("loss_kernels.cu", [], "loss_kernels.o"),
           ("gn_kernels.cu", [], "gn_kernels.o"), ("smooth_kernels.cu", [], "smooth_kernels.o")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--threads", "2"]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libdiffus_b200.so cannot be built")
    return nvcc


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "diffus_b200.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    os.makedirs(BUILD, exist_ok=True)

    def compile_one(item):
        src, extra, objname = item
        obj = os.path.join(BUILD, objname)
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 4)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
