"""In-tree build of libstellar_rhmc.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m hmc_stellar_toy_model_b200.build [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libstellar_rhmc.so")
SOURCES = ["stellar_rhmc.cu", "field_kernels_f64.cu", "field_kernels_f32.cu", "chain_kernels.cu", "ls_kernels.cu", "big_field.cu",
           "misc_kernels.cu", "mock_kernels.cu", "stats_kernels.cu", "peaks_kernels.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMPILE_FLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c"]
# -cudart shared: the library depends on libcudart.so.12 (found through the rpath below or the loader path) instead of
# embedding a static copy of the whole runtime and its entry-point name table
CUDA_LIB = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64")
LINK_FLAGS = ARCH + ["-shared", "-Xcompiler", "-fPIC", "-cudart", "shared", "-Xlinker", "-rpath=" + CUDA_LIB]
OBJ_DIR = os.path.join(HERE, "build")


def _deps():
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "stellar_rhmc.h"))
    return deps


def up_to_date() -> bool:
    if not os.path.isfile(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(d) <= t for d in _deps())


def _stale(obj, src):
    if not os.path.isfile(obj):
        return True
    t = os.path.getmtime(obj)
    heads = [d for d in _deps() if d.endswith((".cuh", ".h"))]
    return any(os.path.getmtime(d) > t for d in heads + [src])


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every translation unit for sm_100a (in parallel) and link libstellar_rhmc.so in-tree."""
    if not force and up_to_date():
        return OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        raise RuntimeError("nvcc not found; cannot build libstellar_rhmc.so")
    os.makedirs(OBJ_DIR, exist_ok=True)
    jobs = []
    for name in SOURCES:
        src = os.path.join(CSRC, name)
        obj = os.path.join(OBJ_DIR, name[:-3] + ".o")
        if force or _stale(obj, src):
            cmd = [nvcc] + COMPILE_FLAGS + ["-o", obj, src]
            jobs.append((name, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log_lines = []
    failed = []
    for name, cmd, proc in jobs:
        out, _ = proc.communicate()
        log_lines.append(" ".join(cmd) + "\n" + out)
        if proc.returncode != 0:
            failed.append((name, out))
    objs = [os.path.join(OBJ_DIR, n[:-3] + ".o") for n in SOURCES]
    if not failed:
        cmd = [nvcc] + LINK_FLAGS + ["-o", OUT + ".tmp"] + objs
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        log_lines.append(" ".join(cmd) + "\n" + proc.stdout)
        if proc.returncode != 0:
            failed.append(("link", proc.stdout))
    log = os.path.join(HERE, "build.log")
    with open(log, "w") as fh:
        fh.write("\n".join(log_lines))
    if verbose:
        print("\n".join(log_lines))
    if failed:
        raise RuntimeError("nvcc failed for %s (see %s):\n%s" % (failed[0][0], log, failed[0][1][-4000:]))
    os.replace(OUT + ".tmp", OUT)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
