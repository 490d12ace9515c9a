"""Build the CUDA library in-tree with nvcc (sm_100a only).

``python -m ramannoodle_b200._build`` or ``ramannoodle_b200._build.build()``.  The shared
object lands next to this file (``ramannoodle_b200/libramannoodle_b200.so``) so that it
travels with the repo snapshot; nothing is installed into site-packages.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libramannoodle_b200.so")
SOURCES = ["rn_model.cu", "rn_polarizability.cu", "rn_dense.cu", "rn_spectrum.cu", "rn_trajectory.cu", "rn_smear.cu", "rn_rdf.cu", "rn_van_hove.cu", "rn_host.cu", "rn_ingest.cu", "rn_vasprun.cu", "rn_sweep.cu", "rn_dense_sweep.cu"]
HEADERS = [os.path.join(CSRC, "rn_common.cuh"), os.path.join(CSRC, "rn_device.cuh"), os.path.join(CSRC, "rn_dense_tp.cuh"),
           os.path.join(CSRC, "rn_fft.cuh"), os.path.join(CSRC, "rn_spectrum_plan.cuh"), os.path.join(CSRC, "rn_textparse.hpp"),
           os.path.join(os.path.dirname(HERE), "include", "ramannoodle_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; the CUDA library cannot be built")
    return nvcc


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    stamp = os.path.getmtime(target)
    return any(os.path.getmtime(d) > stamp for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every ``.cu`` for sm_100a and link ``libramannoodle_b200.so``."""
    os.makedirs(BUILD, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + HEADERS):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", path, "-o", obj]
            res = subprocess.run(cmd, capture_output=True, text=True)
            with open(obj.replace(".o", ".ptxas.log"), "w", encoding="utf-8") as log:
                log.write(res.stdout + res.stderr)
            if res.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
            if verbose:
                print(f"compiled {src}", file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        objects = list(pool.map(compile_one, SOURCES))
    if force or _stale(LIB, objects):
        cmd = [nvcc, "-shared", "-o", LIB] + objects + ["-gencode", "arch=compute_100a,code=sm_100a", "-lpthread"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
