"""Build libpds_b200 in-tree with nvcc for sm_100a (no torch involved: the library only needs the CUDA runtime).

    python -m polars_ds_extension_b200.build          # incremental
    python -m polars_ds_extension_b200.build --force

Output: polars_ds_extension_b200/_polars_ds_b200.so (git-ignored; travels to the GPU box with gpurun).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
OBJ = PKG / "_build"
LIB = PKG / "_polars_ds_b200.so"

SOURCES = [
    "kernels/k1_pack.cu",
    "kernels/k2_gram_simt.cu",
    "kernels/k2_gram_tcgen05.cu",
    "kernels/k3_solve.cu",
    "kernels/k4_predict.cu",
    "kernels/k5_grouped.cu",
    "kernels/k6_online.cu",
    "kernels/k9_report.cu",
    "kernels/k10_models.cu",
    "kernels/k11_logistic.cu",
    "host/context.cc",
    "host/api_dev.cc",
    "host/h2d.cc",
    "host/multi_gpu.cc",
    "host/lr_host.cc",
    "host/models_host.cc",
    "host/glm_host.cc",
    "abi/plugin.cc",
]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=default,-Wall,-Wno-unused-function",
          "-I", str(ROOT / "include"), "--expt-relaxed-constexpr", "-x", "cu"]


def _headers_mtime() -> float:
    m = 0.0
    for p in list(CSRC.rglob("*.h")) + list(CSRC.rglob("*.cuh")) + list((ROOT / "include").glob("*.h")):
        m = max(m, p.stat().st_mtime)
    return m


def _compile(src: str, force: bool, hm: float, verbose: bool) -> Path:
    s = CSRC / src
    o = OBJ / (src.replace("/", "_") + ".o")
    if not force and o.exists() and o.stat().st_mtime > max(s.stat().st_mtime, hm):
        return o
    cmd = [NVCC, *ARCH, *COMMON, *os.environ.get("PDSB_EXTRA_NVCC_FLAGS", "").split(), "-c", str(s), "-o", str(o)]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    if verbose or r.stderr.strip():
        sys.stderr.write(f"--- {src}\n{r.stderr}\n")
    return o


def build(force: bool = False, verbose: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    hm = _headers_mtime()
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 4)) as ex:
        objs = list(ex.map(lambda s: _compile(s, force, hm, verbose), SOURCES))
    if force or not LIB.exists() or any(o.stat().st_mtime > LIB.stat().st_mtime for o in objs):
        cmd = [NVCC, *ARCH, "-shared", "-o", str(LIB), *map(str, objs), "-cudart", "static", "-lpthread", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
