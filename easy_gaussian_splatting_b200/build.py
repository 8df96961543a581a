"""Builds csrc/*.cu into easy_gaussian_splatting_b200/_C/libegs_raster.so with nvcc for sm_100a.

In-tree build (the .so travels to the GPU box with the repo snapshot; it is git-ignored).
``python -m easy_gaussian_splatting_b200.build [--force] [--verbose]``.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OUT_DIR = PKG / "_C"
LIB = OUT_DIR / "libegs_raster.so"
INCLUDE = PKG.parent / "include"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
          "-Xptxas", "-v", f"-I{INCLUDE}"]
# Translation units whose fp32 results must be bit-identical to the oracle: no FMA contraction,
# IEEE division / sqrt (nvcc defaults), no fast-math.
EXACT_UNITS = {"projection.cu", "projection_ortho.cu", "projection_fisheye.cu", "binning.cu"}
# FP32-throughput-bound units: FMA contraction on, fast intrinsics are explicit in the source.
FLAGS = {
    "projection.cu": ["-fmad=false"],
    "projection_ortho.cu": ["-fmad=false"],
    "projection_fisheye.cu": ["-fmad=false"],
    "binning.cu": ["-fmad=false"],
}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _sources():
    return sorted(CSRC.glob("*.cu"))


def _digest() -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [INCLUDE / "egs_raster.h", Path(__file__)]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()


def needs_build() -> bool:
    stamp = OUT_DIR / "build.stamp"
    return not (LIB.exists() and stamp.exists() and stamp.read_text().strip() == _digest())


def build(force: bool = False, verbose: bool = False) -> Path:
    override = os.environ.get("EGS_RASTER_LIB")  # development only: an A/B variant from scripts/build_variant.py
    if override:
        if not Path(override).exists():
            raise RuntimeError(f"EGS_RASTER_LIB={override} does not exist")
        return Path(override)
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    OUT_DIR.mkdir(exist_ok=True)
    objdir = OUT_DIR / "obj"
    objdir.mkdir(exist_ok=True)
    logs = []

    def compile_one(src: Path):
        obj = objdir / (src.stem + ".o")
        cmd = [nvcc, *ARCH, *COMMON, *FLAGS.get(src.name, []), "-c", str(src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        logs.append((src.name, r.stdout + r.stderr))
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _sources()))
    cmd = [nvcc, *ARCH, "-shared", "-o", str(LIB), *map(str, objs), "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    (OUT_DIR / "ptxas.log").write_text("\n".join(f"==== {n} ====\n{t}" for n, t in sorted(logs)))
    (OUT_DIR / "build.stamp").write_text(_digest())
    if verbose:
        print((OUT_DIR / "ptxas.log").read_text())
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(p)
