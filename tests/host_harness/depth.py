"""Builds and binds tests/host_harness/depth_harness.cpp (test infrastructure, see the .cpp header)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "libegs_depth_harness.so"
SRC = HERE / "depth_harness.cpp"
HDR = HERE.parent.parent / "easy_gaussian_splatting_b200" / "csrc" / "egs_math.cuh"


def load():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or LIB.stat().st_mtime < max(SRC.stat().st_mtime, HDR.stat().st_mtime):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                        "-x", "c++", str(SRC), "-o", str(LIB)], check=True)
    return ctypes.CDLL(str(LIB))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def depth_grad(sc, radii, v_means2d, v_depths, v_conics, eps2d=0.3, v_comps=None):
    """-> (v_means [N,3], v_viewmats [C,4,4], v_Ks [C,3,3]) (numpy fp32) for the cotangents of means2d, depths, conics
    (and compensations) of the visible pairs."""
    lib = load()
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    f = lambda t: np.ascontiguousarray(t.detach().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
    arrs = [f(sc.means), f(sc.quats), f(sc.scales), f(sc.viewmats), f(sc.Ks), f(v_means2d), f(v_depths), f(v_conics)]
    radii = np.ascontiguousarray(radii, dtype=np.int32)
    vc = None if v_comps is None else f(v_comps)
    v_means = np.full((N, 3), np.nan, np.float32)
    v_vm = np.full((C, 4, 4), np.nan, np.float32)
    v_ks = np.full((C, 3, 3), np.nan, np.float32)
    lib.hh_depth_grad(C, N, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), _p(arrs[4]), sc.width, sc.height,
                      ctypes.c_float(eps2d), _p(radii), _p(arrs[5]), _p(arrs[6]), _p(arrs[7]),
                      None if vc is None else _p(vc), _p(v_means), _p(v_vm), _p(v_ks))
    return v_means, v_vm, v_ks
