"""Builds and binds tests/host_harness/intrinsics_harness.cpp (test infrastructure, see the .cpp header)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "libegs_intrinsics_harness.so"
SRC = HERE / "intrinsics_harness.cpp"
HDR = HERE.parent.parent / "easy_gaussian_splatting_b200" / "csrc" / "egs_math.cuh"


def load():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or LIB.stat().st_mtime < max(SRC.stat().st_mtime, HDR.stat().st_mtime):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                        "-x", "c++", str(SRC), "-o", str(LIB)], check=True)
    return ctypes.CDLL(str(LIB))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def intrinsics_grad(sc, sh_degree, radii, colors, v_means2d, v_conics, v_colors, eps2d=0.3, v_comps=None):
    """-> v_Ks [C,3,3] (numpy fp32) for the cotangents of means2d / conics / colours (/ compensations)."""
    lib = load()
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    K = sc.colors.shape[1] if sc.colors.dim() == 3 else 1
    f = lambda t: np.ascontiguousarray(t.detach().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
    arrs = [f(sc.means), f(sc.quats), f(sc.scales), f(sc.colors), f(sc.viewmats), f(sc.Ks), f(colors), f(v_means2d),
            f(v_conics), f(v_colors)]
    radii = np.ascontiguousarray(radii, dtype=np.int32)
    vc = None if v_comps is None else f(v_comps)
    out = np.full((C, 3, 3), np.nan, np.float32)
    lib.hh_intrinsics_grad(C, N, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), K, sh_degree, _p(arrs[4]),
                           _p(arrs[5]), sc.width, sc.height, ctypes.c_float(eps2d), _p(radii), _p(arrs[6]), _p(arrs[7]),
                           _p(arrs[8]), _p(arrs[9]), None if vc is None else _p(vc), _p(out))
    return out
