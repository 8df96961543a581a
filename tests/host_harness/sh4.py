"""Builds and binds tests/host_harness/sh4_harness.cpp (test infrastructure, see the .cpp header)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "libegs_sh4_harness.so"
SRC = HERE / "sh4_harness.cpp"
HDR = HERE.parent.parent / "easy_gaussian_splatting_b200" / "csrc" / "egs_math.cuh"


def load():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or LIB.stat().st_mtime < max(SRC.stat().st_mtime, HDR.stat().st_mtime):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                        "-x", "c++", str(SRC), "-o", str(LIB)], check=True)
    return ctypes.CDLL(str(LIB))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def sh4_grads(sc, shs, radii, v_means2d, v_conics, v_colors, eps2d=0.3, v_comps=None):
    """shs: [N,K,3] or per-camera [C,N,K,3], K >= 25.  -> dict of numpy fp32 arrays: colors [C,N,3], v_sh (shape of
    shs), v_means [N,3], v_viewmats [C,4,4], v_Ks [C,3,3]."""
    lib = load()
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    K, per_cam = shs.shape[-2], int(shs.dim() == 4)
    f = lambda t: np.ascontiguousarray(t.detach().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
    arrs = [f(sc.means), f(sc.quats), f(sc.scales), f(shs), f(sc.viewmats), f(sc.Ks), f(v_means2d), f(v_conics),
            f(v_colors)]
    radii = np.ascontiguousarray(radii, dtype=np.int32)
    vc = None if v_comps is None else f(v_comps)
    out = dict(colors=np.zeros((C, N, 3), np.float32), v_sh=np.full(tuple(shs.shape), np.nan, np.float32),
               v_means=np.zeros((N, 3), np.float32), v_viewmats=np.zeros((C, 4, 4), np.float32),
               v_Ks=np.zeros((C, 3, 3), np.float32))
    lib.hh_sh4(C, N, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), K, per_cam, _p(arrs[4]), _p(arrs[5]),
               sc.width, sc.height, ctypes.c_float(eps2d), _p(radii), _p(arrs[6]), _p(arrs[7]), _p(arrs[8]),
               None if vc is None else _p(vc), _p(out["colors"]), _p(out["v_sh"]), _p(out["v_means"]),
               _p(out["v_viewmats"]), _p(out["v_Ks"]))
    return out
