"""Builds and binds tests/host_harness/camera_model_harness.cpp (test infrastructure, see the .cpp header)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "_build" / "libegs_camera_model_harness.so"
SRC = HERE / "camera_model_harness.cpp"
HDR = HERE.parent.parent / "easy_gaussian_splatting_b200" / "csrc" / "egs_math.cuh"

MODELS = {"pinhole": 0, "ortho": 1, "fisheye": 2}


def load():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or LIB.stat().st_mtime < max(SRC.stat().st_mtime, HDR.stat().st_mtime):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                        "-x", "c++", str(SRC), "-o", str(LIB)], check=True)
    return ctypes.CDLL(str(LIB))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _f(t):
    return np.ascontiguousarray(t.detach().numpy() if hasattr(t, "detach") else t, dtype=np.float32)


def projection_fwd(model, means, quats, scales, viewmats, Ks, width, height, eps2d=0.3, near=0.01, far=1e10, clip=0.0):
    """-> dict radii, means2d, depths, conics, compensations (numpy) of the host-compiled project_fwd<model>."""
    lib = load()
    C, N = viewmats.shape[0], means.shape[0]
    arrs = [_f(t) for t in (means, quats, scales, viewmats, Ks)]
    out = dict(radii=np.zeros((C, N), np.int32), means2d=np.zeros((C, N, 2), np.float32),
               depths=np.zeros((C, N), np.float32), conics=np.zeros((C, N, 3), np.float32),
               compensations=np.zeros((C, N), np.float32))
    lib.hh_cm_fwd(MODELS[model], C, N, *[_p(a) for a in arrs], int(width), int(height), ctypes.c_float(eps2d),
                  ctypes.c_float(near), ctypes.c_float(far), ctypes.c_float(clip), _p(out["radii"]), _p(out["means2d"]),
                  _p(out["depths"]), _p(out["conics"]), _p(out["compensations"]))
    return out


def projection_bwd(model, means, quats, scales, viewmats, Ks, width, height, radii, v_means2d, v_depths, v_conics,
                   eps2d=0.3, v_comps=None):
    """-> dict v_means, v_quats, v_scales, v_viewmats [C,4,4], v_Ks [C,3,3] (numpy fp32)."""
    lib = load()
    C, N = viewmats.shape[0], means.shape[0]
    arrs = [_f(t) for t in (means, quats, scales, viewmats, Ks)]
    cot = [_f(t) for t in (v_means2d, v_depths, v_conics)]
    radii = np.ascontiguousarray(radii, dtype=np.int32)
    vc = None if v_comps is None else _f(v_comps)
    out = dict(v_means=np.full((N, 3), np.nan, np.float32), v_quats=np.full((N, 4), np.nan, np.float32),
               v_scales=np.full((N, 3), np.nan, np.float32), v_viewmats=np.full((C, 4, 4), np.nan, np.float32),
               v_Ks=np.full((C, 3, 3), np.nan, np.float32))
    lib.hh_cm_bwd(MODELS[model], C, N, *[_p(a) for a in arrs], int(width), int(height), ctypes.c_float(eps2d), _p(radii),
                  *[_p(a) for a in cot], None if vc is None else _p(vc), _p(out["v_means"]), _p(out["v_quats"]),
                  _p(out["v_scales"]), _p(out["v_viewmats"]), _p(out["v_Ks"]))
    return out


def theta_over_r(r, z):
    """-> (s, g) of fisheye_theta_over_r for fp32 arrays r >= 0, z."""
    lib = load()
    r, z = _f(r), _f(z)
    s, g = np.zeros_like(r), np.zeros_like(r)
    lib.hh_theta_over_r(r.size, _p(r), _p(z), _p(s), _p(g))
    return s, g
