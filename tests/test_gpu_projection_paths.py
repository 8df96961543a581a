"""-m gpu: every kernel path of the projection stage (csrc/projection.cu), output by output, against the fp32 oracle,
fp64 references and the host-compiled per-thread math (tests/host_harness).

projection_fwd_impl / projection_bwd_impl pick the kernel from the arguments:
  sh16    raw, or K == 16 with 16-byte aligned SH (and v_sh)  projection_fwd_sh16_kernel   projection_bwd_sh16_kernel<AA, VG>
  vec4    sh_degree >= 0, K*3 % 4 == 0, aligned, K != 16        projection_fwd_kernel<true>   projection_bwd_kernel<true, VG>
  scalar  everything else: direct colours, K = 1, 9, 25 or a     projection_fwd_kernel<false>  projection_bwd_kernel<false, VG>
          misaligned K = 16
Each path runs on seeded cases built from populations placed on purpose (near plane, behind the camera, fov clamp,
off screen, tiny / huge / needle-thin scales, unnormalised quaternions, opacities at both ends, clamped SH colours,
Gaussians seen by some cameras only) with a warp layout that exercises the partial-warp and empty-warp code of the
row tiles and ballots.  All calls go through the C ABI with every output buffer poisoned (NaN / 0x7fffffff), so each
check also proves that the header's "written for every entry" promise holds.  The population census of the cases
runs on the CPU in tests/test_projection_paths_reference.py."""
import ctypes
import math
from dataclasses import dataclass
from functools import lru_cache

import numpy as np
import pytest
import torch

from oracle import gsplat_oracle as O
from tests import host_harness as hh

pytestmark = pytest.mark.gpu

# ---- cases ----------------------------------------------------------------------------------------------------------

W, H = 157, 91                 # ragged: 10 x 6 tiles, the last column and row partial
FX, FY = 120.0, 118.0
CX, CY = 0.5 * W + 0.37, 0.5 * H - 0.21
TAN_X, TAN_Y = 0.5 * W / FX, 0.5 * H / FY   # tan(fov / 2); the Jacobian clamps at 1.3 x these
NEAR, FAR, EPS2D, CLIP, TILE = 0.01, 1e10, 0.3, 0.0, 16
TW, TH = -(-W // TILE), -(-H // TILE)
K_MAX = 25

# populations a case is assembled from (the census in the CPU file checks each is present with the property it names)
POPULATIONS = ("general", "near_plane", "behind", "fov_clamped", "fov_inside", "off_screen", "tiny", "huge",
               "needle", "opacity_low", "opacity_high", "sh_clamped", "edge")

CASES = [  # (N, C, seed): N around warp and block boundaries; C = 65 is the first camera past the 64-camera cache
    (1, 1, 11), (31, 3, 12), (32, 65, 13), (33, 64, 14), (127, 3, 15), (128, 1, 16), (129, 65, 17), (4097, 3, 18),
]


@dataclass
class Case:
    N: int
    C: int
    seed: int
    means: torch.Tensor      # [N,3]
    quats: torch.Tensor      # [N,4] wxyz, unnormalised
    scales: torch.Tensor     # [N,3]
    opacities: torch.Tensor  # [N]
    sh: torch.Tensor         # [N,25,3]
    rgb: torch.Tensor        # [N,3]
    rgb_cam: torch.Tensor    # [C,N,3]
    viewmats: torch.Tensor   # [C,4,4]
    Ks: torch.Tensor         # [C,3,3]
    labels: list             # population of each Gaussian
    layout: dict             # warp layout: {"empty_warp": w, "one_lane_warp": w, "last_warp": w} (N >= 97)


def _rot(yaw, pitch):
    cy_, sy_, cp, sp = math.cos(yaw), math.sin(yaw), math.cos(pitch), math.sin(pitch)
    Ry = np.array([[cy_, 0, sy_], [0, 1, 0], [-sy_, 0, cy_]])
    Rx = np.array([[1, 0, 0], [0, cp, -sp], [0, sp, cp]])
    return Ry @ Rx


def _cameras(C):
    """Camera 0 is the world frame; the others are turned by up to ~5.7 degrees and shifted sideways by up to 1 cm, so
    Gaussians placed at camera 0's image border are seen by some cameras only."""
    vm = np.zeros((C, 4, 4))
    for c in range(C):
        R = np.eye(3) if c == 0 else _rot(0.1 * math.sin(1.7 * c + 0.3), 0.06 * math.cos(2.3 * c))
        t = np.zeros(3) if c == 0 else np.array([0.01 * math.sin(c), 0.01 * math.cos(1.3 * c), 0.0])
        vm[c, :3, :3], vm[c, :3, 3], vm[c, 3, 3] = R, t, 1.0
    K = np.array([[FX, 0, CX], [0, FY, CY], [0, 0, 1.0]])
    return torch.tensor(vm, dtype=torch.float32), torch.tensor(np.broadcast_to(K, (C, 3, 3)).copy(), dtype=torch.float32)


def _labels(N, rng):
    """Population of every slot.  N >= 97: warp 1 sees nothing, warp 2 has exactly one visible lane and the last warp
    only its final lane; the remaining slots cycle through the populations in a seeded order."""
    labels = [None] * N
    layout = {}
    if N >= 97:
        last = (N - 1) // 32
        layout = {"empty_warp": 1, "one_lane_warp": 2, "last_warp": last}
        for n in range(32, 96):
            labels[n] = "behind"
        labels[64 + 17] = "general"
        for n in range(last * 32, N - 1):
            labels[n] = "behind"
        labels[N - 1] = "general"
    elif N > 32:
        labels[N - 1] = "general"  # the last, partial warp: its only lane is visible
    free = [n for n in range(N) if labels[n] is None]
    order = list(POPULATIONS)
    for i, n in enumerate(free):
        if i % len(order) == 0:
            rng.shuffle(order)
        labels[n] = order[i % len(order)]
    if N == 1:
        labels[0] = "general"
    return labels, layout


def _random_quat(rng, n=1):
    q = rng.normal(size=(n, 4))
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def make_case(N, C, seed):
    rng = np.random.default_rng(seed)
    labels, layout = _labels(N, rng)
    means, quats, scales = np.zeros((N, 3)), np.zeros((N, 4)), np.zeros((N, 3))
    opac = rng.uniform(0.05, 0.95, N)
    sh = rng.normal(size=(N, K_MAX, 3)) * 0.15
    sh[:, 0, :] = rng.uniform(-0.4, 1.2, (N, 3))
    u = lambda a, b: rng.uniform(a, b)
    seen = {}
    for n, lab in enumerate(labels):
        k = seen[lab] = seen.get(lab, -1) + 1  # occurrence of this population: alternates the sides of an edge
        z = u(1.5, 6.0)
        xr, yr = u(-0.8, 0.8) * TAN_X, u(-0.8, 0.8) * TAN_Y
        s = z * np.exp(rng.uniform(math.log(0.002), math.log(0.03), 3))
        q = _random_quat(rng)[0]
        if lab == "general" and n == N - 1:
            xr, yr = u(-0.4, 0.4) * TAN_X, u(-0.4, 0.4) * TAN_Y
        elif lab == "near_plane":   # centres within 30 % of the near plane: culled on one side, projected on the other
            z = NEAR * (u(0.7, 0.95) if k % 2 == 0 else u(1.05, 1.3))
            xr, yr, s = u(-0.3, 0.3) * TAN_X, u(-0.3, 0.3) * TAN_Y, z * np.full(3, 0.02)
        elif lab == "behind":
            z = -u(1.0, 4.0)
        elif lab in ("fov_clamped", "fov_inside"):  # past / just inside 1.3 tan(fov/2), large enough to reach the image
            side = rng.choice([-1.0, 1.0])
            f = u(1.45, 2.2) if lab == "fov_clamped" else u(1.2, 1.28)
            if k % 2 == 0:
                xr = side * f * TAN_X
            else:
                yr = side * f * TAN_Y
            s = z * rng.uniform(0.8, 1.2, 3)
        elif lab == "off_screen":
            xr = rng.choice([-1.0, 1.0]) * u(3.0, 6.0) * TAN_X
            s = z * np.full(3, 0.004)
        elif lab == "tiny":         # a thousandth of a pixel: eps2d is the whole 2D covariance
            s = z * rng.uniform(1e-6, 1e-5, 3)
        elif lab == "huge":
            s = z * rng.uniform(3.0, 8.0, 3)
        elif lab == "needle":       # ~45 degrees in the image plane, 250-500 px long, far thinner than a pixel
            a = rng.choice([-1.0, 1.0]) * math.pi / 4 + u(-0.1, 0.1)
            q = np.array([math.cos(a / 2), 0.0, 0.0, math.sin(a / 2)])
            s = z * np.array([u(2.0, 4.0), 1e-5, 1e-5])
        elif lab == "opacity_low":
            opac[n] = (1.0 / 255.0) * (1.0 + u(1e-3, 1e-2))
        elif lab == "opacity_high":
            opac[n] = u(0.999, 0.99995)
        elif lab == "sh_clamped":   # one channel's DC term pulls sum + 0.5 below zero
            sh[n, 0, rng.integers(0, 3)] = -u(3.0, 6.0)
        elif lab == "edge":         # on camera 0's left or right border, a couple of pixels wide
            xr = rng.choice([-1.0, 1.0]) * (TAN_X + u(-2.0, 2.0) / FX)
            s = z * np.full(3, 0.004)
        means[n] = (xr * abs(z), yr * abs(z), z)
        # unnormalised, norm in [0.2, 5] (log-uniform), either sign (the same rotation)
        quats[n] = q * math.exp(u(math.log(0.2), math.log(5.0))) * rng.choice([-1.0, 1.0])
        scales[n] = s
    viewmats, Ks = _cameras(C)
    f32 = lambda a: torch.tensor(a, dtype=torch.float32)
    return Case(N=N, C=C, seed=seed, means=f32(means), quats=f32(quats), scales=f32(scales), opacities=f32(opac),
                sh=f32(sh), rgb=f32(rng.uniform(0, 1, (N, 3))), rgb_cam=f32(rng.uniform(0, 1, (C, N, 3))),
                viewmats=viewmats, Ks=Ks, labels=labels, layout=layout)


@lru_cache(maxsize=None)
def get_case(N, C, seed):
    return make_case(N, C, seed)


def case_id(c):
    return f"N{c[0]}-C{c[1]}"


# ---- paths ----------------------------------------------------------------------------------------------------------

@dataclass(frozen=True)
class Path:
    name: str
    kind: str        # "sh", "rgb" ([N,3]), "rgb_cam" ([C,N,3]) or "raw"
    K: int
    deg: int
    aligned: bool
    family: str      # "sh16", "vec4" or "scalar": which kernels the dispatch must pick


PATHS = (
    [Path(f"sh16_d{d}", "sh", 16, d, True, "sh16") for d in range(4)]
    + [Path("vec4_K4_d1", "sh", 4, 1, True, "vec4"), Path("vec4_K20_d3", "sh", 20, 3, True, "vec4")]
    + [Path("scalar_K1_d0", "sh", 1, 0, True, "scalar"), Path("scalar_K9_d2", "sh", 9, 2, True, "scalar"),
       Path("scalar_K25_d3", "sh", 25, 3, True, "scalar")]
    + [Path(f"scalar_K16_d{d}_misaligned", "sh", 16, d, False, "scalar") for d in (0, 2, 3)]
    + [Path("rgb", "rgb", 1, -1, True, "scalar"), Path("rgb_per_camera", "rgb_cam", 1, -1, True, "scalar")]
    + [Path(f"raw_d{d}", "raw", 16, d, True, "sh16") for d in (0, 3)]
)


def expected_kernels(path, aa):
    a = "true" if aa else "false"
    if path.family == "sh16":
        return "projection_fwd_sh16_kernel", f"projection_bwd_sh16_kernel<{a}, false>"
    v = "true" if path.family == "vec4" else "false"
    return f"projection_fwd_kernel<{v}>", f"projection_bwd_kernel<{v}, false>"


def aa_modes(path):
    return (False,) if path.kind == "raw" else (False, True)


# ---- device calls through the C ABI, every output poisoned -------------------------------------------------------

POISON_I32 = 0x7FFFFFFF


def _lib():
    from easy_gaussian_splatting_b200 import _lib as L
    return L.load()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _fpoison(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


def _ipoison(*shape):
    return torch.full(shape, POISON_I32, dtype=torch.int32, device="cuda")


def _misaligned(t):
    """A copy of t that starts 4 bytes past a 16-byte boundary, inside a NaN-filled buffer (returns view, buffer)."""
    buf = _fpoison(t.numel() + 8)
    view = buf[1:1 + t.numel()].view(t.shape)
    view.copy_(t)
    assert view.data_ptr() % 16 == 4
    return view, buf


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: {_lib().egs_last_error_string()}")


def device_inputs(case, path):
    """The parameters the path's entry takes, on the device, and the activated fp32 values the kernels work with
    (for the raw entry: torch.exp / torch.sigmoid on CUDA, which the folded activations reproduce)."""
    d = dict(means=case.means.cuda(), quats=case.quats.cuda(), viewmats=case.viewmats.cuda(), Ks=case.Ks.cuda())
    if path.kind == "raw":
        d["log_scales"] = case.scales.log().cuda()
        d["logits"] = torch.logit(case.opacities).cuda()
        d["scales"] = torch.exp(d["log_scales"])
        d["opacities"] = torch.sigmoid(d["logits"])
        d["sh"] = case.sh[:, :16].contiguous().cuda()
        d["sh_0"], d["sh_rest"] = d["sh"][:, :1].clone(), d["sh"][:, 1:].clone()  # own, 16-byte aligned buffers
    else:
        d["scales"], d["opacities"] = case.scales.cuda(), case.opacities.cuda()
        if path.kind == "sh":
            d["sh"] = case.sh[:, :path.K].contiguous().cuda()
        elif path.kind == "rgb":
            d["sh"] = case.rgb.cuda()
        else:
            d["sh"] = case.rgb_cam.cuda()
    return d


def run_fwd(case, path, aa, d=None, raw_entry=None):
    """-> dict of CPU tensors.  raw_entry: False runs a raw path's activated twin (K = 16, aligned)."""
    d = d or device_inputs(case, path)
    C, N = case.C, case.N
    raw = path.kind == "raw" if raw_entry is None else raw_entry
    out = dict(radii=_ipoison(C, N), means2d=_fpoison(C, N, 2), depths=_fpoison(C, N), conics=_fpoison(C, N, 3),
               colors=_fpoison(C, N, 3), tiles_per_gauss=_ipoison(C, N), tight_rects=_ipoison(C, N, 2),
               splats=_fpoison(C, N, 12))
    deg, per_cam = (path.deg, 0) if path.kind in ("sh", "raw") else (-1, int(path.kind == "rgb_cam"))
    K = path.K if path.kind != "raw" else 16
    sh = d["sh"]
    if not path.aligned:
        sh, _keep = _misaligned(sh)
    tail = (_p(d["viewmats"]), _p(d["Ks"]), W, H, EPS2D, NEAR, FAR, CLIP, TILE, TW, TH, *[_p(out[k]) for k in
            ("radii", "means2d", "depths", "conics", "colors", "tiles_per_gauss", "tight_rects", "splats")])
    lib = _lib()
    if raw:
        rc = lib.egs_projection_fwd_raw(C, N, _p(d["means"]), _p(d["quats"]), _p(d["log_scales"]), _p(d["logits"]),
                                        _p(d["sh_0"]), _p(d["sh_rest"]), deg, *tail, _stream())
    elif aa:
        out["compensations"] = _fpoison(C, N)
        rc = lib.egs_projection_fwd_antialiased(C, N, _p(d["means"]), _p(d["quats"]), _p(d["scales"]),
                                                _p(d["opacities"]), _p(sh), K, deg, per_cam, *tail,
                                                _p(out["compensations"]), _stream())
    else:
        rc = lib.egs_projection_fwd(C, N, _p(d["means"]), _p(d["quats"]), _p(d["scales"]), _p(d["opacities"]), _p(sh),
                                    K, deg, per_cam, *tail, _stream())
    _check(rc, "projection_fwd")
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in out.items()}


def run_bwd(case, path, aa, d, fwd, rec, extra, absgrad, raw_entry=None):
    """-> dict of CPU tensors (v_sh is [N,K,3]; the raw entry's v_sh_0 / v_sh_rest are concatenated into it)."""
    C, N = case.C, case.N
    raw = path.kind == "raw" if raw_entry is None else raw_entry
    deg, per_cam = (path.deg, 0) if path.kind in ("sh", "raw") else (-1, int(path.kind == "rgb_cam"))
    K = path.K if path.kind != "raw" else 16
    out = dict(v_means=_fpoison(N, 3), v_quats=_fpoison(N, 4), v_scales=_fpoison(N, 3), v_opacities=_fpoison(N))
    if absgrad:
        out["absgrad"] = _fpoison(C, N, 2)
    sh = d["sh"]
    bufs = {}
    if raw:
        out["v_sh_0"], out["v_sh_rest"] = _fpoison(N, 1, 3), _fpoison(N, 15, 3)
    elif not path.aligned:
        sh, bufs["sh"] = _misaligned(sh)
        out["v_sh"], bufs["v_sh"] = _misaligned(_fpoison(*sh.shape))
    else:
        out["v_sh"] = _fpoison(*sh.shape)
    radii, colors = fwd["radii"].cuda(), fwd["colors"].cuda()
    rec_d = rec.cuda()
    ex = None if extra is None else extra.cuda()
    mid = (_p(d["viewmats"]), _p(d["Ks"]), W, H, EPS2D, _p(radii), _p(colors), _p(rec_d), _p(ex), _p(out["v_means"]),
           _p(out["v_quats"]), _p(out["v_scales"]), _p(out["v_opacities"]))
    lib = _lib()
    if raw:
        rc = lib.egs_projection_bwd_raw(C, N, _p(d["means"]), _p(d["quats"]), _p(d["log_scales"]), _p(d["logits"]),
                                        _p(d["sh_0"]), _p(d["sh_rest"]), deg, *mid, _p(out["v_sh_0"]),
                                        _p(out["v_sh_rest"]), _p(out.get("absgrad")), _stream())
    elif aa:
        rc = lib.egs_projection_bwd_antialiased(C, N, _p(d["means"]), _p(d["quats"]), _p(d["scales"]),
                                                _p(d["opacities"]), _p(sh), K, deg, per_cam, *mid, _p(out["v_sh"]),
                                                _p(out.get("absgrad")), _stream())
    else:
        rc = lib.egs_projection_bwd(C, N, _p(d["means"]), _p(d["quats"]), _p(d["scales"]), _p(sh), K, deg, per_cam,
                                    *mid, _p(out["v_sh"]), _p(out.get("absgrad")), _stream())
    _check(rc, "projection_bwd")
    torch.cuda.synchronize()
    res = {k: v.cpu() for k, v in out.items()}
    if raw:
        res["v_sh"] = torch.cat([res.pop("v_sh_0"), res.pop("v_sh_rest")], 1)
    for name, buf in bufs.items():  # the floats around a misaligned buffer stay untouched
        b = buf.cpu()
        assert torch.isnan(b[0]) and torch.isnan(b[1 + sh.numel():]).all(), f"{name}: write outside the buffer"
    return res


# ---- references ---------------------------------------------------------------------------------------------------

def records(case, radii):
    """Random gradient records {v_x,v_y,v_ca,v_cb | v_cc,v_opacity,v_r,v_g | v_b,|v_x|,|v_y|,0}, zero where culled
    (the layout of test_gpu_viewmat_grad._records)."""
    g = torch.Generator().manual_seed(1000 + case.seed)
    v = torch.randn(case.C, case.N, 12, generator=g)
    v[..., 9:11] = v[..., 0:2].abs()
    v[..., 11] = 0.0
    return v * (radii > 0)[..., None]


def extra_grad(case):
    return 0.1 * torch.randn(case.C, case.N, 2, generator=torch.Generator().manual_seed(2000 + case.seed))


@lru_cache(maxsize=None)
def oracle_fwd(key, raw):
    """fp32 oracle projection of a case (effective activated parameters for the raw entry)."""
    case = get_case(*key)
    scales = torch.exp(case.scales.log().cuda()).cpu() if raw else case.scales
    r, m2, dep, con, comp = O.fully_fused_projection(case.means, case.quats, scales, case.viewmats, case.Ks, W, H,
                                                     EPS2D, NEAR, FAR, CLIP, calc_compensations=True)
    tpg, _, _ = O.isect_tiles(m2, r, dep, TILE, TW, TH, sort=False)
    return dict(radii=r, means2d=m2, depths=dep, conics=con, compensations=comp, tiles_per_gauss=tpg)


def campos64(viewmats):
    return torch.inverse(viewmats.double())[:, :3, 3]


def sh_colors64(case, deg, sh, radii):
    """fp64 clamp_min(SH + 0.5, 0), zero where culled."""
    vis = radii > 0
    dirs = case.means.double()[None] - campos64(case.viewmats)[:, None]
    cols = O.spherical_harmonics(deg, dirs, sh.double()[None].expand(case.C, -1, -1, -1), vis)
    return torch.where(vis[..., None], torch.clamp_min(cols + 0.5, 0), torch.zeros((), dtype=torch.float64))


def ulp_diff(a, b):
    """|a - b| in units in the last place of fp32 (same-sign values; inf where signs differ)."""
    a, b = np.asarray(a, np.float32).ravel(), np.asarray(b, np.float32).ravel()
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    d = np.abs(ia - ib).astype(np.float64)
    d[(np.signbit(a) != np.signbit(b)) & ~((a == 0) & (b == 0))] = np.inf
    d[a == b] = 0
    return d


def assert_bit_identical(got, ref, what):
    got, ref = np.asarray(got), np.asarray(ref)
    if np.array_equal(got, ref):
        return
    if got.dtype == np.float32:
        u = ulp_diff(got, ref)
        raise AssertionError(f"{what}: not bit-identical, {int((u > 0).sum())} elements differ, max {u.max()} ulp")
    raise AssertionError(f"{what}: not bit-identical, {int((got != ref).sum())} elements differ")


def harness_scene(case, d, path):
    sh = d["sh"].cpu() if path.kind in ("sh", "raw") else torch.zeros(case.N, 1, 3)
    return type("S", (), dict(means=case.means, quats=case.quats, scales=d["scales"].cpu(), colors=sh,
                              viewmats=case.viewmats, Ks=case.Ks, width=W, height=H))


def harness_bwd(case, d, path, aa, fwd, rec, extra):
    """The same egs_math.cuh compiled for the host (-ffp-contract=off), fed the kernel's fp32 cotangents."""
    v_xy = rec[..., 0:2] + (extra if extra is not None else 0.0)  # fp32, as the kernel adds it
    v_comps = rec[..., 5] * d["opacities"].cpu()[None] if aa else None
    deg = path.deg if path.kind in ("sh", "raw") else -1
    return hh.projection_bwd(harness_scene(case, d, path), deg, fwd["radii"].numpy(), fwd["colors"], v_xy,
                             rec[..., 2:5], rec[..., 6:9], EPS2D, v_comps)


def v_opacities_ref(rec, fwd, aa):
    """fp32 sum over cameras, in camera order, of the records' opacity slot (times the compensation when
    antialiased) — what the kernels accumulate."""
    acc = np.zeros(rec.shape[1], np.float32)
    o = rec[..., 5].numpy()
    comp = fwd["compensations"].numpy() if aa else None
    for c in range(rec.shape[0]):
        acc = acc + (o[c] * comp[c] if aa else o[c]).astype(np.float32)
    return acc


_REF64 = {}


class _GuardedSqrt(torch.autograd.Function):
    """sqrt(max(x, 0)) whose VJP is gsplat 1.0.0's add_blur_vjp: v * 0.5 / (sqrt(x) + 1e-6), the guard the kernels
    reproduce (plain autograd of sqrt diverges at the Gaussians whose footprint is all eps2d)."""

    @staticmethod
    def forward(ctx, x):
        c = torch.sqrt(torch.clamp_min(x, 0))
        ctx.save_for_backward(c)
        return c

    @staticmethod
    def backward(ctx, g):
        (c,) = ctx.saved_tensors
        return g * 0.5 / (c + 1e-6)


def compensation64(con):
    """sqrt(det(cov2d) / det(cov2d + eps2d I)) from the blurred conic, differentiable in fp64."""
    ca, cb, cc = con.unbind(-1)
    det_b = 1.0 / (ca * cc - cb * cb)
    a, b, d = cc * det_b, -cb * det_b, ca * det_b
    return _GuardedSqrt.apply(((a - EPS2D) * (d - EPS2D) - b * b) / det_b)


def ref64_bwd(key, path, aa, d, fwd, rec, extra, use_cache=True):
    """fp64 autograd through the oracle of the functional whose cotangents the records hold, masked with the kernel's
    radii; the colour clamp is gated on the kernel's stored fp32 colour (a tie at 0 cannot flip)."""
    ck = (key, path.kind, path.deg, aa)
    if use_cache and ck in _REF64:
        return _REF64[ck]
    case = get_case(*key)
    m = case.means.double().requires_grad_(True)
    q = case.quats.double().requires_grad_(True)
    s = d["scales"].cpu().double().requires_grad_(True)
    op = d["opacities"].cpu().double().requires_grad_(True)
    vis = fwd["radii"] > 0
    r64 = rec.double()
    _, m2, _, con = O.fully_fused_projection(m, q, s, case.viewmats.double(), case.Ks.double(), W, H, EPS2D,
                                             -1e30, 1e30, -1.0)
    v_xy = r64[..., 0:2] + (extra.double() if extra is not None else 0.0)
    # only the entries the kernel projected take part (indexing, not masking: culled entries may hold inf / NaN)
    total = (m2[vis] * v_xy[vis]).sum() + (con[vis] * r64[..., 2:5][vis]).sum()
    opv = op[None].expand(case.C, -1)[vis]
    total = total + ((opv * compensation64(con[vis])) if aa else opv).mul(r64[..., 5][vis]).sum()
    leaves = dict(v_means=m, v_quats=q, v_scales=s, v_opacities=op)
    if path.kind in ("sh", "raw"):
        nb = (path.deg + 1) ** 2
        sh = d["sh"].cpu()[:, :nb].double().requires_grad_(True)
        dirs = m[None] - campos64(case.viewmats)[:, None]
        cols = O.spherical_harmonics(path.deg, dirs[vis], sh[None].expand(case.C, -1, -1, -1)[vis]) + 0.5
        gate = (fwd["colors"][vis] > 0).double()
        total = total + (cols * gate * r64[..., 6:9][vis]).sum()
        leaves["v_sh"] = sh
    total.backward()
    res = {k: v.grad.detach() for k, v in leaves.items()}
    if use_cache:
        _REF64[ck] = res
    return res


# ---- forward ------------------------------------------------------------------------------------------------------

def assert_forward_contract(out, aa, what):
    """Every element the header promises is written (no poison left), culled entries zero-filled."""
    culled = out["radii"] == 0
    for k in ("radii", "tiles_per_gauss", "tight_rects"):
        assert not (out[k] == POISON_I32).any(), f"{what}: {k} not fully written"
    for k in ("means2d", "depths", "conics", "colors") + (("compensations",) if aa else ()):
        assert not torch.isnan(out[k]).any(), f"{what}: {k} not fully written"
        assert (out[k][culled] == 0).all(), f"{what}: {k} of culled entries not zero"
    assert (out["tiles_per_gauss"][culled] == 0).all() and (out["tight_rects"][culled] == 0).all(), what
    assert (out["radii"] >= 0).all(), what


def unpack_rects(packed):
    x0, y0 = packed[..., 0] & 0xFFFF, (packed[..., 0] >> 16) & 0xFFFF
    return x0, y0, x0 + (packed[..., 1] & 0xFFFF), y0 + ((packed[..., 1] >> 16) & 0xFFFF)


_RECTS_CHECKED = set()
ALPHA_MIN = (1.0 / 255.0) * (1.0 + 1e-4)


def check_tight_rects(key, out, rec_opac, what, check_reach):
    """Bit-identical to the host-compiled rectangle of the kernel's own means2d / radii / conics / record opacities,
    inside the classic rectangle and conservative: no pixel centre of the classic rectangle with fp64 alpha >= 1/255
    lies outside it."""
    C, N = out["radii"].shape
    m2, rad, con = out["means2d"].reshape(-1, 2).numpy(), out["radii"].reshape(-1).numpy(), out["conics"].reshape(-1, 3).numpy()
    op = rec_opac.reshape(-1).numpy()
    classic, packed = hh.tight_rects(m2, rad, con, op, TW, TH, TILE)
    got = out["tight_rects"].reshape(-1, 2).numpy()
    assert_bit_identical(got, packed, f"{what}: tight_rects vs host harness")
    x0, y0, x1, y1 = unpack_rects(got)
    ne = (x1 > x0) & (y1 > y0)
    assert np.all(x0[ne] >= classic[ne, 0]) and np.all(x1[ne] <= classic[ne, 2]), f"{what}: tight rect outside classic"
    assert np.all(y0[ne] >= classic[ne, 1]) and np.all(y1[ne] <= classic[ne, 3]), f"{what}: tight rect outside classic"
    if not check_reach:
        return
    vis = np.nonzero(rad > 0)[0]
    px = np.arange(W) + 0.5
    py = np.arange(H) + 0.5
    tx, ty = (px // TILE).astype(np.int64), (py // TILE).astype(np.int64)
    bad = 0
    for s in range(0, vis.size, 256):
        i = vis[s:s + 256]
        dx = px[None, None, :] - m2[i, 0].astype(np.float64)[:, None, None]
        dy = py[None, :, None] - m2[i, 1].astype(np.float64)[:, None, None]
        a_, b_, c_ = (con[i, j].astype(np.float64)[:, None, None] for j in range(3))
        sigma = 0.5 * (a_ * dx * dx + c_ * dy * dy) + b_ * dx * dy
        alpha = np.minimum(0.999, op[i].astype(np.float64)[:, None, None] * np.exp(-sigma))
        in_classic = ((tx[None, None, :] >= classic[i, 0, None, None]) & (tx[None, None, :] < classic[i, 2, None, None])
                      & (ty[None, :, None] >= classic[i, 1, None, None]) & (ty[None, :, None] < classic[i, 3, None, None]))
        in_tight = ((tx[None, None, :] >= x0[i, None, None]) & (tx[None, None, :] < x1[i, None, None])
                    & (ty[None, :, None] >= y0[i, None, None]) & (ty[None, :, None] < y1[i, None, None]))
        bad += int(((alpha >= ALPHA_MIN) & in_classic & ~in_tight).sum())
    assert bad == 0, f"{what}: {bad} pixel centres with alpha >= 1/255 outside the tight rectangle"


def sigma_cutoff_ref(opac):
    """sigma_cutoff(opacity) = ln(255 o) * 1.001 + 2e-3 (-1 when 255 o <= 1), one fp32 operation per torch call on
    the device, so logf is CUDA's own and nothing is contracted."""
    t = 255.0 * opac.cuda()
    return torch.where(t > 1.0, torch.log(t) * 1.001 + 2e-3, torch.full_like(t, -1.0)).cpu()


@pytest.mark.parametrize("path", PATHS, ids=lambda p: p.name)
@pytest.mark.parametrize("ck", CASES, ids=case_id)
def test_forward(ck, path):
    case = get_case(*ck)
    d = device_inputs(case, path)
    for aa in aa_modes(path):
        what = f"{case_id(ck)} {path.name} {'antialiased' if aa else 'classic'}"
        out = run_fwd(case, path, aa, d)
        assert_forward_contract(out, aa, what)
        ref = oracle_fwd(ck, path.kind == "raw")
        for k in ("radii", "means2d", "depths", "conics", "tiles_per_gauss") + (("compensations",) if aa else ()):
            assert_bit_identical(out[k], ref[k], f"{what}: {k} vs oracle")
        vis = out["radii"] > 0
        if path.kind in ("sh", "raw"):
            col64 = sh_colors64(case, path.deg, d["sh"].cpu(), out["radii"])
            err = (out["colors"].double() - col64).abs().max().item()
            print(f"MEASURE colors_fp64 {path.name} {err:.3g} bound 2e-6")
            assert err <= 2e-6, f"{what}: colours vs fp64 SH {err:.3g} > 2e-6"
        else:
            src = case.rgb[None].expand(case.C, -1, -1) if path.kind == "rgb" else case.rgb_cam
            assert torch.equal(out["colors"], torch.where(vis[..., None], src, torch.zeros(()))), f"{what}: colours"
        # splat records of visible entries
        op = d["opacities"].cpu()[None].expand(case.C, -1)
        if aa:
            op = op * out["compensations"]
        sp = out["splats"][vis]
        want = torch.cat([out["means2d"][vis], out["conics"][vis], op[vis][:, None], out["colors"][vis],
                          out["depths"][vis][:, None], torch.zeros(int(vis.sum()), 1)], 1)
        want = torch.cat([want, sigma_cutoff_ref(op[vis])[:, None]], 1)
        assert_bit_identical(sp.numpy(), want.numpy(), f"{what}: splat records")
        rec_op = torch.where(vis, out["splats"][..., 5], torch.zeros(()))
        rk = (ck, aa, path.kind == "raw")
        check_tight_rects(ck, out, rec_op, what, rk not in _RECTS_CHECKED)
        _RECTS_CHECKED.add(rk)
        # same inputs, same bits
        again = run_fwd(case, path, aa, d)
        for k in out:
            if k != "splats":
                assert torch.equal(out[k], again[k]), f"{what}: {k} differs between two identical calls"
        if path.kind == "raw":  # the folded exp / sigmoid / cat against the activated entry fed torch's CUDA results
            act = run_fwd(case, path, False, d, raw_entry=False)
            for k in out:
                a, b = (out[k][vis], act[k][vis]) if k == "splats" else (out[k], act[k])
                assert_bit_identical(a.numpy(), b.numpy(), f"{what}: {k} raw vs activated entry")


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("ck", [CASES[3], CASES[7]], ids=case_id)
def test_sh16_and_generic_colours_bit_identical(ck, deg):
    """projection_fwd_sh16_kernel claims the accumulation order of sh_color_fwd (the generic kernels' colour)."""
    case = get_case(*ck)
    a = run_fwd(case, Path("a", "sh", 16, deg, True, "sh16"), False)
    b = run_fwd(case, Path("b", "sh", 16, deg, False, "scalar"), False)
    assert_bit_identical(a["colors"].numpy(), b["colors"].numpy(), f"{case_id(ck)} deg {deg}: sh16 vs generic colours")


# ---- backward -----------------------------------------------------------------------------------------------------

def assert_backward_contract(case, path, out, fwd, what):
    for k in ("v_means", "v_quats", "v_scales", "v_opacities", "v_sh") + (("absgrad",) if "absgrad" in out else ()):
        assert not torch.isnan(out[k]).any(), f"{what}: {k} not fully written"
    if path.kind in ("sh", "raw"):
        nb = (path.deg + 1) ** 2
        assert (out["v_sh"][:, nb:] == 0).all(), f"{what}: inactive SH bands / rows 48..3K not zero"
        never = ~(fwd["radii"] > 0).any(0)
        assert (out["v_sh"][never] == 0).all(), f"{what}: v_sh of Gaussians no camera sees not zero"
    never = ~(fwd["radii"] > 0).any(0)
    for k in ("v_means", "v_quats", "v_scales", "v_opacities"):
        assert (out[k][never] == 0).all(), f"{what}: {k} of Gaussians no camera sees not zero"


def check_against_fp64(name, got, h, ref, what):
    """Norm-wise: rel <= max(4 e32, 1e-6) with e32 the fp32 harness's own error on this case; element-wise:
    |got - ref| <= 4 |harness - ref| + 4 ulp(max |ref|)."""
    got, h, ref = got.double(), torch.as_tensor(np.asarray(h)).double(), ref.double()
    nref = ref.norm().clamp_min(1e-30)
    e32 = ((h - ref).norm() / nref).item()
    e = ((got - ref).norm() / nref).item()
    bound = max(4 * e32, 1e-6)
    print(f"MEASURE fp64_rel {name} {e:.3g} bound {bound:.3g}")
    assert e <= bound, f"{what}: {name} rel err vs fp64 {e:.3g} > bound {bound:.3g} (harness {e32:.3g})"
    floor = 4 * float(np.spacing(np.float32(ref.abs().max().item())))
    over = (got - ref).abs() - (4 * (h - ref).abs() + floor)
    worst = over.max().item() if over.numel() else -1.0
    assert worst <= 0, f"{what}: {name} element-wise error exceeds 4x harness + 4 ulp by {worst:.3g}"


@pytest.mark.parametrize("path", PATHS, ids=lambda p: p.name)
@pytest.mark.parametrize("ck", CASES, ids=case_id)
def test_backward(ck, path):
    case = get_case(*ck)
    d = device_inputs(case, path)
    for aa in aa_modes(path):
        fwd = run_fwd(case, path, aa, d)
        rec = records(case, fwd["radii"])
        vis = fwd["radii"] > 0
        for with_extra in (False, True):
            what = f"{case_id(ck)} {path.name} {'antialiased' if aa else 'classic'} {'extra+absgrad' if with_extra else 'plain'}"
            extra = extra_grad(case) if with_extra else None
            out = run_bwd(case, path, aa, d, fwd, rec, extra, absgrad=with_extra)
            assert_backward_contract(case, path, out, fwd, what)
            again = run_bwd(case, path, aa, d, fwd, rec, extra, absgrad=with_extra)
            for k in out:
                assert torch.equal(out[k], again[k]), f"{what}: {k} differs between two identical calls"
            if with_extra:
                want = torch.where(vis[..., None], rec[..., 9:11], torch.zeros(()))
                assert torch.equal(out["absgrad"], want), f"{what}: absgrad is not the records' |v_x|, |v_y|"
            if path.kind != "raw":
                assert_bit_identical(out["v_opacities"].numpy(), v_opacities_ref(rec, fwd, aa), f"{what}: v_opacities")
            if path.kind == "rgb":
                acc = np.zeros((case.N, 3), np.float32)
                for c in range(case.C):
                    acc = acc + rec[c, :, 6:9].numpy()
                assert_bit_identical(out["v_sh"].numpy(), acc, f"{what}: v_colors")
            elif path.kind == "rgb_cam":  # written for every (c, n): the record's colour slots, 0 where culled
                assert torch.equal(out["v_sh"], rec[..., 6:9]), f"{what}: per-camera v_colors"
            if path.kind == "raw":
                act = run_bwd(case, path, False, d, fwd, rec, extra, absgrad=with_extra, raw_entry=False)
                # the activations' VJPs on the device, in the kernel's operation order
                o = d["opacities"]
                v_ls = (act["v_scales"].cuda() * torch.exp(d["log_scales"])).cpu()
                v_lg = (act["v_opacities"].cuda() * (o * (1.0 - o))).cpu()
                for k, want in (("v_means", act["v_means"]), ("v_quats", act["v_quats"]), ("v_scales", v_ls),
                                ("v_opacities", v_lg), ("v_sh", act["v_sh"])):
                    assert_bit_identical(out[k].numpy(), want.numpy(), f"{what}: raw {k} vs activated + chain rule")
                continue
            h = harness_bwd(case, d, path, aa, fwd, rec, extra)
            names = ("v_means", "v_quats", "v_scales") + (("v_sh",) if path.kind == "sh" else ())
            for k in names:  # generic and sh16 kernels run the harness's functions in its order, camera by camera
                assert_bit_identical(out[k].numpy(), h[k], f"{what}: {k} vs host harness")
            if with_extra:
                r64 = ref64_bwd(ck, path, aa, d, fwd, rec, extra)
                hv = dict(h)
                hv["v_opacities"] = v_opacities_ref(rec, fwd, aa)
                # needles lose their conic's determinant (and, antialiased, their compensation) to fp32 cancellation:
                # there the fp32 harness is off fp64 by orders of magnitude and would make the bound meaningless.  They
                # stay covered by the bit-identity with the harness above.
                keep = torch.tensor([lab != "needle" for lab in case.labels])
                for k in names + ("v_opacities",):
                    ref = r64[k]
                    if k == "v_sh":
                        ref = torch.nn.functional.pad(ref, (0, 0, 0, path.K - ref.shape[1]))
                    check_against_fp64(f"{k}_{path.name}", out[k][keep], np.asarray(hv[k])[keep.numpy()], ref[keep], what)


# ---- dispatch guard -----------------------------------------------------------------------------------------------

def test_dispatch_picks_the_expected_kernel_per_path():
    """One profiled call per dispatch-table row: the kernel name and template arguments that ran.  If the dispatch
    moves, this fails instead of the coverage above silently moving to another kernel."""
    from torch.profiler import ProfilerActivity, profile
    case = get_case(*CASES[4])
    for path in PATHS:
        for aa in aa_modes(path):
            d = device_inputs(case, path)
            fwd = run_fwd(case, path, aa, d)
            rec = records(case, fwd["radii"])
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run_fwd(case, path, aa, d)
                run_bwd(case, path, aa, d, fwd, rec, None, absgrad=False)
            names = [e.key for e in prof.key_averages() if "projection_" in e.key]
            f, b = expected_kernels(path, aa)
            ran = [n for n in names if "_kernel" in n]
            assert any(f + "(" in n or n.endswith(f) or f + " " in n for n in ran), (path.name, aa, f, ran)
            assert any(b in n for n in ran), (path.name, aa, b, ran)
            assert len(ran) == 2, (path.name, aa, ran)
