"""fp32 / fp64 reference of the orthographic and equidistant fisheye camera models for the tests: a torch restatement of
project_fwd<kOrtho> / project_fwd<kFisheye> of csrc/egs_math.cuh in the kernel's CANONICAL OP ORDER (so that its fp32
forward equals the kernels' bit for bit), differentiable by autograd in fp64, and the whole rasterization() built on
it the way tests/depth_reference.py builds the depth modes: the oracle's covariance, culling rules, SH colours, tile
lists and tests/features_oracle.py's blend in 32-channel chunks.  "pinhole" is the oracle's own projection.  The oracle
module itself is not changed."""
import math
from typing import Optional

import torch
from torch import Tensor

from oracle import gsplat_oracle as O
from tests import features_oracle as FO
from tests.sh_degree4_reference import sh_colors4

MODELS = ("pinhole", "ortho", "fisheye")

# fisheye_poly_p / fisheye_poly_h of egs_math.cuh, highest term first (scripts/fit_fisheye_theta.py)
P_COEFFS = (0.0010774789843708277, -0.007134431507438421, 0.022145025432109833, -0.044218774884939194,
            0.0670754536986351, -0.0879582092165947, 0.11054043471813202, -0.142791748046875, 0.1999961882829666,
            -0.33333325386047363, 1.0)
H_COEFFS = (-0.015319157391786575, 0.09921801835298538, -0.29700547456741333, 0.5588876008987427, -0.7710589170455933,
            0.876106321811676, -0.9004436731338501, 0.8879852890968323, -0.8571013808250427, 0.7999998927116394,
            -0.6666666865348816)
PI_HI, PI_LO = 3.1415927410125732, -8.742277657347586e-08
PIO2_HI, PIO2_LO = 1.5707963705062866, -4.371138828673793e-08
PIO4_HI, PIO4_LO = 0.7853981852531433, -2.1855694143368964e-08


def _horner(coeffs, u: Tensor) -> Tensor:
    p = torch.full_like(u, coeffs[0])
    for c in coeffs[1:]:
        p = p * u + c
    return p


def theta_over_r(r2: Tensor, z: Tensor, q: Tensor):
    """(s = atan2(r, z) / r, g = (1/r) ds/dr) of fisheye_theta_over_r, r = sqrt(r2).  The range is chosen on detached
    values, and each range sees only its own elements' inputs (the others get harmless stand-ins), so that fp64
    autograd has no 0 * inf from ranges not taken, e.g. at r = 0."""
    with torch.no_grad():
        r_nd = O._sqrt_rn(r2)
        near = r_nd <= z
        low = ~near & (z >= 0.5 * r_nd)
        mid = ~near & ~low & (r_nd > -z)
        far = ~near & ~low & ~mid
    one = torch.ones((), dtype=z.dtype)
    zn = torch.where(near, z, one)
    u1 = torch.where(near, r2, torch.zeros((), dtype=z.dtype)) / (zn * zn)
    s1 = _horner(P_COEFFS, u1) / zn
    g1 = _horner(H_COEFFS, u1) / ((zn * zn) * zn)
    r2o = torch.where(near, one, r2)
    r = O._sqrt_rn(r2o)
    zl = torch.where(low, z, torch.zeros((), dtype=z.dtype))
    zf = torch.where(far, -z, one)
    t = torch.where(low, (r - zl) / (r + zl), torch.where(mid, z / r, r / zf))
    at = t * _horner(P_COEFFS, t * t)
    full = lambda v: torch.full_like(z, v)
    hi = torch.where(low, full(PIO4_HI), torch.where(mid, full(PIO2_HI), full(PI_HI)))
    d = torch.where(low, PIO4_LO + at, torch.where(mid, full(PIO2_LO), full(PI_LO)) - at)
    th = d + hi
    tl = d - (th - hi)
    s0 = th / r
    p, e = _two_prod(s0, r)
    s2 = s0 + (((th - p) - e) + tl) / r
    g2 = (z * q - s2) / r2o
    return torch.where(near, s1, s2), torch.where(near, g1, g2)


def _two_prod(a: Tensor, b: Tensor):
    """two_prod of egs_math.cuh: a * b = p + e exactly in fp32 (Veltkamp split).  In fp64 the split terms are not
    exact, but p + e is still a * b to fp64 precision, and e then carries no gradient (e is a constant correction)."""
    if a.dtype != torch.float32:
        return a * b, torch.zeros_like(a)
    ca, cb = 4097.0 * a, 4097.0 * b
    ah, bh = ca - (ca - a), cb - (cb - b)
    al, bl = a - ah, b - bh
    p = a * b
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _project_elementwise(model, px, py, pz, cov6, V, fx, fy, cx, cy, eps2d):
    """The oracle's _project_elementwise with the camera model's means2d and Jacobian."""
    c00, c01, c02, c11, c12, c22 = cov6
    x = ((V["r00"] * px + V["r01"] * py) + V["r02"] * pz) + V["t0"]
    y = ((V["r10"] * px + V["r11"] * py) + V["r12"] * pz) + V["t1"]
    z = ((V["r20"] * px + V["r21"] * py) + V["r22"] * pz) + V["t2"]
    S = [[c00, c01, c02], [c01, c11, c12], [c02, c12, c22]]
    Wm = [[V["r00"], V["r01"], V["r02"]], [V["r10"], V["r11"], V["r12"]], [V["r20"], V["r21"], V["r22"]]]
    A = [[(Wm[i][0] * S[0][j] + Wm[i][1] * S[1][j]) + Wm[i][2] * S[2][j] for j in range(3)] for i in range(3)]

    def sc(i, j):
        return (A[i][0] * Wm[j][0] + A[i][1] * Wm[j][1]) + A[i][2] * Wm[j][2]

    k00, k01, k02, k11, k12, k22 = sc(0, 0), sc(0, 1), sc(0, 2), sc(1, 1), sc(1, 2), sc(2, 2)
    if model == "ortho":
        a = (fx * k00) * fx
        b = (fx * k01) * fy
        d = (fy * k11) * fy
        m2x = fx * x + cx
        m2y = fy * y + cy
    else:
        xx, yy = x * x, y * y
        r2 = xx + yy
        q = 1.0 / (r2 + z * z)
        s, g = theta_over_r(r2, z, q)
        xyg = (x * y) * g
        J = [[fx * (s + xx * g), fx * xyg, -(fx * (x * q))], [fy * xyg, fy * (s + yy * g), -(fy * (y * q))]]
        k = [[k00, k01, k02], [k01, k11, k12], [k02, k12, k22]]
        B = [[(J[i][0] * k[0][j] + J[i][1] * k[1][j]) + J[i][2] * k[2][j] for j in range(3)] for i in range(2)]

        def cv(i, j):
            return (B[i][0] * J[j][0] + B[i][1] * J[j][1]) + B[i][2] * J[j][2]

        a, b, d = cv(0, 0), cv(0, 1), cv(1, 1)
        m2x = (fx * x) * s + cx
        m2y = (fy * y) * s + cy
    det_orig = a * d - b * b
    a = a + eps2d
    d = d + eps2d
    det = a * d - b * b
    return x, y, z, a, b, d, det, m2x, m2y, det_orig


def fully_fused_projection(means, quats, scales, viewmats, Ks, width, height, eps2d=0.3, near_plane=0.01,
                           far_plane=1e10, radius_clip=0.0, calc_compensations=False, camera_model="pinhole"):
    """oracle.fully_fused_projection for a camera model: radii, means2d, depths, conics (+ compensations), culled
    entries exactly 0, the cull decided on a no-grad pass, the differentiable values recomputed on the visible pairs."""
    assert camera_model in MODELS, camera_model
    if camera_model == "pinhole":
        return O.fully_fused_projection(means, quats, scales, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
                                        radius_clip, calc_compensations=calc_compensations)
    C, N = viewmats.shape[0], means.shape[0]
    dt = means.dtype
    V, fx, fy, cx, cy = O._view_entries(viewmats, Ks)

    def body(mn, qt, sc, Vd, fx_, fy_, cx_, cy_):
        px, py, pz = mn.unbind(-1)
        return _project_elementwise(camera_model, px, py, pz, O.quat_scale_to_covar(qt, sc), Vd, fx_, fy_, cx_, cy_,
                                    eps2d)

    with torch.no_grad():
        x, y, z, a, b, d, det, m2x, m2y, det_orig = body(
            means.detach().expand(C, N, 3), quats.detach().expand(C, N, 4), scales.detach().expand(C, N, 3),
            {k: v.detach().expand(C, N) for k, v in V.items()}, fx.detach().expand(C, N), fy.detach().expand(C, N),
            cx.detach().expand(C, N), cy.detach().expand(C, N))
        valid = (z >= near_plane) & (z <= far_plane)
        valid &= det > 0
        mid = 0.5 * (a + d)
        v1 = mid + O._sqrt_rn(torch.clamp_min(mid * mid - det, 0.01))
        radius = torch.ceil(3.0 * O._sqrt_rn(v1))
        valid &= radius > radius_clip
        valid &= ~((m2x + radius <= 0) | (m2x - radius >= width) | (m2y + radius <= 0) | (m2y - radius >= height))
        valid &= torch.isfinite(radius) & torch.isfinite(m2x) & torch.isfinite(m2y)
        radius = torch.where(valid, radius, torch.zeros_like(radius))
        radii = radius.clamp(max=2147483520.0).to(torch.int32).contiguous()
    ci, ni = valid.nonzero(as_tuple=True)
    Vs = {k: v[ci, 0] for k, v in V.items()}
    x, y, z, a, b, d, det, m2x, m2y, det_orig = body(means[ni], quats[ni], scales[ni], Vs, fx[ci, 0], fy[ci, 0],
                                                     cx[ci, 0], cy[ci, 0])
    inv_det = 1.0 / det
    ca, cb, cc = d * inv_det, -(b * inv_det), a * inv_det
    means2d = torch.zeros(C, N, 2, dtype=dt).index_put((ci, ni), torch.stack([m2x, m2y], -1))
    depths = torch.zeros(C, N, dtype=dt).index_put((ci, ni), z)
    conics = torch.zeros(C, N, 3, dtype=dt).index_put((ci, ni), torch.stack([ca, cb, cc], -1))
    if calc_compensations:
        comp = torch.zeros(C, N, dtype=dt).index_put((ci, ni), O._CompensationSqrt.apply(det_orig / det))
        return radii, means2d, depths, conics, comp
    return radii, means2d, depths, conics


def rasterization_camera_model(means: Tensor, quats: Tensor, scales: Tensor, opacities: Tensor, colors: Tensor,
                               viewmats: Tensor, Ks: Tensor, width: int, height: int, camera_model: str = "pinhole",
                               render_mode: str = "RGB", sh_degree: Optional[int] = None,
                               backgrounds: Optional[Tensor] = None, absgrad: bool = False,
                               rasterize_mode: str = "classic", near_plane: float = 0.01, far_plane: float = 1e10,
                               radius_clip: float = 0.0, eps2d: float = 0.3, tile_size: int = 16,
                               counters: Optional[dict] = None, **_unused):
    """-> (render_colors, render_alphas, meta) of rasterization_camera_model(): "RGB" [C,H,W,D], "RGB+ED" [C,H,W,D+1],
    "ED" [C,H,W,1]; meta holds radii, means2d, depths, conics, isect_ids, flatten_ids, isect_offsets."""
    assert render_mode in ("RGB", "ED", "RGB+ED"), render_mode
    N, C = means.shape[0], viewmats.shape[0]
    proj = fully_fused_projection(means, quats, scales, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
                                  radius_clip, calc_compensations=rasterize_mode == "antialiased",
                                  camera_model=camera_model)
    radii, means2d, depths, conics = proj[:4]
    opac = opacities[None, :].expand(C, N)
    if rasterize_mode == "antialiased":
        opac = opac * proj[4]
    if sh_degree is None:
        cols = colors[None].expand(C, N, colors.shape[-1]) if colors.dim() == 2 else colors
    elif sh_degree == 4:
        cols = sh_colors4(means, viewmats, colors, radii)
    else:
        campos = torch.inverse(viewmats)[:, :3, 3]
        shs = colors[None].expand(C, *colors.shape) if colors.dim() == 3 else colors
        cols = torch.clamp_min(O.spherical_harmonics(sh_degree, means[None] - campos[:, None], shs, masks=radii > 0) + 0.5,
                               0.0)
    if render_mode == "RGB+ED":
        cols = torch.cat([cols, depths[..., None]], -1)
        if backgrounds is not None:
            backgrounds = torch.cat([backgrounds, torch.zeros(C, 1, dtype=backgrounds.dtype)], -1)
    elif render_mode == "ED":
        cols = depths[..., None]
        backgrounds = None
    tw, th = math.ceil(width / tile_size), math.ceil(height / tile_size)
    _, isect_ids, flatten_ids = O.isect_tiles(means2d.detach(), radii, depths.detach(), tile_size, tw, th)
    isect_offsets = O.isect_offset_encode(isect_ids, C, tw, th)
    D = cols.shape[-1]
    chunks, views = [], []
    for c0 in range(0, D, FO.CHANNEL_CHUNK):
        m2 = means2d.view_as(means2d) if absgrad and D > FO.CHANNEL_CHUNK else means2d
        views.append(m2)
        bg = None if backgrounds is None else backgrounds[:, c0:c0 + FO.CHANNEL_CHUNK]
        chunks.append(FO.rasterize_to_pixels(m2, conics, cols[..., c0:c0 + FO.CHANNEL_CHUNK], opac, width, height,
                                             tile_size, isect_offsets, flatten_ids, backgrounds=bg, absgrad=absgrad,
                                             counters=counters if c0 == 0 else None))
    render_colors = torch.cat([ch[0] for ch in chunks], -1)
    render_alphas = chunks[0][1]
    if absgrad and D > FO.CHANNEL_CHUNK and means2d.requires_grad:
        def _sum_absgrad(grad):
            means2d.absgrad = sum(v.absgrad for v in views)
        means2d.register_hook(_sum_absgrad)
    if render_mode != "RGB":
        render_colors = torch.cat([render_colors[..., :-1],
                                   render_colors[..., -1:] / render_alphas.clamp(min=1e-10)], -1)
    meta = {"radii": radii, "means2d": means2d, "depths": depths, "conics": conics, "isect_ids": isect_ids,
            "flatten_ids": flatten_ids, "isect_offsets": isect_offsets}
    return render_colors, render_alphas, meta
