"""fp64-capable reference of SH degree 4 for the tests: band 4 (indices 16..24) on top of the oracle's degrees 0..3, in
the oracle's CANONICAL OP ORDER style (the expressions of csrc/egs_math.cuh sh_basis4), and the whole-path reference
rasterization at degree 4 built from it.  The constants are those of gsplat's fast SH code (sh_coeffs_to_color_fast);
parity with gsplat's own degree-4 output is not pinned (gsplat is not a test dependency), the basis is pinned to the
complex spherical harmonics instead (tests/test_sh_degree4_oracle.py)."""
import torch

from oracle import gsplat_oracle as O

N_BANDS = 25


def sh_basis4(dirs):
    """dirs [...,3] (unnormalised) -> basis [..., 25]; entries 0..15 are oracle.sh_basis(3, dirs)."""
    b3 = O.sh_basis(3, dirs)
    inorm = 1.0 / torch.sqrt((dirs * dirs).sum(-1))
    x, y, z = (dirs * inorm[..., None]).unbind(-1)
    z2 = z * z
    fC1 = x * x - y * y
    fS1 = 2.0 * x * y
    fC2 = x * fC1 - y * fS1
    fS2 = x * fS1 + y * fC1
    fC3 = x * fC2 - y * fS2
    fS3 = x * fS2 + y * fC2
    fTmp0D = 3.31161143515146 * z2 - 0.47308734787878
    fTmp1C = z * (-4.683325804901025 * z2 + 2.007139630671868)
    fTmp2B = -1.770130769779931 * z
    b4 = [0.6258357354491763 * fS3, fTmp2B * fS2, fTmp0D * fS1, fTmp1C * y,
          1.984313483298443 * z * b3[..., 12] - 1.006230589874905 * b3[..., 6],
          fTmp1C * x, fTmp0D * fC1, fTmp2B * fC2, 0.6258357354491763 * fC3]
    return torch.cat([b3, torch.stack(b4, -1)], -1)


def sh_colors4(means, viewmats, shs, radii):
    """clamp_min(SH4(means - campos) + 0.5, 0) per (camera, Gaussian), [C,N,3]; shs [N,K,3] or [C,N,K,3], K >= 25.
    Culled pairs hold 0.5, as the oracle's."""
    C, N = viewmats.shape[0], means.shape[0]
    campos = torch.inverse(viewmats)[:, :3, 3]
    dirs = means[None, :, :] - campos[:, None, :]
    shs = shs[None].expand(C, *shs.shape) if shs.dim() == 3 else shs
    col = (sh_basis4(dirs)[..., None] * shs[..., :N_BANDS, :]).sum(-2)
    col = torch.where((radii > 0)[..., None], col, torch.zeros((), dtype=col.dtype))
    return torch.clamp_min(col + 0.5, 0.0)


def rasterization4(means, quats, scales, opacities, shs, viewmats, Ks, width, height, near_plane=0.01, far_plane=1e10,
                   radius_clip=0.0, eps2d=0.3, rasterize_mode="classic", **kw):
    """oracle.rasterization with sh_degree=4: the degree-4 colours are computed here and handed to the oracle as
    per-camera colours, so geometry, binning and blending are the oracle's own."""
    radii = O.fully_fused_projection(means.detach(), quats.detach(), scales.detach(), viewmats.detach(), Ks.detach(),
                                     width, height, eps2d, near_plane, far_plane, radius_clip)[0]
    cols = sh_colors4(means, viewmats, shs, radii)
    return O.rasterization(means, quats, scales, opacities, cols, viewmats, Ks, width, height, near_plane=near_plane,
                           far_plane=far_plane, radius_clip=radius_clip, eps2d=eps2d, sh_degree=None,
                           rasterize_mode=rasterize_mode, **kw)
