"""fp32 / fp64 reference of the expected-depth render modes ("ED", "RGB+ED") for the tests, built the way gsplat 1.0.0's
rasterization() builds them: the oracle's projection, then the colours (SH of degree 0-3 through the oracle, degree 4
through tests/sh_degree4_reference.py, or the colours as given), then cat(colours, depths[..., None]) with a zero
background column ("RGB+ED") or the depths alone ("ED", background not used), the blend of tests/features_oracle.py in
32-channel chunks (as rasterization() blends wider colours: absgrad is the sum over the chunks), and the division of
the depth channel by render_alphas.clamp(min=1e-10).  The oracle module itself is not changed."""
import math
from typing import Optional

import torch
from torch import Tensor

from oracle import gsplat_oracle as O
from tests import features_oracle as FO
from tests.sh_degree4_reference import sh_colors4


def rasterization_depth(means: Tensor, quats: Tensor, scales: Tensor, opacities: Tensor, colors: Tensor,
                        viewmats: Tensor, Ks: Tensor, width: int, height: int, render_mode: str = "RGB+ED",
                        sh_degree: Optional[int] = None, backgrounds: Optional[Tensor] = None, absgrad: bool = False,
                        rasterize_mode: str = "classic", near_plane: float = 0.01, far_plane: float = 1e10,
                        radius_clip: float = 0.0, eps2d: float = 0.3, tile_size: int = 16,
                        counters: Optional[dict] = None, **_unused):
    """-> (render_colors [C,H,W,D+1] or [C,H,W,1], render_alphas [C,H,W,1], meta) for render_mode "RGB+ED" / "ED"."""
    assert render_mode in ("ED", "RGB+ED"), render_mode
    N, C = means.shape[0], viewmats.shape[0]
    proj = O.fully_fused_projection(means, quats, scales, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
                                    radius_clip, calc_compensations=rasterize_mode == "antialiased")
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
    else:
        cols = depths[..., None]
        backgrounds = None
    tw, th = math.ceil(width / tile_size), math.ceil(height / tile_size)
    _, isect_ids, flatten_ids = O.isect_tiles(means2d.detach(), radii, depths.detach(), tile_size, tw, th)
    isect_offsets = O.isect_offset_encode(isect_ids, C, tw, th)
    D = cols.shape[-1]
    chunks, views = [], []
    for c0 in range(0, D, FO.CHANNEL_CHUNK):
        # as tests/features_oracle.py: every chunk tags .absgrad on its own view of means2d, a hook sums them
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
    render_colors = torch.cat([render_colors[..., :-1],
                               render_colors[..., -1:] / render_alphas.clamp(min=1e-10)], -1)
    meta = {"radii": radii, "means2d": means2d, "depths": depths, "conics": conics}
    return render_colors, render_alphas, meta
