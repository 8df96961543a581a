"""CPU oracle for colours with any number of channels: gsplat 1.0.0's ``rasterize_to_pixels`` and ``rasterization``
with ``sh_degree=None`` and ``[N,D]`` / ``[C,N,D]`` colours, D >= 1.

Built from the pieces of ``oracle/gsplat_oracle.py`` — its per-tile blend ``_blend_tile`` (written over matrices, so
it blends any number of channels), its projection and its binning — with only the per-tile loop and its autograd node
restated here for D channels.  ``rasterization_features`` blends in chunks of ``CHANNEL_CHUNK`` channels, as gsplat's
default ``channel_chunk`` does: alphas come from the first chunk, geometry gradients add up over the chunks, and
``means2d.absgrad`` is the SUM of the chunks' absgrads (gsplat 1.0.0 assigns it inside each chunk's backward, so its
value for D > channel_chunk is whichever chunk's backward ran last)."""
import math
from typing import Optional

import torch
from torch import Tensor

from oracle import gsplat_oracle as O

CHANNEL_CHUNK = 32  # gsplat 1.0.0's default channel_chunk


class _RasterizeFeatures(torch.autograd.Function):
    """``oracle.gsplat_oracle._Rasterize`` for colours[C,N,D]: the same tile loop and per-tile blend."""

    @staticmethod
    def forward(ctx, means2d, conics, colors, opacities, backgrounds, width, height, tile_size, isect_offsets,
                flatten_ids, absgrad, counters):
        C, N, D = colors.shape
        dt = means2d.dtype
        th, tw = isect_offsets.shape[1:]
        out_c = torch.zeros(C, height, width, D, dtype=dt)
        out_a = torch.zeros(C, height, width, 1, dtype=dt)
        last_ids = torch.zeros(C, height, width, dtype=torch.int32)
        border = torch.zeros(C, height, width, dtype=torch.bool)
        offs = isect_offsets.reshape(-1).tolist() + [flatten_ids.shape[0]]
        m2, cn, cl, op = (means2d.reshape(C * N, 2), conics.reshape(C * N, 3), colors.reshape(C * N, D),
                          opacities.reshape(C * N))
        for c in range(C):
            bg = backgrounds[c] if backgrounds is not None else None
            for ty in range(th):
                for tx in range(tw):
                    t = (c * th + ty) * tw + tx
                    s, e = offs[t], offs[t + 1]
                    yy, xx, px, py = O._tile_pixels(ty, tx, tile_size, width, height, dt)
                    if e == s:  # nothing blended: T = 1, the background shows
                        if bg is not None:
                            out_c[c, yy, xx] = bg
                        continue
                    g = flatten_ids[s:e].long()
                    col, alp, last, _, _, _, bl = O._blend_tile(m2[g], cn[g], op[g], cl[g], px, py, bg)
                    border[c, yy, xx] = bl
                    out_c[c, yy, xx] = col
                    out_a[c, yy, xx, 0] = alp
                    last_ids[c, yy, xx] = torch.where(last >= 0, last + s, torch.zeros((), dtype=torch.int64)).to(torch.int32)
        if counters is not None:
            counters["borderline"] = border
        ctx.save_for_backward(means2d, conics, colors, opacities, backgrounds, isect_offsets, flatten_ids)
        ctx.meta = (width, height, tile_size, absgrad)
        ctx.mark_non_differentiable(last_ids)
        return out_c, out_a, last_ids

    @staticmethod
    def backward(ctx, v_c, v_a, _v_last):
        means2d, conics, colors, opacities, backgrounds, isect_offsets, flatten_ids = ctx.saved_tensors
        width, height, tile_size, absgrad = ctx.meta
        C, N, D = colors.shape
        dt = means2d.dtype
        th, tw = isect_offsets.shape[1:]
        offs = isect_offsets.reshape(-1).tolist() + [flatten_ids.shape[0]]
        m2, cn = means2d.detach().reshape(C * N, 2), conics.detach().reshape(C * N, 3)
        cl, op = colors.detach().reshape(C * N, D), opacities.detach().reshape(C * N)
        g_m2, g_abs, g_cn = torch.zeros_like(m2), torch.zeros_like(m2), torch.zeros_like(cn)
        g_cl, g_op = torch.zeros_like(cl), torch.zeros_like(op)
        g_bg = torch.zeros_like(backgrounds) if backgrounds is not None else None
        for c in range(C):
            for ty in range(th):
                for tx in range(tw):
                    t = (c * th + ty) * tw + tx
                    s, e = offs[t], offs[t + 1]
                    yy, xx, px, py = O._tile_pixels(ty, tx, tile_size, width, height, dt)
                    vc, va = v_c[c, yy, xx], v_a[c, yy, xx, 0]
                    if e == s:
                        if g_bg is not None:
                            g_bg[c] += vc.sum(0)  # T = 1 everywhere
                        continue
                    g = flatten_ids[s:e].long()
                    with torch.enable_grad():
                        lx, lc = m2[g].clone().requires_grad_(True), cn[g].clone().requires_grad_(True)
                        lr, lo = cl[g].clone().requires_grad_(True), op[g].clone().requires_grad_(True)
                        lb = backgrounds[c].detach().clone().requires_grad_(True) if backgrounds is not None else None
                        col, alp, _, (dx, dy), _, _, _ = O._blend_tile(lx, lc, lo, lr, px, py, lb, want_delta=True)
                        ((col * vc).sum() + (alp * va).sum()).backward()
                    g_m2.index_add_(0, g, lx.grad)
                    g_cn.index_add_(0, g, lc.grad)
                    g_cl.index_add_(0, g, lr.grad)
                    g_op.index_add_(0, g, lo.grad)
                    if g_bg is not None:
                        g_bg[c] += lb.grad
                    if absgrad:
                        g_abs.index_add_(0, g, torch.stack([dx.grad.abs().sum(0), dy.grad.abs().sum(0)], -1))
        if absgrad:
            means2d.absgrad = g_abs.reshape(C, N, 2)
        return (g_m2.reshape(C, N, 2), g_cn.reshape(C, N, 3), g_cl.reshape(C, N, D), g_op.reshape(C, N), g_bg,
                None, None, None, None, None, None, None)


def rasterize_to_pixels(means2d, conics, colors, opacities, width, height, tile_size, isect_offsets, flatten_ids,
                        backgrounds=None, absgrad=False, counters=None):
    """means2d[C,N,2] conics[C,N,3] colors[C,N,D] opacities[C,N] backgrounds[C,D] -> colors[C,H,W,D],
    alphas[C,H,W,1], last_ids (one blend of all D channels)."""
    return _RasterizeFeatures.apply(means2d, conics, colors, opacities, backgrounds, width, height, tile_size,
                                    isect_offsets, flatten_ids, absgrad, counters)


def rasterization_features(
    means: Tensor, quats: Tensor, scales: Tensor, opacities: Tensor, colors: Tensor, viewmats: Tensor, Ks: Tensor,
    width: int, height: int, near_plane: float = 0.01, far_plane: float = 1e10, radius_clip: float = 0.0,
    eps2d: float = 0.3, backgrounds: Optional[Tensor] = None, absgrad: bool = False, rasterize_mode: str = "classic",
    counters: Optional[dict] = None, tile_size: int = 16, **_unused,
):
    """``oracle.gsplat_oracle.rasterization`` with ``sh_degree=None`` for colours [N,D] / [C,N,D] of any width, blended in
    CHANNEL_CHUNK-channel chunks (module docstring).  Returns (render_colors[C,H,W,D], render_alphas[C,H,W,1], meta)."""
    if rasterize_mode not in ("classic", "antialiased"):
        raise NotImplementedError("oracle covers rasterize_mode='classic'/'antialiased'")
    N, C = means.shape[0], viewmats.shape[0]
    proj = O.fully_fused_projection(means, quats, scales, viewmats, Ks, width, height, eps2d, near_plane, far_plane,
                                    radius_clip, calc_compensations=rasterize_mode == "antialiased")
    radii, means2d, depths, conics = proj[:4]
    opac = opacities[None, :].expand(C, N)
    if rasterize_mode == "antialiased":
        opac = opac * proj[4]
    cols = colors[None].expand(C, N, colors.shape[-1]) if colors.dim() == 2 else colors
    tw, th = math.ceil(width / tile_size), math.ceil(height / tile_size)
    tiles_per_gauss, isect_ids, flatten_ids = O.isect_tiles(means2d.detach(), radii, depths.detach(), tile_size, tw, th)
    isect_offsets = O.isect_offset_encode(isect_ids, C, tw, th)
    D = cols.shape[-1]
    chunks, views = [], []
    for c0 in range(0, D, CHANNEL_CHUNK):
        # with several chunks every chunk tags .absgrad on its own view of means2d; a hook on means2d sums them once all
        # chunks' backward passes have run
        m2 = means2d.view_as(means2d) if absgrad and D > CHANNEL_CHUNK else means2d
        views.append(m2)
        bg = None if backgrounds is None else backgrounds[:, c0:c0 + CHANNEL_CHUNK]
        chunks.append(rasterize_to_pixels(m2, conics, cols[..., c0:c0 + CHANNEL_CHUNK], opac, width, height, tile_size,
                                          isect_offsets, flatten_ids, backgrounds=bg, absgrad=absgrad,
                                          counters=counters if c0 == 0 else None))
    render_colors = torch.cat([ch[0] for ch in chunks], -1)
    render_alphas, last_ids = chunks[0][1], chunks[0][2]
    if absgrad and D > CHANNEL_CHUNK and means2d.requires_grad:
        def _sum_absgrad(grad):
            means2d.absgrad = sum(v.absgrad for v in views)
        means2d.register_hook(_sum_absgrad)
    meta = {
        "camera_ids": None, "gaussian_ids": None, "radii": radii, "means2d": means2d, "depths": depths,
        "conics": conics, "opacities": opac, "colors": cols, "tile_width": tw, "tile_height": th,
        "tiles_per_gauss": tiles_per_gauss, "isect_ids": isect_ids, "flatten_ids": flatten_ids,
        "isect_offsets": isect_offsets, "last_ids": last_ids, "width": width, "height": height,
        "tile_size": tile_size, "n_cameras": C,
    }
    return render_colors, render_alphas, meta
