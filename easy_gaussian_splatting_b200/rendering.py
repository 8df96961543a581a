"""Drop-in for ``gsplat.rendering.rasterization`` — the one call the reference makes into its
rasterizer (/root/reference/model/gaussian.py:8 import, :353-367 call site).

Same Python signature, same outputs: ``(render_colors[C,H,W,3], render_alphas[C,H,W,1], meta)``
with ``meta["radii"]`` int32 ``[C,N]`` (> 0 iff visible) and ``meta["means2d"]`` fp32 ``[C,N,2]`` which,
after ``backward()`` with ``absgrad=True``, carries the attribute ``.absgrad`` ``[C,N,2]`` that
``GaussianModel.update_statistics`` reads (/root/reference/model/gaussian.py:188-197).

The host side is PyTorch (allocation, autograd wiring, streams) over the C-ABI library in
``include/egs_raster.h``; every stage is a hand-written sm_100a kernel and there is no CPU path.

One autograd node covers the whole pipeline so the backward pass stays fused:
``rasterize_bwd`` accumulates packed 48-byte gradient records that the fused SH+projection
backward consumes directly (no unpacking pass, no per-stage autograd nodes).
"""
from __future__ import annotations

import weakref
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import stages

__all__ = ["rasterization", "rasterization_camera_model", "rasterization_from_parameters"]


class _LazyMeta(dict):
    """``meta`` dict whose ``isect_ids`` entry (64-bit sorted keys, pure meta data: nothing downstream of the
    reference reads it) is rebuilt on first access instead of costing a pass over every intersection per call.
    Every way of reading the dict resolves the entry first — ``meta[k]``, ``get``, ``pop``, ``items``, ``values``,
    ``copy``, ``dict(meta)`` / ``{**meta}`` (``__iter__`` is overridden on purpose: CPython then builds the copy
    through ``keys()`` + ``__getitem__`` instead of memcpy-ing the raw slots) and pickling / ``torch.save``."""

    def _resolve(self, key):
        v = dict.__getitem__(self, key)
        if callable(v) and not isinstance(v, torch.Tensor):
            v = v()
            dict.__setitem__(self, key, v)
        return v

    def _resolve_all(self):
        for k in dict.keys(self):
            self._resolve(k)
        return self

    def __getitem__(self, key):
        return self._resolve(key)

    def __iter__(self):
        return dict.__iter__(self)

    def get(self, key, default=None):
        return self._resolve(key) if key in self else default

    def pop(self, key, *default):
        if key in self:
            self._resolve(key)
        return dict.pop(self, key, *default)

    def popitem(self):
        self._resolve_all()
        return dict.popitem(self)

    def setdefault(self, key, default=None):
        if key in self:
            return self._resolve(key)
        return dict.setdefault(self, key, default)

    def items(self):
        return [(k, self._resolve(k)) for k in self.keys()]

    def values(self):
        return [self._resolve(k) for k in self.keys()]

    def copy(self):
        return dict(self.items())

    __copy__ = copy

    def __or__(self, other):
        return {**self.copy(), **other}

    def __ror__(self, other):
        return {**other, **self.copy()}

    def __reduce__(self):
        return (dict, (self.copy(),))


class _ClassicLists:
    """gsplat's own intersection lists — ``isect_ids``, ``flatten_ids``, ``isect_offsets``: every Gaussian in every
    tile of its 3-sigma square — computed on first access with the classic route (64-bit keys, 6-pass sort, offset
    encode; bit-identical to gsplat 1.0.0's ``isect_tiles`` / ``isect_offset_encode``).  The blend kernels work from
    TIGHT lists (stages.isect_sorted_async(splats=...): a third fewer entries, same pixels and gradients), and nothing
    downstream of the reference reads these three meta entries, so building them per call would be wasted work."""

    def __init__(self, means2d: Tensor, radii: Tensor, depths: Tensor, tiles_per_gauss: Tensor, tile_width: int, tile_height: int):
        self._args = (means2d.detach(), radii, depths, tiles_per_gauss, tile_width, tile_height)
        self._lists = None

    def _get(self):
        if self._lists is None:
            means2d, radii, depths, tpg, tw, th = self._args
            _, ids, flat = stages.isect_tiles(means2d, radii, depths, stages.TILE_SIZE, tw, th, sort=True, tiles_per_gauss=tpg)
            self._lists = (ids, flat, stages.isect_offset_encode(ids, radii.shape[0], tw, th))
            self._args = None
        return self._lists

    def isect_ids(self) -> Tensor:
        return self._get()[0]

    def flatten_ids(self) -> Tensor:
        return self._get()[1]

    def isect_offsets(self) -> Tensor:
        return self._get()[2]


def _tag_absgrad(target: Tensor, absgrad: Tensor, packed_index: Optional[Tensor]) -> None:
    """``meta["means2d"].absgrad`` in the layout of ``meta["means2d"]``: dense [C,N,2], or [nnz,2] when packed."""
    target.absgrad = absgrad if packed_index is None else absgrad.reshape(-1, 2)[packed_index]


def _bin_and_blend(ctx, proj, backgrounds, width, height, grad_enabled=True, features=None, depth=False):
    """Binning + blend forward, enqueued without waiting for the intersection count (stages.isect_sorted_async): the
    buffers are sized from the previous call of this shape, the count is looked at only after the blend forward is
    in the queue, and a guess that turns out too small is repaired by running both again with the exact size.
    When a backward pass will follow and the previous call saw outlier-long tile lists, the checkpointed forward is
    used so that the backward pass can replay those lists in segments (stages.segment_policy).
    (grad_enabled is the CALLER's grad mode: inside Function.forward it is always off, and needs_input_grad stays
    true under no_grad.)  features: colours of any width ([N,D] / [C,N,D]) blended by the feature kernels instead of
    the colours in the splat records; they are never checkpointed.  depth: the RGB blend with the depth as a fourth
    channel (stages.rasterize_fwd_depth), never checkpointed either."""
    tw, th = stages.tile_grid(width, height)
    C = proj["radii"].shape[0]
    dev = proj["radii"].device
    seg, seg_min = 0, 0
    if features is None and not depth and grad_enabled and any(ctx.needs_input_grad):
        seg, seg_min = stages.segment_policy(stages.binning_hint(C, tw, th, dev), C * tw * th)
    capacity = None
    while True:
        with stages.nvtx_range("egs.binning"):
            b = stages.isect_sorted_async(proj["means2d"], proj["radii"], proj["depths"], proj["tiles_per_gauss"],
                                          stages.TILE_SIZE, tw, th, capacity=capacity, tight_rects=proj["tight_rects"])
        with stages.nvtx_range("egs.rasterize_fwd"):
            ckpt = None
            if features is not None:
                rc, ra, last = stages.rasterize_fwd_features(proj["splats"], b.offsets, b.flat_cap, features, backgrounds,
                                                             width, height, n_isects=b.raster_n, tile_order=b.tile_order)
            elif depth:
                rc, ra, last = stages.rasterize_fwd_depth(proj["splats"], b.offsets, b.flat_cap, backgrounds, width, height,
                                                          n_isects=b.raster_n, tile_order=b.tile_order)
            elif seg > 0:
                rc, ra, last, ckpt = stages.rasterize_fwd_checkpointed(proj["splats"], b.offsets, b.flat_cap, backgrounds, width,
                                                                       height, seg, seg_min_len=seg_min, n_isects=b.raster_n,
                                                                       tile_order=b.tile_order)
            else:
                rc, ra, last = stages.rasterize_fwd(proj["splats"], b.offsets, b.flat_cap, backgrounds, width, height,
                                                    n_isects=b.raster_n, tile_order=b.tile_order)
        if b.resolve():
            break
        capacity = b.n_isects  # the guess was too small (rare): same route again, exactly sized
    b.note_for_next_call()
    ctx.segment, ctx.seg_min_len, ctx.raster_n, ctx.tile_order = seg, seg_min, b.raster_n, b.tile_order
    return b, rc, ra, last, ckpt


def _blend_backward(ctx, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_colors, render_alphas,
                    last_ids, v_colors, v_alphas, ckpt):
    with stages.nvtx_range("egs.rasterize_bwd"):
        if ckpt is not None:
            return stages.rasterize_bwd_segmented(splats, isect_offsets, flatten_ids, backgrounds, width, height,
                                                  render_colors, render_alphas, last_ids, v_colors, v_alphas, ckpt, ctx.segment,
                                                  seg_min_len=ctx.seg_min_len, n_isects=ctx.raster_n, tile_order=ctx.tile_order)
        return stages.rasterize_bwd(splats, isect_offsets, flatten_ids, backgrounds, width, height, render_alphas, last_ids,
                                    v_colors, v_alphas, n_isects=ctx.raster_n, tile_order=ctx.tile_order)


def _zero_rgb(means: Tensor) -> Tensor:
    """The [N,3] colours the projection is given when the blend takes its colours from elsewhere (feature path)."""
    return torch.zeros(means.shape[0], 3, dtype=torch.float32, device=means.device)


DEPTH_MODES = ("ED", "RGB+ED")


def _depth_blend_inputs(mode: str, features: Optional[Tensor], backgrounds: Optional[Tensor], depths: Tensor):
    """What the blend of a depth mode takes, as gsplat builds it: (features, backgrounds).  With feature colours the
    depth is one more feature column ("RGB+ED": [C,N,D+1] rows of the colours and the depth, "ED": the depth alone)
    and its background is 0; with RGB colours the depth comes from the splat records and features stays None.  In "ED"
    the output does not depend on the background, which is not passed."""
    if mode == "ED":
        return (None if features is None else depths[..., None]), None
    if features is None:
        return None, backgrounds
    C, N = depths.shape
    rows = features if features.dim() == 3 else features[None].expand(C, N, -1)
    bg = None if backgrounds is None else torch.cat([backgrounds, backgrounds.new_zeros(C, 1)], -1)
    return torch.cat([rows, depths[..., None]], -1), bg


class _Rasterization(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means, quats, scales, opacities, colors, viewmats, Ks, backgrounds, cfg):
        width, height, sh_degree = cfg["width"], cfg["height"], cfg["sh_degree"]
        C, N = viewmats.shape[0], means.shape[0]
        # Dense, 16-byte-aligned copies ONCE (no-ops for the reference's own tensors): the same tensors feed the
        # forward kernels and are saved for the backward pass, which reads them through raw pointers — a strided
        # input such as ``viewmats = torch.linalg.inv(camtoworlds)`` must not reach it as is.
        means, quats, scales, opacities, colors, viewmats, Ks, backgrounds = stages.dense_inputs(
            means, quats, scales, opacities, colors, viewmats, Ks, backgrounds)
        # colours that are not RGB (cfg["features"], set by rasterization()) go to the feature blend; the projection gets
        # zero RGB colours
        feat = cfg.get("features", False)
        features = colors if feat else None
        rgb = _zero_rgb(means) if feat else colors
        depth = cfg.get("render_mode", "RGB") in DEPTH_MODES
        with stages.nvtx_range("egs.projection_fwd"):
            proj = stages.projection_fwd(means, quats, scales, opacities, rgb, viewmats, Ks, width, height, sh_degree,
                                         eps2d=cfg["eps2d"], near_plane=cfg["near_plane"], far_plane=cfg["far_plane"],
                                         radius_clip=cfg["radius_clip"], antialiased=cfg["antialiased"],
                                         **_camera_model_keyword(cfg))
        cfg["compensations"] = proj.get("compensations")  # non-differentiable side output, like the thunk below
        tiles_per_gauss = proj["tiles_per_gauss"]
        blend_bg = backgrounds
        if depth:
            features, blend_bg = _depth_blend_inputs(cfg["render_mode"], features, backgrounds, proj["depths"])
        binned, render_colors, render_alphas, last_ids, ckpt = _bin_and_blend(ctx, proj, blend_bg, width, height,
                                                                             cfg.get("grad_enabled", True), features,
                                                                             depth=depth and features is None)
        # meta's three list entries are gsplat's lists, built on first access (not tensors: cannot be outputs); the
        # outputs below carry the tight lists the kernels used
        cfg["classic_lists"] = _ClassicLists(proj["means2d"], proj["radii"], proj["depths"], tiles_per_gauss,
                                             *stages.tile_grid(width, height))
        flatten_ids, isect_offsets = binned.flat_cap, binned.offsets  # (capacity-sized: the exact length would be a wait)

        means2d = proj["means2d"]
        ctx.cfg = cfg
        ctx.set_materialize_grads(False)
        # the backward pass walks the same (capacity-sized) list buffer the forward kernels used
        ctx.save_for_backward(means, quats, scales, colors, viewmats, Ks, backgrounds, proj["radii"], proj["colors"],
                              proj["splats"], isect_offsets, binned.flat_cap, render_alphas, last_ids,
                              opacities, ckpt, render_colors if ckpt is not None else None,
                              *((features, blend_bg) if depth else ()))
        nondiff = (proj["radii"], proj["depths"], proj["conics"], proj["colors"], tiles_per_gauss,
                   flatten_ids, isect_offsets, last_ids)
        ctx.mark_non_differentiable(*nondiff)
        return (render_colors, render_alphas, means2d) + nondiff

    @staticmethod
    def backward(ctx, v_colors, v_alphas, v_means2d, *_unused):
        (means, quats, scales, colors, viewmats, Ks, backgrounds, radii, colors_rgb, splats, isect_offsets,
         flatten_ids, render_alphas, last_ids, opacities, ckpt, render_colors, *depth_saved) = ctx.saved_tensors
        cfg = ctx.cfg
        width, height = cfg["width"], cfg["height"]
        C = viewmats.shape[0]
        feat = cfg.get("features", False)
        mode = cfg.get("render_mode", "RGB")
        depth = mode in DEPTH_MODES
        # what the blend took: the colours and backgrounds as given, or in a depth mode _depth_blend_inputs'
        blend_feat, blend_bg = depth_saved if depth else (colors if feat else None, backgrounds)
        if v_colors is None:
            n_out = blend_feat.shape[-1] if blend_feat is not None else 4 if depth else 3
            v_colors = torch.zeros(C, height, width, n_out, dtype=torch.float32, device=means.device)
        if v_alphas is None:
            v_alphas = torch.zeros(C, height, width, 1, dtype=torch.float32, device=means.device)
        if blend_feat is not None:
            with stages.nvtx_range("egs.rasterize_bwd"):
                v_splats, v_features = stages.rasterize_bwd_features(
                    splats, isect_offsets, flatten_ids, blend_feat, blend_bg, width, height, render_alphas, last_ids,
                    v_colors, v_alphas, n_isects=ctx.raster_n, tile_order=ctx.tile_order,
                    want_features_grad=ctx.needs_input_grad[4] or depth)
            if depth:  # the depth column's gradient is the v_depth slot of the records; the rest the colours'
                v_splats[..., 11] = v_features[..., -1]
                v_features = v_features[..., :-1]
                if colors.dim() == 2 and mode != "ED":
                    v_features = v_features.sum(0)  # [N,D] colours were expanded to every camera's rows
            colors = _zero_rgb(means)  # what the projection saw; its colour gradient is discarded
        elif depth:
            with stages.nvtx_range("egs.rasterize_bwd"):
                v_splats = stages.rasterize_bwd_depth(splats, isect_offsets, flatten_ids, blend_bg, width, height,
                                                      render_alphas, last_ids, v_colors, v_alphas, n_isects=ctx.raster_n,
                                                      tile_order=ctx.tile_order)
        else:
            v_splats = _blend_backward(ctx, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_colors,
                                       render_alphas, last_ids, v_colors, v_alphas, ckpt)
        ref = getattr(ctx, "means2d_ref", None) if cfg["absgrad"] else None
        target = ref() if ref is not None else None
        # the camera keywords are passed only when their gradients are wanted: without them the call is exactly the
        # classic one
        want_cam = _camera_grad_keywords(ctx.needs_input_grad[5], ctx.needs_input_grad[6])
        if depth:
            want_cam["depth_grad"] = True
        with stages.nvtx_range("egs.projection_bwd"):
            out = stages.projection_bwd(means, quats, scales, colors, viewmats, Ks, width, height, cfg["sh_degree"],
                                        cfg["eps2d"], radii, colors_rgb, v_splats, v_means2d, want_absgrad=target is not None,
                                        antialiased_opacities=opacities if cfg["antialiased"] else None, opacities=opacities,
                                        **_camera_model_keyword(cfg), **want_cam)
        v_means, v_quats, v_scales, v_opac, v_cols = out[:5]
        if feat:
            v_cols = v_features
        v_viewmats, v_Ks = _camera_grads(out, want_cam)
        if target is not None:
            # same contract as gsplat: attribute tagging on the tensor object handed out in meta
            _tag_absgrad(target, out[5], getattr(ctx, "packed_index", None))
        v_bg = None
        if mode == "ED":  # gsplat: the output depends neither on the colours nor on the background
            v_cols = None
        elif backgrounds is not None and ctx.needs_input_grad[7]:
            vc = v_colors[..., :backgrounds.shape[-1]] if depth else v_colors  # the colour channels only
            v_bg = ((1.0 - render_alphas) * vc).sum(dim=(1, 2))
        return v_means, v_quats, v_scales, v_opac, v_cols, v_viewmats, v_Ks, v_bg, None


def _camera_model_keyword(cfg: dict) -> Dict[str, str]:
    """The projection stages' camera_model keyword: passed only for a model other than the pinhole, so that pinhole
    calls are exactly the ones rasterization() makes."""
    return {} if cfg["camera_model"] == "pinhole" else {"camera_model": cfg["camera_model"]}


def _camera_grad_keywords(want_viewmats: bool, want_Ks: bool) -> Dict[str, bool]:
    """The keywords of the projection backward stages for the camera gradients that are wanted (none: {})."""
    kw = {}
    if want_viewmats:
        kw["want_viewmats_grad"] = True
    if want_Ks:
        kw["want_Ks_grad"] = True
    return kw


def _camera_grads(out: tuple, kw: Dict[str, bool]) -> Tuple[Optional[Tensor], Optional[Tensor]]:
    """(v_viewmats, v_Ks) from the end of a projection backward stage's outputs; None for those not requested."""
    v_Ks = out[-1] if "want_Ks_grad" in kw else None
    v_viewmats = out[-2 if v_Ks is not None else -1] if "want_viewmats_grad" in kw else None
    return v_viewmats, v_Ks


class _RasterizationRaw(torch.autograd.Function):
    """Same pipeline fed with the reference's raw parameters (SURVEY.md §8f-2): exp / sigmoid / cat and their VJPs
    live inside the projection kernels, nothing else changes."""

    @staticmethod
    def forward(ctx, means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds, cfg):
        width, height, sh_degree = cfg["width"], cfg["height"], cfg["sh_degree"]
        C = viewmats.shape[0]
        means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds = stages.dense_inputs(
            means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds)
        with stages.nvtx_range("egs.projection_fwd_raw"):
            proj = stages.projection_fwd_raw(means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width,
                                             height, sh_degree, eps2d=cfg["eps2d"], near_plane=cfg["near_plane"],
                                             far_plane=cfg["far_plane"], radius_clip=cfg["radius_clip"])
        tiles_per_gauss = proj["tiles_per_gauss"]
        binned, render_colors, render_alphas, last_ids, ckpt = _bin_and_blend(ctx, proj, backgrounds, width, height,
                                                                             cfg.get("grad_enabled", True))
        cfg["classic_lists"] = _ClassicLists(proj["means2d"], proj["radii"], proj["depths"], tiles_per_gauss,
                                             *stages.tile_grid(width, height))
        flatten_ids, isect_offsets = binned.flat_cap, binned.offsets  # (capacity-sized: the exact length would be a wait)
        ctx.cfg = cfg
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds,
                              proj["radii"], proj["colors"], proj["splats"], isect_offsets, binned.flat_cap, render_alphas,
                              last_ids, ckpt, render_colors if ckpt is not None else None)
        nondiff = (proj["radii"], proj["depths"], proj["conics"], proj["colors"], tiles_per_gauss,
                   flatten_ids, isect_offsets, last_ids)
        ctx.mark_non_differentiable(*nondiff)
        return (render_colors, render_alphas, proj["means2d"]) + nondiff

    @staticmethod
    def backward(ctx, v_colors, v_alphas, v_means2d, *_unused):
        (means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds, radii, colors_rgb, splats,
         isect_offsets, flatten_ids, render_alphas, last_ids, ckpt, render_colors) = ctx.saved_tensors
        cfg = ctx.cfg
        width, height = cfg["width"], cfg["height"]
        C = viewmats.shape[0]
        if v_colors is None:
            v_colors = torch.zeros(C, height, width, 3, dtype=torch.float32, device=means.device)
        if v_alphas is None:
            v_alphas = torch.zeros(C, height, width, 1, dtype=torch.float32, device=means.device)
        v_splats = _blend_backward(ctx, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_colors,
                                   render_alphas, last_ids, v_colors, v_alphas, ckpt)
        ref = getattr(ctx, "means2d_ref", None) if cfg["absgrad"] else None
        target = ref() if ref is not None else None
        want_cam = _camera_grad_keywords(ctx.needs_input_grad[6], ctx.needs_input_grad[7])
        out = stages.projection_bwd_raw(means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width,
                                        height, cfg["sh_degree"], cfg["eps2d"], radii, colors_rgb, v_splats, v_means2d,
                                        want_absgrad=target is not None, **want_cam)
        v_viewmats, v_Ks = _camera_grads(out, want_cam)
        if target is not None:
            _tag_absgrad(target, out[6], None)
        v_bg = None
        if backgrounds is not None and ctx.needs_input_grad[8]:
            v_bg = ((1.0 - render_alphas) * v_colors).sum(dim=(1, 2))
        return (*out[:6], v_viewmats, v_Ks, v_bg, None)


def _check_inputs(means, quats, scales, opacities, colors, viewmats, Ks, sh_degree, backgrounds):
    N = means.shape[0]
    C = viewmats.shape[0]
    if means.shape != (N, 3):
        raise ValueError(f"means must be [N,3], got {tuple(means.shape)}")
    if quats.shape != (N, 4):
        raise ValueError(f"quats must be [N,4], got {tuple(quats.shape)}")
    if scales.shape != (N, 3):
        raise ValueError(f"scales must be [N,3], got {tuple(scales.shape)}")
    if opacities.shape != (N,):
        raise ValueError(f"opacities must be [N], got {tuple(opacities.shape)}")
    if viewmats.shape != (C, 4, 4):
        raise ValueError(f"viewmats must be [C,4,4], got {tuple(viewmats.shape)}")
    if Ks.shape != (C, 3, 3):
        raise ValueError(f"Ks must be [C,3,3], got {tuple(Ks.shape)}")
    D = 3
    if sh_degree is None:
        ok = (colors.dim() == 2 and colors.shape[0] == N) or (colors.dim() == 3 and colors.shape[:2] == (C, N))
        if not ok or colors.shape[-1] < 1:
            raise ValueError(f"colors must be [N,D] or [C,N,D] with D >= 1 when sh_degree is None, got {tuple(colors.shape)}")
        D = colors.shape[-1]
    else:
        ok = (colors.dim() == 3 and colors.shape[0] == N) or (colors.dim() == 4 and colors.shape[:2] == (C, N))
        if not ok or colors.shape[-1] != 3:
            raise ValueError(f"colors must be [N,K,3] or per-camera [C,N,K,3] SH coefficients, got {tuple(colors.shape)}")
        if not 0 <= sh_degree <= 4:
            raise NotImplementedError(f"sh_degree={sh_degree}: degrees 0..4 are implemented (gsplat's fast SH evaluates 0..4)")
        if (sh_degree + 1) ** 2 > colors.shape[-2]:
            raise ValueError(f"sh_degree={sh_degree} needs K >= {(sh_degree + 1) ** 2}, got K={colors.shape[-2]}")
    if backgrounds is not None and backgrounds.shape != (C, D):
        raise ValueError(f"backgrounds must be [C,{D}], got {tuple(backgrounds.shape)}")
    for name, t in (("means", means), ("quats", quats), ("scales", scales), ("opacities", opacities),
                    ("colors", colors), ("viewmats", viewmats), ("Ks", Ks), ("backgrounds", backgrounds)):
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(f"{name} is on {t.device}: this rasterizer is CUDA-only and has no CPU fallback")
        if t.device != means.device:
            raise RuntimeError(f"{name} is on {t.device} but means is on {means.device}")
        if t.dtype != torch.float32:
            raise TypeError(f"{name} must be float32, got {t.dtype}")
    if C * N >= 2 ** 31:
        raise ValueError("C*N must fit an int32 flatten id")


def rasterization(
    means: Tensor,  # [N, 3]
    quats: Tensor,  # [N, 4] wxyz, need not be normalised
    scales: Tensor,  # [N, 3]
    opacities: Tensor,  # [N]
    colors: Tensor,  # [N, K, 3] / [C, N, K, 3] SH coefficients (sh_degree given) or [N, D] / [C, N, D], D >= 1
    viewmats: Tensor,  # [C, 4, 4] world -> camera
    Ks: Tensor,  # [C, 3, 3]
    width: int,
    height: int,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    eps2d: float = 0.3,
    sh_degree: Optional[int] = None,
    packed: bool = True,
    tile_size: int = 16,
    backgrounds: Optional[Tensor] = None,
    render_mode: str = "RGB",
    sparse_grad: bool = False,
    absgrad: bool = False,
    rasterize_mode: str = "classic",
    channel_chunk: int = 32,
) -> Tuple[Tensor, Tensor, Dict]:
    """See module docstring.  The combination the reference uses — SH colours, ``packed=False``,
    ``absgrad=True``, one camera, a [1,3] background — and C > 1 are implemented; modes the
    reference never requests raise ``NotImplementedError`` instead of silently approximating.
    As in gsplat, ``viewmats`` receive a gradient when they require one (camera pose refinement: projection and SH
    view directions, campos = inverse(viewmats)[:, :3, 3]).  Beyond gsplat 1.0.0, which gives ``Ks`` no gradient,
    ``Ks`` receive one when they require it (intrinsics refinement): [C,3,3] with v_fx, v_fy, v_cx, v_cy at (0,0),
    (1,1), (0,2), (1,2) and 0 elsewhere, the exact derivative of the projection (means2d, conics and, in antialiased
    mode, the compensation), summed over each camera's visible Gaussians.
    Without SH, colours may have any number of channels D (features, masks, RGB plus extra channels): the images are
    [C,H,W,D], ``backgrounds`` [C,D], and D != 3 is blended in chunks of 32 channels by the feature kernels.  For
    D > 32, ``meta["means2d"].absgrad`` is the sum over the chunks of each chunk's absgrad (gsplat 1.0.0 keeps the
    value of whichever chunk's backward ran last).  ``channel_chunk`` is accepted and has no effect.
    With SH, coefficients may also be per camera, [C,N,K,3] (e.g. shared coefficients plus a learned per-view
    offset): camera c colours Gaussian n from its own row colors[c, n], and colors.grad is [C,N,K,3], one row per
    (camera, Gaussian), 0 for pairs the camera culls.
    ``sh_degree`` may be 0..4, as gsplat's fast SH evaluates; degree 4 needs K >= 25 and leaves the bands past 4 a
    zero gradient.
    ``render_mode`` "RGB", "ED" or "RGB+ED" (gsplat's expected depth): the camera-space depth of each Gaussian
    (``meta["depths"]``) is blended as one more channel with background 0 and divided by
    ``render_alphas.clamp(min=1e-10)``.  "RGB+ED" returns [C,H,W,D+1] (the colours, then the expected depth), "ED"
    [C,H,W,1]; ``render_alphas`` and ``meta`` are those of "RGB".  Gradients of the depth reach the geometry,
    ``viewmats`` and absgrad; in "ED" ``colors`` and ``backgrounds`` get none, in "RGB+ED" ``backgrounds`` [C,D] get the
    colour channels' gradient.  "D" and "RGB+D" raise ``NotImplementedError``.
    The camera is a pinhole; ``rasterization_camera_model`` takes orthographic and fisheye cameras as well."""
    return _rasterization(means, quats, scales, opacities, colors, viewmats, Ks, width, height, near_plane, far_plane,
                          radius_clip, eps2d, sh_degree, packed, tile_size, backgrounds, render_mode, sparse_grad, absgrad,
                          rasterize_mode, "pinhole")


CAMERA_MODELS = ("pinhole", "ortho", "fisheye")


def rasterization_camera_model(
    means: Tensor,
    quats: Tensor,
    scales: Tensor,
    opacities: Tensor,
    colors: Tensor,
    viewmats: Tensor,
    Ks: Tensor,
    width: int,
    height: int,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    eps2d: float = 0.3,
    sh_degree: Optional[int] = None,
    packed: bool = True,
    tile_size: int = 16,
    backgrounds: Optional[Tensor] = None,
    render_mode: str = "RGB",
    sparse_grad: bool = False,
    absgrad: bool = False,
    rasterize_mode: str = "classic",
    channel_chunk: int = 32,
    camera_model: str = "pinhole",
) -> Tuple[Tensor, Tensor, Dict]:
    """``rasterization()`` with a camera model, as later gsplat releases take it: ``camera_model`` "pinhole", "ortho" or
    "fisheye"; every other argument, output and gradient (``viewmats`` and ``Ks`` included) as in ``rasterization()``,
    which ``camera_model="pinhole"`` is exactly.  With (x, y, z) the camera-space mean and fx, fy, cx, cy from ``Ks``:

    - "pinhole": means2d = (fx x / z + cx, fy y / z + cy), with gsplat's 1.3 x fov clamp in the Jacobian.
    - "ortho": means2d = (fx x + cx, fy y + cy) (fx, fy in pixels per world unit), J = [[fx, 0, 0], [0, fy, 0]].
    - "fisheye": equidistant, r = sqrt(x^2 + y^2), theta = atan2(r, z): means2d = (fx x theta / r + cx,
      fy y theta / r + cy), J the exact Jacobian of means2d (gsplat's fisheye_proj).  theta / r is a polynomial that
      is exact in fp32 to 2 ulp for theta in [0, pi) and equals 1 / z on the optical axis.

    Neither "ortho" nor "fisheye" has an fov clamp, and both project z <= 0 as well: with ``near_plane <= 0``, Gaussians
    behind the camera are rendered and differentiated (fisheye theta up to pi).  The near / far cull on z, the eps2d blur, the radius, the
    off-screen test and the antialiased compensation are the same for all models, and ``meta["depths"]`` is the
    camera-space z for all of them, so "ED" renders the expected z.  ``Ks`` gradients: v_cx, v_cy sum the means2d
    cotangents and v_fx = (v_m2x (m2x - cx) + sum_j v_J0j J0j) / fx (likewise v_fy).  Any other ``camera_model`` raises
    ``ValueError``."""
    if camera_model not in CAMERA_MODELS:
        raise ValueError(f"camera_model must be one of {CAMERA_MODELS}, got {camera_model!r}")
    return _rasterization(means, quats, scales, opacities, colors, viewmats, Ks, width, height, near_plane, far_plane,
                          radius_clip, eps2d, sh_degree, packed, tile_size, backgrounds, render_mode, sparse_grad, absgrad,
                          rasterize_mode, camera_model)


def _rasterization(means, quats, scales, opacities, colors, viewmats, Ks, width, height, near_plane, far_plane,
                   radius_clip, eps2d, sh_degree, packed, tile_size, backgrounds, render_mode, sparse_grad, absgrad,
                   rasterize_mode, camera_model):
    """The one path of rasterization() and rasterization_camera_model()."""
    if render_mode not in ("RGB",) + DEPTH_MODES:
        raise NotImplementedError(f"render_mode={render_mode!r}: 'RGB', 'ED' and 'RGB+ED' are implemented")
    if rasterize_mode not in ("classic", "antialiased"):
        raise ValueError(f"rasterize_mode must be 'classic' or 'antialiased', got {rasterize_mode!r}")
    if sparse_grad:
        raise NotImplementedError("sparse_grad=True is not implemented")
    if tile_size != stages.TILE_SIZE:
        raise NotImplementedError(f"tile_size={tile_size}: the blending kernels are specialised for 16")
    width, height = int(width), int(height)
    if width < 1 or height < 1:
        raise ValueError(f"width and height must be >= 1, got {width} x {height}")
    _check_inputs(means, quats, scales, opacities, colors, viewmats, Ks, sh_degree, backgrounds)
    C = viewmats.shape[0]
    cfg = dict(width=width, height=height, sh_degree=sh_degree, eps2d=float(eps2d), near_plane=float(near_plane),
               far_plane=float(far_plane), radius_clip=float(radius_clip), absgrad=bool(absgrad),
               antialiased=rasterize_mode == "antialiased", grad_enabled=torch.is_grad_enabled(),
               features=sh_degree is None and colors.shape[-1] != 3, render_mode=render_mode, camera_model=camera_model)
    outs = _Rasterization.apply(means, quats, scales, opacities, colors, viewmats, Ks, backgrounds, cfg)
    meta_colors = None
    if cfg["features"]:  # gsplat: the colours as given, per (camera, Gaussian)
        meta_colors = colors.detach() if colors.dim() == 3 else colors.detach()[None].expand(C, -1, -1)
    opacities_cn = opacities.detach()[None].expand(C, -1)
    comp = cfg.pop("compensations", None)
    if comp is not None:
        opacities_cn = opacities_cn * comp  # gsplat: meta["opacities"] = opacities * compensations
    render_colors, render_alphas, meta = _finish(outs, cfg, opacities_cn, width, height, tile_size, C, absgrad,
                                                 packed=bool(packed), meta_colors=meta_colors)
    if render_mode in DEPTH_MODES:
        # gsplat: the accumulated depth (last channel) over the alpha is the expected depth; autograd carries the
        # division into the alpha gradient
        ed = render_colors[..., -1:] / render_alphas.clamp(min=1e-10)
        render_colors = ed if render_mode == "ED" else torch.cat([render_colors[..., :-1], ed], dim=-1)
    return render_colors, render_alphas, meta


def _finish(outs, cfg, opacities_cn, width, height, tile_size, C, absgrad, packed=False, meta_colors=None):
    (render_colors, render_alphas, means2d, radii, depths, conics, colors_rgb, tiles_per_gauss,
     _blend_flatten_ids, _blend_offsets, _last_ids) = outs
    if meta_colors is not None:
        colors_rgb = meta_colors
    classic = cfg.pop("classic_lists")
    isect_ids, flatten_ids, isect_offsets = classic.isect_ids, classic.flatten_ids, classic.isect_offsets
    cfg.pop("compensations", None)
    camera_ids = gaussian_ids = None
    node = render_colors.grad_fn
    if packed:
        # gsplat's packed layout (SURVEY.md §8b / §8f-4): per-(camera, Gaussian) tensors hold only the nnz visible
        # entries, in flat (camera, Gaussian) order, with camera_ids / gaussian_ids naming them, and flatten_ids
        # index that packed list.  The kernels above still work on the dense [C,N] intermediates — this reproduces
        # the packed INTERFACE, not upstream's memory saving; rendered images and gradients are the same either way.
        N = radii.shape[1]
        visible = radii.reshape(-1) > 0
        packed_index = visible.nonzero(as_tuple=True)[0]  # one host sync (sizes the packed tensors), as upstream
        camera_ids = torch.div(packed_index, N, rounding_mode="floor")
        gaussian_ids = packed_index - camera_ids * N
        rank = torch.cumsum(visible, 0, dtype=torch.int32) - 1  # flat (c,n) index -> row of the packed list
        dense_flatten_ids = flatten_ids
        flatten_ids = lambda: rank[dense_flatten_ids().long()]  # stays lazy: built from gsplat's list on first access
        means2d = means2d.reshape(-1, 2)[packed_index]  # differentiable gather: gradients on it reach the dense one
        radii, depths, tiles_per_gauss = (t.reshape(-1)[packed_index] for t in (radii, depths, tiles_per_gauss))
        conics, colors_rgb = (t.reshape(-1, t.shape[-1])[packed_index] for t in (conics, colors_rgb))
        opacities_cn = opacities_cn.reshape(-1)[packed_index]
        if node is not None:
            node.packed_index = packed_index
    if absgrad and node is not None:
        # the backward node tags .absgrad on exactly this tensor object (weak: no reference cycle)
        node.means2d_ref = weakref.ref(means2d)
    tw, th = stages.tile_grid(width, height)
    meta = _LazyMeta({
        "camera_ids": camera_ids,
        "gaussian_ids": gaussian_ids,
        "radii": radii,
        "means2d": means2d,
        "depths": depths,
        "conics": conics,
        "opacities": opacities_cn,
        "colors": colors_rgb,
        "tile_width": tw,
        "tile_height": th,
        "tiles_per_gauss": tiles_per_gauss,
        "isect_ids": isect_ids,
        "flatten_ids": flatten_ids,
        "isect_offsets": isect_offsets,
        "width": width,
        "height": height,
        "tile_size": tile_size,
        "n_cameras": C,
    })
    return render_colors, render_alphas, meta


def rasterization_from_parameters(
    means: Tensor,  # [N, 3]
    quats: Tensor,  # [N, 4]
    log_scales: Tensor,  # [N, 3]   (GaussianModel.log_scales)
    logit_opacities: Tensor,  # [N]  (GaussianModel.logit_opacities)
    sh_0: Tensor,  # [N, 1, 3]
    sh_rest: Tensor,  # [N, 15, 3]
    viewmats: Tensor,
    Ks: Tensor,
    width: int,
    height: int,
    sh_degree: int,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    eps2d: float = 0.3,
    backgrounds: Optional[Tensor] = None,
    absgrad: bool = False,
) -> Tuple[Tensor, Tensor, Dict]:
    """Opt-in entry point (SURVEY.md §8f-2): identical to
    ``rasterization(means, quats, exp(log_scales), sigmoid(logit_opacities), cat([sh_0, sh_rest], 1), ...,
    packed=False)`` — what ``GaussianModel.forward`` computes through its ``scales`` / ``opacities`` / ``shs``
    properties (/root/reference/model/gaussian.py:97-107, 353-367) — but the three activations and their backward
    passes run inside the projection kernels: no ``cat`` (384 B/Gaussian each way), no separate exp / sigmoid
    kernels, and gradients arrive directly on the six parameter tensors.  ``viewmats`` and ``Ks`` receive gradients
    when they require them, as in ``rasterization()``."""
    width, height = int(width), int(height)
    if width < 1 or height < 1:
        raise ValueError(f"width and height must be >= 1, got {width} x {height}")
    N, C = means.shape[0], viewmats.shape[0]
    if log_scales.shape != (N, 3) or logit_opacities.shape != (N,):
        raise ValueError("log_scales must be [N,3] and logit_opacities [N]")
    if sh_0.shape != (N, 1, 3) or sh_rest.shape != (N, 15, 3):
        raise ValueError("sh_0 must be [N,1,3] and sh_rest [N,15,3] (K = 16, the reference's sh_degree 3 layout)")
    # shape / device / dtype checks shared with rasterization(); sh_0.expand is a zero-copy [N,16,3] stand-in
    _check_inputs(means, quats, log_scales, logit_opacities, sh_0.expand(N, 16, 3), viewmats, Ks, sh_degree, backgrounds)
    for name, t in (("sh_0", sh_0), ("sh_rest", sh_rest)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"{name} must be a float32 CUDA tensor: this rasterizer has no CPU path")
    cfg = dict(width=width, height=height, sh_degree=int(sh_degree), eps2d=float(eps2d), near_plane=float(near_plane),
               far_plane=float(far_plane), radius_clip=float(radius_clip), absgrad=bool(absgrad),
               grad_enabled=torch.is_grad_enabled())
    outs = _RasterizationRaw.apply(means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, backgrounds, cfg)
    opac = torch.sigmoid(logit_opacities.detach())[None].expand(C, -1)
    return _finish(outs, cfg, opac, width, height, 16, C, absgrad)
