"""Per-stage operators over the C-ABI (tensor in -> tensor out, no autograd).

Names and argument meaning mirror the gsplat-1.0.0 operators that sit behind the reference's
``rasterization`` call (/root/reference/model/gaussian.py:353-367; SURVEY.md §2.1): projection (+SH),
``isect_tiles``, ``isect_offset_encode``, ``rasterize_to_pixels`` fwd/bwd.  All tensors must be CUDA,
fp32/int32/int64 and are made contiguous here; every launch goes to the current stream of the
tensors' device (viewer threads never call ``set_device``, SURVEY.md §3.3, so the device is pinned
around each call).
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import os
import threading
import weakref
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib

SPLAT_FLOATS = 12
TILE_SIZE = 16


# Tracing (SURVEY.md section 5: the reference has none): EGS_NVTX=1 wraps every stage of a call in an NVTX range, so an
# Nsight timeline shows projection / binning / blend fwd / blend bwd / projection bwd by name.  Off by default and
# free when off (a shared null context).
_NVTX = os.environ.get("EGS_NVTX", "0") == "1"
_NULL_CONTEXT = contextlib.nullcontext()


@contextlib.contextmanager
def _nvtx_on(name: str):
    torch.cuda.nvtx.range_push(name)
    try:
        yield
    finally:
        torch.cuda.nvtx.range_pop()


def nvtx_range(name: str):
    return _nvtx_on(name) if _NVTX else _NULL_CONTEXT


# Caller-owned gradient storage (see distributed.FlatGradBucket.begin_direct): (device, parameter data_ptr) -> buffer.
# The projection backward writes EVERY element of every parameter gradient exactly once, so it can write straight
# into a registered buffer — no zero fill, no accumulate pass, and ``param.grad`` becomes a view of the caller's bucket.
# A registration is ONE-SHOT: the backward pass that uses it removes it, so a second backward on the same parameters
# inside the same begin_direct / end_direct window takes the ordinary allocate-and-accumulate route instead of
# overwriting the first gradient.  The table is guarded by a lock (a viewer thread may render while the training
# thread is inside the window; renders under no_grad never touch it).
_GRAD_TARGETS: Dict[Tuple[int, int], Tuple["weakref.ref", Tensor]] = {}
_GRAD_TARGETS_LOCK = threading.Lock()


def _target_key(t: Tensor) -> Tuple[int, int]:
    return (t.device.index if t.device.index is not None else -1, t.data_ptr())


def register_grad_target(param: Tensor, buffer: Tensor) -> None:
    if buffer.numel() != param.numel() or buffer.dtype != param.dtype or buffer.device != param.device or not buffer.is_contiguous():
        raise ValueError("gradient target must be a contiguous buffer of the parameter's size, dtype and device")
    with _GRAD_TARGETS_LOCK:
        _GRAD_TARGETS[_target_key(param)] = (weakref.ref(param), buffer)


def clear_grad_targets() -> None:
    with _GRAD_TARGETS_LOCK:
        _GRAD_TARGETS.clear()


def _grad_buffer(inp: Tensor) -> Tensor:
    """Storage for the gradient of ``inp``: always dense row-major (the kernels write row-major whatever the strides
    of the input were) and 16-byte aligned (float4 stores)."""
    if _GRAD_TARGETS:
        with _GRAD_TARGETS_LOCK:
            entry = _GRAD_TARGETS.get(_target_key(inp))
            if entry is not None:
                owner, tgt = entry
                live = owner()  # a registration whose parameter is gone must not capture a new tensor at the same address
                if (live is not None and live.data_ptr() == inp.data_ptr() and live.shape == inp.shape
                        and inp.is_contiguous() and tgt.data_ptr() % 16 == 0):
                    del _GRAD_TARGETS[_target_key(inp)]  # one-shot
                    return tgt.view(inp.shape)  # a fresh tensor object over the caller's storage: autograd adopts it as .grad
    return torch.empty(inp.shape, dtype=inp.dtype, device=inp.device)


def _ptr(t: Optional[Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _f32c(t: Tensor, name: str) -> Tensor:
    """float32 CUDA tensor -> dense row-major and 16-byte aligned (the kernels use 128-bit loads on quats, SH rows
    and the packed records); a no-op for tensors that already are, a copy otherwise (e.g. a slice of a flat
    parameter buffer that starts at an odd element)."""
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: this rasterizer has no CPU path")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    t = t.contiguous()
    if t.data_ptr() % 16 != 0:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


def dense_inputs(*tensors: Optional[Tensor]):
    """The tensors of a rasterization call as dense, aligned fp32 tensors (``None`` stays ``None``).  Identity for
    tensors that already are — in particular parameter tensors keep their identity, which the gradient-target
    registry keys on."""
    out = []
    for t in tensors:
        if t is None or (t.is_contiguous() and t.data_ptr() % 16 == 0):
            out.append(t)
        else:
            out.append(t.clone(memory_format=torch.contiguous_format) if t.is_contiguous() else t.contiguous())
            if out[-1].data_ptr() % 16 != 0:  # cannot happen with the caching allocator; keep the contract explicit
                raise RuntimeError("allocator returned a tensor that is not 16-byte aligned")
    return tuple(out)


def tile_grid(width: int, height: int, tile_size: int = TILE_SIZE) -> Tuple[int, int]:
    return math.ceil(width / tile_size), math.ceil(height / tile_size)


def tile_n_bits(tile_width: int, tile_height: int) -> int:
    return int(math.floor(math.log2(tile_width * tile_height))) + 1


def camera_n_bits(C: int) -> int:
    return int(math.floor(math.log2(C))) + 1 if C > 1 else 0


# Level 1 of the two-level binning route sorts the visible Gaussians of all cameras on these key bits
LEVEL1_KEY_BYTES = 4


def level1_end_bit(C: int) -> int:
    """Depth bits only: level 2 sorts stably on the (camera, tile) index, which also separates the cameras."""
    return 32


# camera_model codes of the ABI's camera-model entries (include/egs_raster.h); "pinhole" uses the other entries
CAMERA_MODELS = {"pinhole": 0, "ortho": 1, "fisheye": 2}


def _camera_model_code(camera_model: str) -> int:
    if camera_model not in CAMERA_MODELS:
        raise ValueError(f"camera_model must be one of {tuple(CAMERA_MODELS)}, got {camera_model!r}")
    return CAMERA_MODELS[camera_model]


def projection_fwd(means: Tensor, quats: Tensor, scales: Tensor, opacities: Tensor, colors: Tensor,
                   viewmats: Tensor, Ks: Tensor, width: int, height: int, sh_degree: Optional[int],
                   eps2d: float = 0.3, near_plane: float = 0.01, far_plane: float = 1e10,
                   radius_clip: float = 0.0, tile_size: int = TILE_SIZE,
                   antialiased: bool = False, camera_model: str = "pinhole") -> Dict[str, Tensor]:
    """g1+g2+count(g3).  colors: [N,K,3] or per-camera [C,N,K,3] SH coefficients when sh_degree is not None, else
    [N,3]/[C,N,3].
    antialiased: gsplat's rasterize_mode="antialiased" — adds out["compensations"] [C,N]; the splat records then
    carry opacity * compensation.
    camera_model: "pinhole", "ortho" or "fisheye" (egs_projection_fwd_camera_model for the latter two)."""
    cm = _camera_model_code(camera_model)
    lib = _lib.load()
    means, quats, scales = _f32c(means, "means"), _f32c(quats, "quats"), _f32c(scales, "scales")
    opacities, colors = _f32c(opacities, "opacities"), _f32c(colors, "colors")
    viewmats, Ks = _f32c(viewmats, "viewmats"), _f32c(Ks, "Ks")
    dev = means.device
    N, C = means.shape[0], viewmats.shape[0]
    if sh_degree is None:
        K, deg, per_cam = 1, -1, int(colors.dim() == 3)
    else:
        K, deg, per_cam = colors.shape[-2], int(sh_degree), int(colors.dim() == 4)
    tw, th = tile_grid(width, height, tile_size)
    out = {
        "radii": torch.empty(C, N, dtype=torch.int32, device=dev),
        "means2d": torch.empty(C, N, 2, dtype=torch.float32, device=dev),
        "depths": torch.empty(C, N, dtype=torch.float32, device=dev),
        "conics": torch.empty(C, N, 3, dtype=torch.float32, device=dev),
        "colors": torch.empty(C, N, 3, dtype=torch.float32, device=dev),
        "tiles_per_gauss": torch.empty(C, N, dtype=torch.int32, device=dev),
        "tight_rects": torch.empty(C, N, 2, dtype=torch.int32, device=dev),
        "splats": torch.empty(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev),
    }
    args = (C, N, _ptr(means), _ptr(quats), _ptr(scales), _ptr(opacities), _ptr(colors), K, deg, per_cam,
            _ptr(viewmats), _ptr(Ks), int(width), int(height), float(eps2d), float(near_plane), float(far_plane),
            float(radius_clip), int(tile_size), tw, th, _ptr(out["radii"]), _ptr(out["means2d"]), _ptr(out["depths"]),
            _ptr(out["conics"]), _ptr(out["colors"]), _ptr(out["tiles_per_gauss"]), _ptr(out["tight_rects"]),
            _ptr(out["splats"]))
    with torch.cuda.device(dev):
        if antialiased:
            out["compensations"] = torch.empty(C, N, dtype=torch.float32, device=dev)
        if cm:
            rc = lib.egs_projection_fwd_camera_model(cm, *args, _ptr(out.get("compensations")), _stream(dev))
        elif antialiased:
            rc = lib.egs_projection_fwd_antialiased(*args, _ptr(out["compensations"]), _stream(dev))
        else:
            rc = lib.egs_projection_fwd(*args, _stream(dev))
    _lib.check(rc, "egs_projection_fwd")
    return out


def projection_bwd(means: Tensor, quats: Tensor, scales: Tensor, colors: Tensor, viewmats: Tensor, Ks: Tensor,
                   width: int, height: int, sh_degree: Optional[int], eps2d: float, radii: Tensor,
                   colors_rgb: Tensor, v_splats: Tensor, v_means2d_extra: Optional[Tensor] = None,
                   want_absgrad: bool = False, antialiased_opacities: Optional[Tensor] = None,
                   opacities: Optional[Tensor] = None, want_viewmats_grad: bool = False, want_Ks_grad: bool = False,
                   depth_grad: bool = False, camera_model: str = "pinhole"):
    """g8+g9. -> v_means[N,3], v_quats[N,4], v_scales[N,3], v_opacities[N], v_colors (shape of colors)
    (+ absgrad[C,N,2] when want_absgrad) (+ v_viewmats[C,4,4] when want_viewmats_grad) (+ v_Ks[C,3,3] when
    want_Ks_grad, always last).
    antialiased_opacities: the opacities[N] of an antialiased forward; opacities: only consulted for a registered
    gradient buffer (register_grad_target).
    depth_grad: also take slot 11 of v_splats (v_depth, from rasterize_bwd_depth) as the gradient w.r.t. the
    camera-space depths (egs_projection_bwd_depth); otherwise that slot is not read.
    camera_model: "pinhole", "ortho" or "fisheye"; the latter two always go through egs_projection_bwd_camera_model,
    which always reads slot 11 (0 unless the blend was a depth one)."""
    cm = _camera_model_code(camera_model)
    lib = _lib.load()
    dev = means.device
    means, quats, scales, colors, viewmats, Ks = dense_inputs(means, quats, scales, colors, viewmats, Ks)
    radii, colors_rgb, v_splats = radii.contiguous(), colors_rgb.contiguous(), v_splats.contiguous()
    N, C = means.shape[0], viewmats.shape[0]
    if sh_degree is None:
        K, deg, per_cam = 1, -1, int(colors.dim() == 3)
    else:
        K, deg, per_cam = colors.shape[-2], int(sh_degree), int(colors.dim() == 4)
    op_ref = antialiased_opacities if antialiased_opacities is not None else opacities
    if op_ref is not None:
        v_means, v_quats, v_scales, v_opac, v_colors = [_grad_buffer(t) for t in (means, quats, scales, op_ref, colors)]
    else:
        v_means, v_quats, v_scales, v_colors = [_grad_buffer(t) for t in (means, quats, scales, colors)]
        v_opac = torch.empty(N, dtype=torch.float32, device=dev)
    if v_means2d_extra is not None:
        v_means2d_extra = _f32c(v_means2d_extra, "v_means2d")
    absgrad = torch.empty(C, N, 2, dtype=torch.float32, device=dev) if want_absgrad else None
    tail = (_ptr(colors), K, deg, per_cam, _ptr(viewmats), _ptr(Ks), int(width), int(height), float(eps2d),
            _ptr(radii), _ptr(colors_rgb), _ptr(v_splats), _ptr(v_means2d_extra), _ptr(v_means), _ptr(v_quats),
            _ptr(v_scales), _ptr(v_opac), _ptr(v_colors), _ptr(absgrad), _stream(dev))
    v_viewmats = v_Ks = None
    with torch.cuda.device(dev):
        if want_viewmats_grad:
            v_viewmats = torch.empty(C, 4, 4, dtype=torch.float32, device=dev)
        if want_Ks_grad or want_viewmats_grad or depth_grad or cm:
            aa = antialiased_opacities is not None
            aa_op = _f32c(antialiased_opacities, "opacities") if aa else None
            head = (C, N, _ptr(means), _ptr(quats), _ptr(scales), _ptr(aa_op), *tail[:-1], int(aa), _ptr(v_viewmats))
        if depth_grad or cm:
            if want_Ks_grad:
                v_Ks = torch.empty(C, 3, 3, dtype=torch.float32, device=dev)
            ws = (_intrinsics_workspace(lib, C, N, dev) if want_Ks_grad else _viewmats_workspace(lib, C, N, dev)
                  if want_viewmats_grad else None)
            ws_args = (_ptr(v_Ks), _ptr(ws), 0 if ws is None else ws.numel(), tail[-1])
            if cm:
                rc = lib.egs_projection_bwd_camera_model(cm, *head, *ws_args)
            else:
                rc = lib.egs_projection_bwd_depth(*head, *ws_args)
        elif want_Ks_grad:  # one launch for both camera gradients
            v_Ks = torch.empty(C, 3, 3, dtype=torch.float32, device=dev)
            ws = _intrinsics_workspace(lib, C, N, dev)
            rc = lib.egs_projection_bwd_intrinsics(*head, _ptr(v_Ks), _ptr(ws), ws.numel(), tail[-1])
        elif want_viewmats_grad:
            ws = _viewmats_workspace(lib, C, N, dev)
            rc = lib.egs_projection_bwd_viewmats(*head, _ptr(ws), ws.numel(), tail[-1])
        elif antialiased_opacities is not None:
            aa_op = _f32c(antialiased_opacities, "opacities")
            rc = lib.egs_projection_bwd_antialiased(C, N, _ptr(means), _ptr(quats), _ptr(scales), _ptr(aa_op), *tail)
        else:
            rc = lib.egs_projection_bwd(C, N, _ptr(means), _ptr(quats), _ptr(scales), *tail)
    _lib.check(rc, "egs_projection_bwd")
    out = (v_means, v_quats, v_scales, v_opac, v_colors) + ((absgrad,) if want_absgrad else ())
    return _with_camera_grads(out, v_viewmats, v_Ks)


def _with_camera_grads(out: tuple, v_viewmats: Optional[Tensor], v_Ks: Optional[Tensor]) -> tuple:
    """out (+ v_viewmats) (+ v_Ks): only the camera gradients that were asked for, v_Ks last."""
    return out + tuple(t for t in (v_viewmats, v_Ks) if t is not None)


def _viewmats_workspace(lib, C: int, N: int, dev) -> Tensor:
    """Scratch of the view-matrix gradient (per-warp partials, see include/egs_raster.h); 16-byte aligned."""
    return torch.empty(max(lib.egs_projection_bwd_viewmats_workspace_bytes(C, N), 16), dtype=torch.uint8, device=dev)


def _intrinsics_workspace(lib, C: int, N: int, dev) -> Tensor:
    """Scratch of the intrinsics (and view-matrix) gradients: wider per-warp partials; 16-byte aligned."""
    return torch.empty(max(lib.egs_projection_bwd_intrinsics_workspace_bytes(C, N), 16), dtype=torch.uint8, device=dev)


def projection_fwd_raw(means: Tensor, quats: Tensor, log_scales: Tensor, logit_opacities: Tensor, sh_0: Tensor,
                       sh_rest: Tensor, viewmats: Tensor, Ks: Tensor, width: int, height: int, sh_degree: int,
                       eps2d: float = 0.3, near_plane: float = 0.01, far_plane: float = 1e10,
                       radius_clip: float = 0.0, tile_size: int = TILE_SIZE) -> Dict[str, Tensor]:
    """§8f-2: projection_fwd on the reference's raw parameters (exp / sigmoid / cat folded into the kernel)."""
    lib = _lib.load()
    ts = [_f32c(t, n) for t, n in ((means, "means"), (quats, "quats"), (log_scales, "log_scales"),
                                   (logit_opacities, "logit_opacities"), (sh_0, "sh_0"), (sh_rest, "sh_rest"),
                                   (viewmats, "viewmats"), (Ks, "Ks"))]
    means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks = ts
    dev = means.device
    N, C = means.shape[0], viewmats.shape[0]
    if sh_0.shape != (N, 1, 3) or sh_rest.shape != (N, 15, 3):
        raise ValueError(f"sh_0 must be [N,1,3] and sh_rest [N,15,3], got {tuple(sh_0.shape)} and {tuple(sh_rest.shape)}")
    tw, th = tile_grid(width, height, tile_size)
    out = {
        "radii": torch.empty(C, N, dtype=torch.int32, device=dev),
        "means2d": torch.empty(C, N, 2, dtype=torch.float32, device=dev),
        "depths": torch.empty(C, N, dtype=torch.float32, device=dev),
        "conics": torch.empty(C, N, 3, dtype=torch.float32, device=dev),
        "colors": torch.empty(C, N, 3, dtype=torch.float32, device=dev),
        "tiles_per_gauss": torch.empty(C, N, dtype=torch.int32, device=dev),
        "tight_rects": torch.empty(C, N, 2, dtype=torch.int32, device=dev),
        "splats": torch.empty(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev),
    }
    with torch.cuda.device(dev):
        rc = lib.egs_projection_fwd_raw(C, N, _ptr(means), _ptr(quats), _ptr(log_scales), _ptr(logit_opacities),
                                        _ptr(sh_0), _ptr(sh_rest), int(sh_degree), _ptr(viewmats), _ptr(Ks),
                                        int(width), int(height), float(eps2d), float(near_plane), float(far_plane),
                                        float(radius_clip), int(tile_size), tw, th, _ptr(out["radii"]),
                                        _ptr(out["means2d"]), _ptr(out["depths"]), _ptr(out["conics"]),
                                        _ptr(out["colors"]), _ptr(out["tiles_per_gauss"]), _ptr(out["tight_rects"]),
                                        _ptr(out["splats"]), _stream(dev))
    _lib.check(rc, "egs_projection_fwd_raw")
    return out


def projection_bwd_raw(means: Tensor, quats: Tensor, log_scales: Tensor, logit_opacities: Tensor, sh_0: Tensor,
                       sh_rest: Tensor, viewmats: Tensor, Ks: Tensor, width: int, height: int, sh_degree: int,
                       eps2d: float, radii: Tensor, colors_rgb: Tensor, v_splats: Tensor,
                       v_means2d_extra: Optional[Tensor] = None, want_absgrad: bool = False,
                       want_viewmats_grad: bool = False, want_Ks_grad: bool = False):
    """-> v_means, v_quats, v_log_scales, v_logit_opacities, v_sh_0, v_sh_rest (, absgrad) (, v_viewmats[C,4,4])
    (, v_Ks[C,3,3])."""
    lib = _lib.load()
    dev = means.device
    means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks = dense_inputs(
        means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks)
    radii, colors_rgb, v_splats = radii.contiguous(), colors_rgb.contiguous(), v_splats.contiguous()
    N, C = means.shape[0], viewmats.shape[0]
    outs = [_grad_buffer(t) for t in (means, quats, log_scales, logit_opacities, sh_0, sh_rest)]
    if v_means2d_extra is not None:
        v_means2d_extra = _f32c(v_means2d_extra, "v_means2d")
    absgrad = torch.empty(C, N, 2, dtype=torch.float32, device=dev) if want_absgrad else None
    args = (C, N, _ptr(means), _ptr(quats), _ptr(log_scales), _ptr(logit_opacities), _ptr(sh_0), _ptr(sh_rest),
            int(sh_degree), _ptr(viewmats), _ptr(Ks), int(width), int(height), float(eps2d), _ptr(radii), _ptr(colors_rgb),
            _ptr(v_splats), _ptr(v_means2d_extra), *[_ptr(o) for o in outs], _ptr(absgrad))
    v_viewmats = v_Ks = None
    with torch.cuda.device(dev):
        if want_viewmats_grad:
            v_viewmats = torch.empty(C, 4, 4, dtype=torch.float32, device=dev)
        if want_Ks_grad:  # one launch for both camera gradients
            v_Ks = torch.empty(C, 3, 3, dtype=torch.float32, device=dev)
            ws = _intrinsics_workspace(lib, C, N, dev)
            rc = lib.egs_projection_bwd_raw_intrinsics(*args, _ptr(v_viewmats), _ptr(v_Ks), _ptr(ws), ws.numel(),
                                                       _stream(dev))
        elif want_viewmats_grad:
            ws = _viewmats_workspace(lib, C, N, dev)
            rc = lib.egs_projection_bwd_raw_viewmats(*args, _ptr(v_viewmats), _ptr(ws), ws.numel(), _stream(dev))
        else:
            rc = lib.egs_projection_bwd_raw(*args, _stream(dev))
    _lib.check(rc, "egs_projection_bwd_raw")
    out = (*outs, absgrad) if want_absgrad else tuple(outs)
    return _with_camera_grads(out, v_viewmats, v_Ks)


def exclusive_scan(counts: Tensor) -> Tuple[Tensor, Tensor]:
    """int32[n] -> (exclusive prefix int64[n], total int64[1]) — device side, no sync."""
    lib = _lib.load()
    flat = counts.reshape(-1).contiguous()
    n, dev = flat.numel(), flat.device
    out = torch.empty(n, dtype=torch.int64, device=dev)
    total = torch.empty(1, dtype=torch.int64, device=dev)
    ws_bytes = lib.egs_exclusive_scan_workspace_bytes(n)
    ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.egs_exclusive_scan(n, _ptr(flat), _ptr(out), _ptr(total), _ptr(ws), ws.numel(), _stream(dev))
    _lib.check(rc, "egs_exclusive_scan")
    return out, total


def radix_sort_pairs(keys: Tensor, vals: Tensor, end_bit: int) -> Tuple[Tensor, Tensor]:
    """Stable ascending sort of (int64 key, int32 value) pairs on key bits [0, end_bit).
    The inputs are used as one side of the ping-pong and are clobbered."""
    lib = _lib.load()
    n, dev = keys.numel(), keys.device
    if n == 0:
        return keys, vals
    keys_b, vals_b = torch.empty_like(keys), torch.empty_like(vals)
    ws_bytes = lib.egs_radix_sort_workspace_bytes(n, end_bit)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    in_b = ctypes.c_int32(0)
    with torch.cuda.device(dev):
        rc = lib.egs_radix_sort_pairs_u64_u32(n, _ptr(keys), _ptr(vals), _ptr(keys_b), _ptr(vals_b), int(end_bit),
                                              _ptr(ws), ws_bytes, ctypes.byref(in_b), _stream(dev))
    _lib.check(rc, "egs_radix_sort_pairs_u64_u32")
    return (keys_b, vals_b) if in_b.value else (keys, vals)


def isect_tiles(means2d: Tensor, radii: Tensor, depths: Tensor, tile_size: int, tile_width: int, tile_height: int,
                sort: bool = True, tiles_per_gauss: Optional[Tensor] = None,
                n_isects: Optional[int] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """g3+g4 -> tiles_per_gauss[C,N] i32, isect_ids[n] i64, flatten_ids[n] i32 (sorted when sort=True).

    When ``tiles_per_gauss`` is not given it is recomputed with torch from (means2d, radii) the same
    way the projection kernel counts (exact: divisions by the power-of-two tile size)."""
    lib = _lib.load()
    means2d, depths = _f32c(means2d, "means2d"), _f32c(depths, "depths")
    radii = radii.contiguous()
    C, N = radii.shape
    dev = radii.device
    if tiles_per_gauss is None:
        ts = float(tile_size)
        r = radii.to(torch.float32) / ts
        tx, ty = means2d[..., 0] / ts, means2d[..., 1] / ts
        x0 = torch.floor(tx - r).clamp(0, tile_width)
        x1 = torch.ceil(tx + r).clamp(0, tile_width)
        y0 = torch.floor(ty - r).clamp(0, tile_height)
        y1 = torch.ceil(ty + r).clamp(0, tile_height)
        tiles_per_gauss = torch.where(radii > 0, (x1 - x0) * (y1 - y0), torch.zeros_like(x0)).to(torch.int32)
    cum, total = exclusive_scan(tiles_per_gauss)
    if n_isects is None:
        n_isects = int(total.item())  # the one host sync of the forward pass
    ids = torch.empty(n_isects, dtype=torch.int64, device=dev)
    flat = torch.empty(n_isects, dtype=torch.int32, device=dev)
    nbits = tile_n_bits(tile_width, tile_height)
    with torch.cuda.device(dev):
        rc = lib.egs_isect_emit(C, N, _ptr(means2d), _ptr(radii), _ptr(depths), _ptr(cum), int(tile_size),
                                tile_width, tile_height, nbits, n_isects, _ptr(ids), _ptr(flat), _stream(dev))
    _lib.check(rc, "egs_isect_emit")
    if sort and n_isects > 0:
        ids, flat = radix_sort_pairs(ids, flat, 32 + nbits + camera_n_bits(C))
    return tiles_per_gauss, ids, flat


def radix_sort_pairs_u32(keys: Tensor, vals: Tensor, end_bit: int) -> Tuple[Tensor, Tensor]:
    """Same onesweep sort for (int32-as-uint32 key, int32 value) pairs; inputs are clobbered."""
    lib = _lib.load()
    n, dev = keys.numel(), keys.device
    if n == 0 or end_bit == 0:
        return keys, vals
    keys_b, vals_b = torch.empty_like(keys), torch.empty_like(vals)
    ws_bytes = lib.egs_radix_sort_workspace_bytes(n, end_bit)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    in_b = ctypes.c_int32(0)
    with torch.cuda.device(dev):
        rc = lib.egs_radix_sort_pairs_u32_u32(n, _ptr(keys), _ptr(vals), _ptr(keys_b), _ptr(vals_b), int(end_bit),
                                              _ptr(ws), ws_bytes, ctypes.byref(in_b), _stream(dev))
    _lib.check(rc, "egs_radix_sort_pairs_u32_u32")
    return (keys_b, vals_b) if in_b.value else (keys, vals)


# ---- binning without a host round trip --------------------------------------------------------------------------------
# The sizes of the intersection buffers depend on a count that only the device knows.  Instead of waiting for it
# (one blocking read per forward pass, during which nothing new is enqueued), a call sizes its buffers from what the
# previous call of the same shape needed (+ 25 %), enqueues the whole route — every kernel reads the live counts on
# the device — plus the blend forward, and only THEN looks at the counts, which were copied to pinned host memory
# right after the first scan and have long arrived.  If the guess was too small the route is enqueued again with the
# exact size (rare: the count changes slowly from view to view).  The first call of a shape has no guess and waits.
#
# Two counts travel: the BOUND (gsplat's count, the sum of tiles_per_gauss — known after the first kernel of the route)
# and, for the tight lists, the emitted count (known after the whole route).  Buffers are sized from the previous
# call's bound, so "this call's bound fits" settles the question as soon as the first kernel has run; the host then
# never waits for the route itself, and the device never waits for the host to enqueue what follows the blend
# forward (one view per call: 1.37 -> 1.29 ms per view on the 1 M-Gaussian scene, gpurun_out/c1_*).  Only when the
# bound does not fit is the emitted count waited for.
_HINT_LOCK = threading.Lock()
_HINTS: Dict[Tuple[int, int, int, int], Dict[str, int]] = {}
_PINNED: Dict[int, Tuple[Tensor, List[int]]] = {}
_PINNED_SLOTS = 256
_CAPACITY_SLACK = 1.25


def _round_capacity(n: int) -> int:
    """Rounds a guessed capacity up to the next of 8 steps per octave (at most 12.5 % more).  The bound a view leaves
    differs a little from the one before it; sized exactly, every call would ask the caching allocator for buffers of a
    new size, and a training step of a few milliseconds can end up paying for cudaMalloc calls in its steady state."""
    if n <= 1 << 16:
        return 1 << 16
    step = 1 << (n.bit_length() - 4)  # 8 steps between 2^(k-1) and 2^k
    return ((n + step - 1) // step) * step


def _pinned_slot(dev: torch.device) -> Tensor:
    """A 4 x int64 slot of a per-device ring of pinned host memory (allocated once: cudaHostAlloc is slow)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    with _HINT_LOCK:
        ring = _PINNED.get(key)
        if ring is None:
            ring = (torch.empty(_PINNED_SLOTS, 4, dtype=torch.int64).pin_memory(), [0])
            _PINNED[key] = ring
        buf, nxt = ring
        i = nxt[0]
        nxt[0] = (i + 1) % _PINNED_SLOTS
    return buf[i]


def reset_binning_hints() -> None:
    """Forget what previous calls needed (the next call of every shape sizes its buffers exactly, with one wait)."""
    with _HINT_LOCK:
        _HINTS.clear()


def _hint_count(h) -> Optional[int]:
    """The intersection count a hint knows WITHOUT waiting: its own if it has arrived, else the one before it."""
    if h is None:
        return None
    if h["n_isects"] is None and h["late_event"].query():
        h["n_isects"] = int(h["late"][1])
    return h["n_isects"] if h["n_isects"] is not None else h.get("known")


class SortedIsects:
    """Result of ``isect_sorted_async``: buffers sized for ``capacity`` intersections and the pending counts."""

    def __init__(self, key, C, n_tiles, capacity, tile_keys, flat, offsets_store, offsets, depths, stats_dev, early, early_event, exact,
                 tile_order=None, emitted=None, emitted_event=None):
        self.key, self.C, self.n_tiles, self.capacity = key, C, n_tiles, capacity
        self.tile_keys_cap, self.flat_cap, self.offsets_store, self.offsets = tile_keys, flat, offsets_store, offsets
        # launch order of the blend kernels: tiles by list length, longest first (EGS_TILE_ORDER=0: grid order, for A/B runs)
        self.tile_order = tile_order if os.environ.get("EGS_TILE_ORDER", "1") != "0" else None
        self.depths, self.stats_dev = depths, stats_dev
        self._early, self._early_event = early, early_event        # {n_vis, bound}: after the first kernel of the route
        self._emitted, self._emitted_event = emitted, emitted_event  # tight lists: {.., emitted count} after the route
        self.n_vis: Optional[int] = None
        self.n_bound: Optional[int] = None
        self._n_isects: Optional[int] = None
        self._fits: Optional[bool] = None
        self.exact = exact  # the capacity was sized from this call's own count (first call of a shape, or the re-run)

    @property
    def raster_n(self) -> int:
        """What the egs_rasterize_* entries take as n_isects: -capacity = 'read the live length behind the offsets'."""
        return -self.capacity

    @property
    def n_isects(self) -> int:
        """Length of the lists.  For the tight lists this is known only after the whole route: the first read waits."""
        if self._n_isects is None:
            if self._emitted is None:
                self._early_event.synchronize()
                self._n_isects = int(self._early[1])
            else:
                self._emitted_event.synchronize()
                self._n_isects = int(self._emitted[1])
            if self._n_isects >= 2 ** 31 - 1:
                raise RuntimeError(f"{self._n_isects} tile intersections do not fit int32 offsets; render fewer cameras per call")
        return self._n_isects

    def resolve(self) -> bool:
        """Waits for the BOUND on the count (normally long there).  False = the buffers were too small: they hold a
        truncated binning and the caller must run the route again with ``capacity=self.n_isects``."""
        if self._fits is None:
            self._early_event.synchronize()
            self.n_vis, self.n_bound = int(self._early[0]), int(self._early[1])
            # the bound fits: so does whatever the route emits.  Otherwise the emitted count decides (and is waited for).
            self._fits = self.n_bound <= self.capacity or self.n_isects <= self.capacity
        return self._fits

    def note_for_next_call(self) -> None:
        """Leaves the hint for the next call of this shape and queues the late statistic (longest tile list) for it."""
        dev = self.flat_cap.device
        late = _pinned_slot(dev)
        late.copy_(self.stats_dev, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        with _HINT_LOCK:
            prev = _HINTS.get(self.key)
            # n_isects: None = still on its way in `late` (slot 1); `known` = the last count that did arrive
            _HINTS[self.key] = {"n_isects": self._n_isects, "known": _hint_count(prev), "n_bound": self.n_bound,
                                "late": late, "late_event": ev}

    @property
    def flatten_ids(self) -> Tensor:
        return self.flat_cap[:self.n_isects]

    def isect_ids(self) -> Tensor:
        """The 64-bit sorted keys, rebuilt from the 32-bit (camera, tile) keys and the depths (bit-identical)."""
        lib = _lib.load()
        dev = self.flat_cap.device
        n = self.n_isects
        ids = torch.empty(n, dtype=torch.int64, device=dev)
        if n == 0:
            return ids
        nbits = tile_n_bits_from_count(self.n_tiles)
        with torch.cuda.device(dev):
            rc = lib.egs_isect_finalize(n, _ptr(self.tile_keys_cap), _ptr(self.flat_cap), _ptr(self.depths), self.C, self.n_tiles,
                                        nbits, _ptr(ids), None, _stream(dev))
        _lib.check(rc, "egs_isect_finalize")
        return ids


class ResolvedIsects:
    """A binning whose sizes are already known, behind the interface of ``SortedIsects`` (synchronous producers:
    the classic route, test stand-ins)."""

    exact = True
    raster_n = None  # the rasterize operators then take len(flatten_ids)
    tile_order = None  # grid order

    def __init__(self, isect_ids, flatten_ids: Tensor, offsets: Tensor):
        self._ids, self.flat_cap, self.offsets = isect_ids, flatten_ids, offsets
        self.n_isects = flatten_ids.numel()
        self.capacity = max(self.n_isects, 1)

    def resolve(self) -> bool:
        return True

    def note_for_next_call(self) -> None:
        pass

    @property
    def flatten_ids(self) -> Tensor:
        return self.flat_cap

    def isect_ids(self) -> Tensor:
        return self._ids() if callable(self._ids) else self._ids


def tile_n_bits_from_count(n_tiles: int) -> int:
    return int(math.floor(math.log2(n_tiles))) + 1


def binning_hint(C: int, tile_width: int, tile_height: int, device, tight: bool = True) -> Optional[Dict[str, int]]:
    """What the previous call of this shape on this device needed: {'n_isects', 'max_tile_len' (if it has arrived)}."""
    dev = torch.device(device)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), C, tile_width, tile_height, tight)
    with _HINT_LOCK:
        h = _HINTS.get(key)
        if h is None:
            return None
        n = _hint_count(h)  # never waits: a count that has not arrived yet is simply not used
        out = {"n_bound": h["n_bound"]}
        if n is not None:
            out["n_isects"] = n
            if h["late_event"].query():
                out["max_tile_len"] = int(h["late"][2])
        return out


def isect_sorted_async(means2d: Tensor, radii: Tensor, depths: Tensor, tiles_per_gauss: Tensor, tile_size: int,
                       tile_width: int, tile_height: int, capacity: Optional[int] = None,
                       tight_rects: Optional[Tensor] = None) -> SortedIsects:
    """g3+g4+g5, enqueued without waiting for the intersection count (see the block comment above).  ``capacity``:
    intersections to provide room for; None = from the previous call of this shape, or — first call — wait and size
    from the classic count (an upper bound).

    ``tight_rects`` (that output of ``projection_fwd``): build the TIGHT lists the blend kernels need instead of
    gsplat's — a Gaussian is listed only in the tiles of its classic rectangle that hold a pixel it can reach with
    alpha >= 1/255 (include/egs_raster.h, egs_isect_sorted).  Same pixels and gradients, a third fewer entries to
    sort, stage and cull.  Without it the lists are bit-identical to gsplat's (``isect_tiles`` + offset encode)."""
    lib = _lib.load()
    means2d, depths = _f32c(means2d, "means2d"), _f32c(depths, "depths")
    radii, tiles_per_gauss = radii.contiguous(), tiles_per_gauss.contiguous()
    C, N = radii.shape
    dev = radii.device
    n = C * N
    n_tiles = tile_width * tile_height
    tight = tight_rects is not None
    if tight:
        if tight_rects.shape != (C, N, 2) or tight_rects.dtype != torch.int32:
            raise ValueError(f"tight_rects must be the int32 [C, N, 2] output of projection_fwd (got {tuple(tight_rects.shape)})")
        tight_rects = tight_rects.contiguous()
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), C, tile_width, tile_height, tight)
    ws_scan = max(lib.egs_isect_scan_workspace_bytes(max(n, 1)), 16)
    scan_ws = torch.empty(ws_scan, dtype=torch.uint8, device=dev)
    stats = torch.empty(4, dtype=torch.int64, device=dev)
    keys1 = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    vals1 = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.egs_isect_visible_keys(C, N, _ptr(tiles_per_gauss), _ptr(depths), _ptr(keys1), _ptr(vals1), _ptr(stats),
                                        _ptr(scan_ws), ws_scan, _stream(dev))
    _lib.check(rc, "egs_isect_visible_keys")
    early = _pinned_slot(dev)
    early.copy_(stats, non_blocking=True)
    early_event = torch.cuda.Event()
    early_event.record(torch.cuda.current_stream(dev))
    exact = False
    if capacity is None:
        with _HINT_LOCK:
            h = _HINTS.get(key)
        if h is not None and h.get("n_bound") is not None:
            capacity = _round_capacity(int(h["n_bound"] * _CAPACITY_SLACK) + 65536)
        else:  # no guess: the one blocking read, as in every call before round 2 (the classic count bounds the tight one)
            early_event.synchronize()
            capacity, exact = int(early[1]), True
    else:
        exact = True
    capacity = max(1, min(int(capacity), 2 ** 31 - 2))
    tile_keys = torch.empty(capacity, dtype=torch.int32, device=dev)
    flat = torch.empty(capacity, dtype=torch.int32, device=dev)
    offsets_store = torch.empty(C * n_tiles + 1, dtype=torch.int32, device=dev)
    offsets = offsets_store[:C * n_tiles].view(C, tile_height, tile_width)
    tile_order = torch.empty(max(C * n_tiles, 1), dtype=torch.int32, device=dev)
    ws_bytes = lib.egs_isect_sorted_workspace_bytes(C, N, n_tiles, capacity)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.egs_isect_sorted(C, N, _ptr(tight_rects) if tight else None, _ptr(means2d), _ptr(radii),
                                  _ptr(keys1), _ptr(vals1), _ptr(stats), int(tile_size), tile_width, tile_height, capacity,
                                  _ptr(ws), ws.numel(), _ptr(tile_keys), _ptr(flat), _ptr(offsets_store), _ptr(tile_order),
                                  _stream(dev))
    _lib.check(rc, "egs_isect_sorted")
    emitted = emitted_event = None
    if tight:
        # the length of the lists is the emitted count (stats[1], rewritten by the route): it travels the same way,
        # but is waited for only if the bound did not fit (or when somebody asks for the exact length)
        emitted = _pinned_slot(dev)
        emitted.copy_(stats, non_blocking=True)
        emitted_event = torch.cuda.Event()
        emitted_event.record(torch.cuda.current_stream(dev))
    return SortedIsects(key, C, n_tiles, capacity, tile_keys, flat, offsets_store, offsets, depths, stats, early, early_event, exact,
                        tile_order=tile_order, emitted=emitted, emitted_event=emitted_event)


def isect_sorted(means2d: Tensor, radii: Tensor, depths: Tensor, tiles_per_gauss: Tensor, tile_size: int,
                 tile_width: int, tile_height: int, materialize_ids: bool = True):
    """g3+g4+g5 fast path -> (isect_ids[n] i64 sorted, flatten_ids[n] i32, isect_offsets[C,th,tw] i32).

    Bit-identical to ``isect_tiles(sort=True)`` + ``isect_offset_encode`` (a stable sort on cam|tile|depth
    equals a stable depth sort of the visible entries followed by a stable sort on the (camera, tile) index), but the
    n_isects-sized passes move 8-byte pairs through 2-3 radix passes instead of 12-byte pairs through 6.
    With ``materialize_ids=False`` the first element is a zero-argument callable that builds isect_ids on demand.
    This is the synchronous form (exact-length tensors on return); ``rasterization()`` uses ``isect_sorted_async``."""
    b = isect_sorted_async(means2d, radii, depths, tiles_per_gauss, tile_size, tile_width, tile_height)
    if not b.resolve():
        b = isect_sorted_async(means2d, radii, depths, tiles_per_gauss, tile_size, tile_width, tile_height, capacity=b.n_isects)
        b.resolve()
    assert b.exact or b.n_isects <= b.capacity
    b.note_for_next_call()
    return (b.isect_ids() if materialize_ids else b.isect_ids), b.flatten_ids, b.offsets


def isect_offset_encode(isect_ids: Tensor, C: int, tile_width: int, tile_height: int) -> Tensor:
    """g5 -> offsets[C, tile_height, tile_width] int32."""
    lib = _lib.load()
    dev = isect_ids.device
    offs = torch.empty(C, tile_height, tile_width, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.egs_isect_offset_encode(isect_ids.numel(), _ptr(isect_ids), C, tile_width * tile_height,
                                         tile_n_bits(tile_width, tile_height), _ptr(offs), _stream(dev))
    _lib.check(rc, "egs_isect_offset_encode")
    return offs


def pack_splats(means2d: Tensor, conics: Tensor, colors: Tensor, opacities: Tensor, depths: Optional[Tensor] = None) -> Tensor:
    """Builds the packed 48-byte splat records [C,N,12] from separate tensors (stage-level tests)."""
    C, N = means2d.shape[:2]
    z = torch.zeros(C, N, 1, dtype=torch.float32, device=means2d.device)
    d = z if depths is None else depths[..., None]
    cut = torch.full_like(z, float("inf"))  # sigma_cut = +inf: no warp-level culling, every pair is evaluated
    return torch.cat([means2d, conics, opacities[..., None], colors, d, z, cut], -1).contiguous()


def rasterize_fwd(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, backgrounds: Optional[Tensor],
                  width: int, height: int, count_pairs: bool = False, n_isects: Optional[int] = None,
                  tile_order: Optional[Tensor] = None):
    """g6 -> render_colors[C,H,W,3], render_alphas[C,H,W,1], last_ids[C,H,W] (, (P_eval, P_acc) tensor).
    n_isects: None = len(flatten_ids); negative = -capacity, the live length sits behind the offsets
    (``SortedIsects.raster_n``; isect_offsets must then be the view ``SortedIsects.offsets``).
    tile_order: int32 permutation of the C * tiles flat tile indices = the order thread blocks take them in
    (``SortedIsects.tile_order``: longest lists first); None = grid order.  Results do not depend on it."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    colors = torch.empty(C, height, width, 3, dtype=torch.float32, device=dev)
    alphas = torch.empty(C, height, width, 1, dtype=torch.float32, device=dev)
    last = torch.empty(C, height, width, dtype=torch.int32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    args = [C, N, flatten_ids.numel() if n_isects is None else int(n_isects), _ptr(splats), _ptr(isect_offsets),
            _ptr(flatten_ids), _ptr(bg), int(width), int(height), tw, th, _ptr(colors), _ptr(alphas), _ptr(last)]
    with torch.cuda.device(dev):
        if count_pairs:
            counters = torch.zeros(2, dtype=torch.int64, device=dev)
            rc = lib.egs_rasterize_fwd_count(*args, _ptr(counters), _stream(dev))
        else:
            rc = lib.egs_rasterize_fwd(*args, _ptr(tile_order), _stream(dev))
    _lib.check(rc, "egs_rasterize_fwd")
    return (colors, alphas, last, counters) if count_pairs else (colors, alphas, last)


def backward_segment() -> Optional[int]:
    """EGS_BWD_SEGMENT=<0 or a multiple of 64>: experiment override of the automatic policy below (0 = never segment,
    K = replay every list longer than K in K-entry segments).  Unset (the default) = automatic."""
    v = os.environ.get("EGS_BWD_SEGMENT")
    if v is None or v == "":
        return None
    v = int(v)
    if v < 0 or v % 64 != 0:
        raise ValueError(f"EGS_BWD_SEGMENT={v}: must be 0 or a multiple of 64")
    return v


SEGMENT_ENTRIES = 512       # list entries per replay segment
SEGMENT_MIN_ENTRIES = 1024   # never segment lists shorter than this
SEGMENT_MIN_RATIO = 3.0      # ... or shorter than this many times the average list
SEGMENT_TRIGGER_RATIO = 6.0  # and only in scenes whose longest list is at least this many times the average


def segment_policy(hint: Optional[Dict[str, int]], n_tiles_total: int) -> Tuple[int, int]:
    """-> (segment, seg_min_len) for a forward pass that will be differentiated; (0, 0) = no segmented replay.

    A tile list that is several times longer than the average makes the backward pass wait for ONE warp per tile half
    walking it (object scenes rendered one view per call: a few hundred tiles hold 5-6 k entries, the average is ~500).
    Such lists — and only those — are replayed in 512-entry segments, one warp each (csrc/blend.cu).  Whether a scene
    has them is taken from the previous call of the same shape (``binning_hint``: intersection count and longest
    list, read back without waiting): measured on the one-view-per-call pattern, object scene 1.22 -> 1.10 ms per
    view; a scene without outliers (the 1 M-Gaussian benchmark: longest list 2.2 x the average) is left alone, where
    segmenting everything longer than 512 entries cost 10 % (gpurun_out/r2c_knobs.log)."""
    forced = backward_segment()
    if forced is not None:
        return (forced, forced + 1) if forced > 0 else (0, 0)
    if hint is None or "max_tile_len" not in hint:
        return 0, 0
    mean = hint["n_isects"] / max(n_tiles_total, 1)
    min_len = max(SEGMENT_MIN_ENTRIES, int(SEGMENT_MIN_RATIO * mean))
    if hint["max_tile_len"] >= max(min_len, SEGMENT_TRIGGER_RATIO * mean):
        return SEGMENT_ENTRIES, min_len
    return 0, 0


def rasterize_fwd_checkpointed(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor,
                               backgrounds: Optional[Tensor], width: int, height: int, segment: int,
                               seg_min_len: int = 0, n_isects: Optional[int] = None, tile_order: Optional[Tensor] = None):
    """g6 for a forward that will be differentiated: as rasterize_fwd, plus the per-pixel state after every
    `segment` entries of a tile's list -> render_colors, render_alphas, last_ids, checkpoints."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    n_isects = flatten_ids.numel() if n_isects is None else int(n_isects)
    colors = torch.empty(C, height, width, 3, dtype=torch.float32, device=dev)
    alphas = torch.empty(C, height, width, 1, dtype=torch.float32, device=dev)
    last = torch.empty(C, height, width, dtype=torch.int32, device=dev)
    ckpt = torch.empty(max(lib.egs_rasterize_checkpoint_bytes(n_isects, segment) // 4, 4), dtype=torch.float32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    with torch.cuda.device(dev):
        rc = lib.egs_rasterize_fwd_checkpointed(C, N, n_isects, _ptr(splats), _ptr(isect_offsets), _ptr(flatten_ids),
                                                _ptr(bg), int(width), int(height), tw, th, _ptr(colors), _ptr(alphas),
                                                _ptr(last), _ptr(ckpt), int(segment), int(seg_min_len), _ptr(tile_order),
                                                _stream(dev))
    _lib.check(rc, "egs_rasterize_fwd_checkpointed")
    return colors, alphas, last, ckpt


def rasterize_bwd_segmented(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, backgrounds: Optional[Tensor],
                            width: int, height: int, render_colors: Tensor, render_alphas: Tensor, last_ids: Tensor,
                            v_render_colors: Tensor, v_render_alphas: Tensor, checkpoints: Tensor, segment: int,
                            seg_min_len: int = 0, n_isects: Optional[int] = None, tile_order: Optional[Tensor] = None) -> Tensor:
    """g7 with one warp per list segment (see include/egs_raster.h) -> v_splats[C,N,12]."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    v_splats = torch.zeros(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    v_c, v_a = _f32c(v_render_colors, "v_render_colors"), _f32c(v_render_alphas, "v_render_alphas")
    with torch.cuda.device(dev):
        rc = lib.egs_rasterize_bwd_segmented(C, N, flatten_ids.numel() if n_isects is None else int(n_isects), _ptr(splats),
                                             _ptr(isect_offsets), _ptr(flatten_ids), _ptr(bg), int(width), int(height), tw, th,
                                             _ptr(render_colors), _ptr(render_alphas), _ptr(last_ids), _ptr(v_c), _ptr(v_a),
                                             _ptr(checkpoints), int(segment), int(seg_min_len), _ptr(v_splats), _ptr(tile_order),
                                             _stream(dev))
    _lib.check(rc, "egs_rasterize_bwd_segmented")
    return v_splats


def rasterize_bwd(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, backgrounds: Optional[Tensor],
                  width: int, height: int, render_alphas: Tensor, last_ids: Tensor, v_render_colors: Tensor,
                  v_render_alphas: Tensor, n_isects: Optional[int] = None, tile_order: Optional[Tensor] = None) -> Tensor:
    """g7 -> packed gradient records v_splats[C,N,12] (layout in include/egs_raster.h)."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    v_splats = torch.zeros(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    v_c, v_a = _f32c(v_render_colors, "v_render_colors"), _f32c(v_render_alphas, "v_render_alphas")
    with torch.cuda.device(dev):
        rc = lib.egs_rasterize_bwd(C, N, flatten_ids.numel() if n_isects is None else int(n_isects), _ptr(splats),
                                   _ptr(isect_offsets), _ptr(flatten_ids),
                                   _ptr(bg), int(width), int(height), tw, th, _ptr(render_alphas), _ptr(last_ids),
                                   _ptr(v_c), _ptr(v_a), _ptr(v_splats), _ptr(tile_order), _stream(dev))
    _lib.check(rc, "egs_rasterize_bwd")
    return v_splats


def rasterize_fwd_depth(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, backgrounds: Optional[Tensor],
                        width: int, height: int, n_isects: Optional[int] = None, tile_order: Optional[Tensor] = None):
    """g6 with the depth (record slot 9) as a fourth channel -> render_colors[C,H,W,4] = (r, g, b, accumulated depth),
    render_alphas[C,H,W,1], last_ids[C,H,W].  backgrounds [C,3] apply to r, g, b; the depth's background is 0.
    Arguments as rasterize_fwd."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    colors = torch.empty(C, height, width, 4, dtype=torch.float32, device=dev)
    alphas = torch.empty(C, height, width, 1, dtype=torch.float32, device=dev)
    last = torch.empty(C, height, width, dtype=torch.int32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    with torch.cuda.device(dev):
        rc = lib.egs_rasterize_fwd_depth(C, N, flatten_ids.numel() if n_isects is None else int(n_isects), _ptr(splats),
                                         _ptr(isect_offsets), _ptr(flatten_ids), _ptr(bg), int(width), int(height), tw, th,
                                         _ptr(colors), _ptr(alphas), _ptr(last), _ptr(tile_order), _stream(dev))
    _lib.check(rc, "egs_rasterize_fwd_depth")
    return colors, alphas, last


def rasterize_bwd_depth(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, backgrounds: Optional[Tensor],
                        width: int, height: int, render_alphas: Tensor, last_ids: Tensor, v_render_colors: Tensor,
                        v_render_alphas: Tensor, n_isects: Optional[int] = None,
                        tile_order: Optional[Tensor] = None) -> Tensor:
    """g7 of rasterize_fwd_depth: v_render_colors [C,H,W,4] -> v_splats[C,N,12] with v_depth in slot 11."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    v_splats = torch.zeros(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    v_c, v_a = _f32c(v_render_colors, "v_render_colors"), _f32c(v_render_alphas, "v_render_alphas")
    with torch.cuda.device(dev):
        rc = lib.egs_rasterize_bwd_depth(C, N, flatten_ids.numel() if n_isects is None else int(n_isects), _ptr(splats),
                                         _ptr(isect_offsets), _ptr(flatten_ids), _ptr(bg), int(width), int(height), tw, th,
                                         _ptr(render_alphas), _ptr(last_ids), _ptr(v_c), _ptr(v_a), _ptr(v_splats),
                                         _ptr(tile_order), _stream(dev))
    _lib.check(rc, "egs_rasterize_bwd_depth")
    return v_splats


FEATURE_CHUNK = 32  # colour channels per blend launch: gsplat's default channel_chunk
FEATURE_WIDTHS = (1, 2, 4, 8, 16, 32)  # chunk widths the feature kernels are instantiated for


def feature_chunks(D: int) -> List[Tuple[int, int]]:
    """(c0, CH) of the blend launches for D colour channels: 32-channel chunks, the last one narrowed to the smallest
    instantiated width that holds the remaining channels (the rows are padded with zero channels up to it)."""
    if D < 1:
        raise ValueError(f"colours need at least one channel, got D={D}")
    return [(c0, next(w for w in FEATURE_WIDTHS if w >= min(FEATURE_CHUNK, D - c0))) for c0 in range(0, D, FEATURE_CHUNK)]


def _feature_rows(features: Tensor, chunks: List[Tuple[int, int]]) -> Tensor:
    """features [N,D] / [C,N,D] -> dense fp32 rows [rows, stride] from which every chunk reads its CH channels:
    stride = the padded width, rounded up to the row alignment the widest chunk needs (4 floats from CH = 4 on).
    The tensor itself (a view) when it already is such an array, a zero-padded copy otherwise."""
    D = features.shape[-1]
    c0, ch = chunks[-1]
    align = min(4, max(w for _, w in chunks))
    stride = -(-(c0 + ch) // align) * align
    rows = _f32c(features, "colors").reshape(-1, D)
    if stride == D:
        return rows
    out = torch.zeros(rows.shape[0], stride, dtype=torch.float32, device=rows.device)
    out[:, :D] = rows
    return out


def rasterize_fwd_features(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, features: Tensor,
                           backgrounds: Optional[Tensor], width: int, height: int, n_isects: Optional[int] = None,
                           tile_order: Optional[Tensor] = None):
    """g6 for colours of any width: features [N,D] (shared by the cameras) or [C,N,D], backgrounds [C,D] ->
    render_colors[C,H,W,D], render_alphas[C,H,W,1], last_ids[C,H,W].  One launch per 32-channel chunk on the same
    lists; the first chunk writes the alphas and last_ids (every chunk would write the same)."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    D = features.shape[-1]
    chunks = feature_chunks(D)
    rows = _feature_rows(features, chunks)
    colors = torch.empty(C, height, width, D, dtype=torch.float32, device=dev)
    alphas = torch.empty(C, height, width, 1, dtype=torch.float32, device=dev)
    last = torch.empty(C, height, width, dtype=torch.int32, device=dev)
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    n = flatten_ids.numel() if n_isects is None else int(n_isects)
    with torch.cuda.device(dev):
        for i, (c0, ch) in enumerate(chunks):
            rc = lib.egs_rasterize_fwd_features(C, N, n, _ptr(splats), _ptr(isect_offsets), _ptr(flatten_ids), _ptr(rows),
                                                rows.shape[1], int(features.dim() == 2), D, c0, ch, _ptr(bg), int(width),
                                                int(height), tw, th, _ptr(colors), _ptr(alphas) if i == 0 else None,
                                                _ptr(last) if i == 0 else None, _ptr(tile_order), _stream(dev))
            _lib.check(rc, "egs_rasterize_fwd_features")
    return colors, alphas, last


def rasterize_bwd_features(splats: Tensor, isect_offsets: Tensor, flatten_ids: Tensor, features: Tensor,
                           backgrounds: Optional[Tensor], width: int, height: int, render_alphas: Tensor,
                           last_ids: Tensor, v_render_colors: Tensor, v_render_alphas: Tensor,
                           n_isects: Optional[int] = None, tile_order: Optional[Tensor] = None,
                           want_features_grad: bool = True) -> Tuple[Tensor, Optional[Tensor]]:
    """g7 for colours of any width -> (v_splats[C,N,12] with the geometry slots filled and v_r, v_g, v_b = 0,
    v_features in the shape of features, or None without want_features_grad).  One launch per chunk; the geometry
    gradients, |v_x| and |v_y| included, sum over the chunks."""
    lib = _lib.load()
    dev = splats.device
    C, N = splats.shape[:2]
    th, tw = isect_offsets.shape[1:]
    D = features.shape[-1]
    chunks = feature_chunks(D)
    rows = _feature_rows(features, chunks)
    v_splats = torch.zeros(C, N, SPLAT_FLOATS, dtype=torch.float32, device=dev)
    v_rows = torch.zeros_like(rows) if want_features_grad else None
    bg = None if backgrounds is None else _f32c(backgrounds, "backgrounds")
    v_c, v_a = _f32c(v_render_colors, "v_render_colors"), _f32c(v_render_alphas, "v_render_alphas")
    n = flatten_ids.numel() if n_isects is None else int(n_isects)
    with torch.cuda.device(dev):
        for i, (c0, ch) in enumerate(chunks):
            rc = lib.egs_rasterize_bwd_features(C, N, n, _ptr(splats), _ptr(isect_offsets), _ptr(flatten_ids), _ptr(rows),
                                                rows.shape[1], int(features.dim() == 2), D, c0, ch, _ptr(bg), int(width),
                                                int(height), tw, th, _ptr(render_alphas), _ptr(last_ids), _ptr(v_c),
                                                _ptr(v_a) if i == 0 else None, _ptr(v_splats), _ptr(v_rows),
                                                _ptr(tile_order), _stream(dev))
            _lib.check(rc, "egs_rasterize_bwd_features")
    v_features = None if v_rows is None else v_rows[:, :D].reshape(features.shape)
    return v_splats, v_features


def densify_stats_update(max_radii: Tensor, grad_norm_accum: Tensor, collecting_counts: Tensor, radii: Tensor,
                         absgrad: Tensor, width: int, height: int) -> None:
    """§8f-1: in-place, sync-free equivalent of GaussianModel.update_statistics
    (/root/reference/model/gaussian.py:188-197) for all C views of a call."""
    lib = _lib.load()
    dev = radii.device
    C, N = radii.shape
    absgrad = _f32c(absgrad, "absgrad")
    for t, nm in ((max_radii, "max_radii"), (grad_norm_accum, "grad_norm_accum"), (collecting_counts, "collecting_counts")):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == N):
            raise ValueError(f"{nm} must be a contiguous float32 CUDA tensor of N={N} elements")
    with torch.cuda.device(dev):
        rc = lib.egs_densify_stats_update(C, N, _ptr(radii.contiguous()), _ptr(absgrad), float(max(height, width)),
                                          _ptr(max_radii), _ptr(grad_norm_accum), _ptr(collecting_counts), _stream(dev))
    _lib.check(rc, "egs_densify_stats_update")
