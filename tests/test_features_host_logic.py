"""CPU tests of the host logic of colours with any number of channels: routing in rendering.py (D == 3 keeps the RGB
stage calls, other D go to the feature stages), output / meta / gradient shapes, backgrounds validation, the chunking and
padding of stages.rasterize_*_features (with a stand-in library that records the C calls), and the C entries' argument
checks, which run before any launch and need no GPU."""
import contextlib
import ctypes

import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rendering, stages
from easy_gaussian_splatting_b200.rendering import _check_inputs

SPLAT = stages.SPLAT_FLOATS
W, H = 32, 16


class RecordingStages:
    """Shape-faithful stand-ins that record their calls and return constants."""

    def __init__(self):
        self.calls = []
        self.feature_kwargs = []

    def projection_fwd(self, means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d=0.3,
                       near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16, antialiased=False):
        self.calls.append("projection_fwd")
        self.proj_colors = colors
        C, N = viewmats.shape[0], means.shape[0]
        radii = torch.full((C, N), 4, dtype=torch.int32)
        radii[:, ::3] = 0  # some culled entries, so that packed=True has something to drop
        out = {
            "radii": radii,
            "means2d": means.detach()[None, :, :2].expand(C, N, 2).contiguous(),
            "depths": torch.ones(C, N),
            "conics": torch.ones(C, N, 3),
            "colors": torch.zeros(C, N, 3),
            "tiles_per_gauss": (radii > 0).int(),
            "tight_rects": torch.zeros(C, N, 2, dtype=torch.int32),
            "splats": torch.zeros(C, N, SPLAT),
        }
        if antialiased:
            out["compensations"] = torch.full((C, N), 0.5)
        return out

    def isect_sorted_async(self, means2d, radii, depths, tiles_per_gauss, tile_size, tw, th, capacity=None, tight_rects=None):
        self.calls.append("isect_sorted")
        C = radii.shape[0]
        flat = torch.arange(radii.numel(), dtype=torch.int32)
        return stages.ResolvedIsects(lambda: torch.arange(flat.numel(), dtype=torch.int64), flat,
                                     torch.zeros(C, th, tw, dtype=torch.int32))

    def rasterize_fwd(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, count_pairs=False, n_isects=None,
                      tile_order=None):
        self.calls.append("rasterize_fwd")
        C = splats.shape[0]
        return (torch.full((C, height, width, 3), 0.25), torch.full((C, height, width, 1), 0.5),
                torch.zeros(C, height, width, dtype=torch.int32))

    def rasterize_bwd(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_alphas, last_ids,
                      v_render_colors, v_render_alphas, n_isects=None, tile_order=None):
        self.calls.append("rasterize_bwd")
        return torch.ones_like(splats)

    def rasterize_fwd_features(self, splats, isect_offsets, flatten_ids, features, backgrounds, width, height,
                               n_isects=None, tile_order=None):
        self.calls.append("rasterize_fwd_features")
        C, D = splats.shape[0], features.shape[-1]
        self.fwd_features = features
        return (torch.full((C, height, width, D), 0.25), torch.full((C, height, width, 1), 0.5),
                torch.zeros(C, height, width, dtype=torch.int32))

    def rasterize_bwd_features(self, splats, isect_offsets, flatten_ids, features, backgrounds, width, height,
                               render_alphas, last_ids, v_render_colors, v_render_alphas, n_isects=None, tile_order=None,
                               want_features_grad=True):
        self.calls.append("rasterize_bwd_features")
        self.feature_kwargs.append(dict(want_features_grad=want_features_grad, v_shape=tuple(v_render_colors.shape)))
        return torch.ones_like(splats), (torch.full_like(features, 7.0) if want_features_grad else None)

    def projection_bwd(self, means, quats, scales, colors, viewmats, Ks, width, height, sh_degree, eps2d, radii,
                       colors_rgb, v_splats, v_means2d_extra=None, **kw):
        self.calls.append("projection_bwd")
        self.bwd_colors = colors
        C, N = radii.shape
        outs = tuple(torch.full_like(t, float(i + 1)) for i, t in enumerate((means, quats, scales, means[:, 0], colors)))
        if kw.get("want_absgrad"):
            outs += (torch.full((C, N, 2), 0.125),)
        if kw.get("want_viewmats_grad"):
            outs += (torch.ones(C, 4, 4),)
        return outs


@pytest.fixture()
def rec(monkeypatch):
    f = RecordingStages()
    for name in ("projection_fwd", "isect_sorted_async", "rasterize_fwd", "rasterize_bwd", "rasterize_fwd_features",
                 "rasterize_bwd_features", "projection_bwd"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    monkeypatch.delenv("EGS_BWD_SEGMENT", raising=False)
    return f


def _params(N=10, C=2, D=5, per_camera=False):
    g = torch.Generator().manual_seed(0)
    cols = torch.rand(C, N, D, generator=g) if per_camera else torch.rand(N, D, generator=g)
    p = [torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
         torch.rand(N, generator=g), cols]
    return [t.requires_grad_(True) for t in p], torch.eye(4)[None].repeat(C, 1, 1), torch.eye(3)[None].repeat(C, 1, 1)


FEATURE_CALLS = ["projection_fwd", "isect_sorted", "rasterize_fwd_features", "rasterize_bwd_features", "projection_bwd"]


def test_three_channels_keep_the_rgb_stage_calls(rec):
    p, vm, K = _params(D=3)
    rc, ra, meta = rendering.rasterization(*p, vm, K, W, H, packed=False, absgrad=True, backgrounds=torch.zeros(2, 3))
    rc.sum().backward()
    assert rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd", "rasterize_bwd", "projection_bwd"]
    assert rec.proj_colors is p[4] or torch.equal(rec.proj_colors, p[4])
    assert rc.shape == (2, H, W, 3)


@pytest.mark.parametrize("D", [1, 5, 40])
@pytest.mark.parametrize("per_camera", [False, True])
@pytest.mark.parametrize("packed", [False, True])
def test_feature_routing_and_shapes(rec, D, per_camera, packed):
    C, N = 2, 10
    p, vm, K = _params(N=N, C=C, D=D, per_camera=per_camera)
    bg = torch.rand(C, D).requires_grad_(True)
    rc, ra, meta = rendering.rasterization(*p, vm, K, W, H, packed=packed, absgrad=True, backgrounds=bg)
    assert rc.shape == (C, H, W, D) and ra.shape == (C, H, W, 1)
    assert rec.fwd_features is p[4] or torch.equal(rec.fwd_features, p[4])
    # the projection sees zero RGB colours
    assert rec.proj_colors.shape == (N, 3) and not rec.proj_colors.any()
    nnz = int((meta["radii"] > 0).sum()) if packed else None
    if packed:
        assert meta["colors"].shape == (nnz, D) and meta["means2d"].shape == (nnz, 2)
        expect = p[4].detach()[None].expand(C, N, D) if not per_camera else p[4].detach()
        vis = torch.ones(C, N, dtype=torch.bool)
        vis[:, ::3] = False
        assert torch.equal(meta["colors"], expect[vis])
    else:
        assert meta["colors"].shape == (C, N, D)
        assert torch.equal(meta["colors"], p[4].detach().expand(C, N, D))
    assert meta["conics"].shape[-1] == 3 and meta["radii"].shape == ((C, N) if not packed else (nnz,))
    (rc.sum() + ra.sum()).backward()
    assert rec.calls == FEATURE_CALLS
    assert rec.feature_kwargs == [dict(want_features_grad=True, v_shape=(C, H, W, D))]
    assert not rec.bwd_colors.any() and rec.bwd_colors.shape == (N, 3)
    assert p[4].grad.shape == p[4].shape and torch.all(p[4].grad == 7.0)  # the feature gradient, not the projection's
    assert [t.grad.flatten()[0].item() for t in p[:4]] == [1.0, 2.0, 3.0, 4.0]
    assert bg.grad.shape == (C, D)
    torch.testing.assert_close(bg.grad, torch.full((C, D), 0.5 * H * W))  # sum over pixels of (1 - alpha) * 1
    assert meta["means2d"].absgrad.shape == meta["means2d"].shape


def test_features_without_colour_gradient(rec):
    p, vm, K = _params(D=4)
    p[4].requires_grad_(False)
    rc, _, _ = rendering.rasterization(*p, vm, K, W, H, packed=False)
    rc.sum().backward()
    assert rec.feature_kwargs[-1]["want_features_grad"] is False
    assert p[4].grad is None and p[0].grad is not None


def test_only_alphas_used_still_gives_feature_shaped_cotangent(rec):
    p, vm, K = _params(D=6)
    _, ra, _ = rendering.rasterization(*p, vm, K, W, H, packed=False)
    ra.sum().backward()
    assert rec.feature_kwargs[-1]["v_shape"] == (2, H, W, 6)


def test_no_grad_feature_call(rec):
    p, vm, K = _params(D=8)
    with torch.no_grad():
        rc, ra, meta = rendering.rasterization(*p, vm, K, W, H, packed=False)
    assert rc.grad_fn is None and rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd_features"]
    assert rc.shape == (2, H, W, 8)


def test_backgrounds_and_colour_validation():
    N, C = 5, 2
    f = lambda *s: torch.zeros(*s)
    base = dict(means=f(N, 3), quats=f(N, 4), scales=f(N, 3), opacities=f(N), viewmats=f(C, 4, 4), Ks=f(C, 3, 3),
                sh_degree=None)
    for cols, bg in ((f(N, 7), f(C, 7)), (f(C, N, 7), f(C, 7)), (f(N, 1), f(C, 1)), (f(N, 3), f(C, 3)), (f(N, 40), None)):
        with pytest.raises(RuntimeError, match="CUDA-only"):  # shapes accepted; the CPU tensors are refused next
            _check_inputs(**base, colors=cols, backgrounds=bg)
    for cols, bg in ((f(N, 7), f(C, 3)), (f(N, 7), f(C, 8)), (f(N, 1), f(C, 3)), (f(N, 3), f(C, 4)), (f(N, 7), f(7))):
        with pytest.raises(ValueError, match="backgrounds"):
            _check_inputs(**base, colors=cols, backgrounds=bg)
    for cols in (f(N, 0), f(C, N, 0), f(N + 1, 4), f(C + 1, N, 4), f(N)):
        with pytest.raises(ValueError, match="colors"):
            _check_inputs(**base, colors=cols, backgrounds=None)
    # SH coefficients stay [N,K,3]
    with pytest.raises(ValueError):
        _check_inputs(**{**base, "sh_degree": 0}, colors=f(N, 1, 5), backgrounds=None)


def test_zero_channels_raise_value_error():
    from easy_gaussian_splatting_b200 import rasterization
    N, C = 5, 1
    with pytest.raises(ValueError):
        rasterization(torch.zeros(N, 3), torch.zeros(N, 4), torch.zeros(N, 3), torch.zeros(N), torch.zeros(N, 0),
                      torch.eye(4)[None], torch.eye(3)[None], 16, 16, packed=False)
    with pytest.raises(ValueError):
        stages.feature_chunks(0)


@pytest.mark.parametrize("D,chunks", [(1, [(0, 1)]), (2, [(0, 2)]), (3, [(0, 4)]), (5, [(0, 8)]), (16, [(0, 16)]),
                                      (17, [(0, 32)]), (32, [(0, 32)]), (33, [(0, 32), (32, 1)]),
                                      (40, [(0, 32), (32, 8)]), (64, [(0, 32), (32, 32)]),
                                      (70, [(0, 32), (32, 32), (64, 8)])])
def test_feature_chunks(D, chunks):
    assert stages.feature_chunks(D) == chunks


class FakeLib:
    """Records the feature entries' arguments instead of launching."""

    def __init__(self):
        self.fwd, self.bwd = [], []

    def egs_rasterize_fwd_features(self, *a):
        self.fwd.append(a)
        return 0

    def egs_rasterize_bwd_features(self, *a):
        self.bwd.append(a)
        return 0


@pytest.fixture()
def fake_lib(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(stages, "_stream", lambda dev: None)
    monkeypatch.setattr(stages, "_f32c", lambda t, name: t.contiguous())  # the real one refuses CPU tensors
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    return lib


def _ptr_val(p):
    return None if p is None else p.value


@pytest.mark.parametrize("D,stride,n_calls", [(1, 1, 1), (3, 4, 1), (5, 8, 1), (8, 8, 1), (33, 36, 2), (40, 40, 2),
                                              (64, 64, 2)])
@pytest.mark.parametrize("per_camera", [False, True])
def test_stage_chunking_and_padding(fake_lib, D, stride, n_calls, per_camera):
    C, N = 2, 7
    feats = torch.rand(C, N, D) if per_camera else torch.rand(N, D)
    splats = torch.zeros(C, N, SPLAT)
    offs = torch.zeros(C, 1, 2, dtype=torch.int32)
    flat = torch.zeros(5, dtype=torch.int32)
    bg = torch.rand(C, D)
    rc, ra, last = stages.rasterize_fwd_features(splats, offs, flat, feats, bg, W, H)
    assert rc.shape == (C, H, W, D) and ra.shape == (C, H, W, 1) and last.shape == (C, H, W)
    assert len(fake_lib.fwd) == n_calls
    for i, a in enumerate(fake_lib.fwd):
        c0, ch = stages.feature_chunks(D)[i]
        assert a[7:12] == (stride, int(not per_camera), D, c0, ch)  # feat_stride, shared_rows, D, c0, CH
        # first chunk writes alphas and last_ids, the others pass NULL
        assert (_ptr_val(a[18]) is not None, _ptr_val(a[19]) is not None) == (i == 0, i == 0)
        assert _ptr_val(a[17]) == rc.data_ptr()
    rows_ptr = _ptr_val(fake_lib.fwd[0][6])
    assert (rows_ptr == feats.data_ptr()) == (stride == D)  # no copy when the rows already have the kernels' width

    v_rc, v_ra = torch.rand(C, H, W, D), torch.rand(C, H, W, 1)
    v_splats, v_feats = stages.rasterize_bwd_features(splats, offs, flat, feats, bg, W, H, ra, last, v_rc, v_ra)
    assert v_splats.shape == (C, N, SPLAT) and v_feats.shape == feats.shape
    assert len(fake_lib.bwd) == n_calls
    for i, a in enumerate(fake_lib.bwd):
        assert a[7] == stride
        assert (_ptr_val(a[20]) is not None) == (i == 0)  # v_render_alphas: first chunk only
        assert _ptr_val(a[21]) == v_splats.data_ptr() and _ptr_val(a[22]) is not None
    fake_lib.bwd.clear()
    _, none = stages.rasterize_bwd_features(splats, offs, flat, feats, bg, W, H, ra, last, v_rc, v_ra,
                                            want_features_grad=False)
    assert none is None and all(_ptr_val(a[22]) is None for a in fake_lib.bwd)


def test_feature_entries_reject_bad_arguments_before_any_launch():
    lib = _lib.load()
    aligned, odd = ctypes.c_void_p(1 << 20), ctypes.c_void_p((1 << 20) + 4)

    def fwd(stride, D, c0, CH, feats=aligned):
        return lib.egs_rasterize_fwd_features(1, 10, 0, None, None, None, feats, stride, 1, D, c0, CH, None, 16, 16, 1, 1,
                                              None, None, None, None, None)

    def bwd(stride, D, c0, CH, feats=aligned):
        return lib.egs_rasterize_bwd_features(1, 10, 5, None, None, None, feats, stride, 1, D, c0, CH, None, 16, 16, 1, 1,
                                              None, None, None, None, None, None, None, None)

    for call in (fwd, bwd):
        for CH in (0, 3, 5, 64):
            assert call(64, 40, 0, CH) == -1 and b"CH=" in lib.egs_last_error_string()
        assert call(40, 40, 40, 8) == -1 and b"c0=40" in lib.egs_last_error_string()
        assert call(40, 40, -1, 8) == -1 and b"c0=-1" in lib.egs_last_error_string()
        assert call(8, 0, 0, 8) == -1 and b"D=0" in lib.egs_last_error_string()
        assert call(33, 33, 0, 32) == -1 and b"aligned" in lib.egs_last_error_string()  # stride 33 for CH = 32
        assert call(6, 5, 0, 4) == -1 and b"aligned" in lib.egs_last_error_string()
        assert call(8, 5, 0, 8, feats=odd) == -1 and b"aligned" in lib.egs_last_error_string()
        assert call(3, 3, 0, 2) == -1 and b"aligned" in lib.egs_last_error_string()
        assert call(4, 5, 0, 8) == -1 and b"feat_stride=4" in lib.egs_last_error_string()
        assert call(8, 5, 0, 8, feats=None) == -1 and b"features" in lib.egs_last_error_string()
    # the tile grid is checked first, as in the RGB entries
    assert lib.egs_rasterize_fwd_features(1, 10, 0, None, None, None, aligned, 8, 1, 5, 0, 8, None, 100, 100, 3, 3, None,
                                          None, None, None, None) == -1
    assert b"tile grid" in lib.egs_last_error_string()
