"""CPU tests of the host logic of the expected-depth render modes ("ED", "RGB+ED") in rendering.py, with the stages
replaced by shape-faithful stand-ins: mode validation, the stage calls of each mode and colour kind (no checkpointed
forward in the depth modes), what the blend is given (the depth column and its zero background), output shapes, the
ED division with its 1e-10 clamp and its gradient into the alphas, the gradients that stay None in "ED", the depth
cotangent routed into slot 11 of the gradient records, and meta equal to "RGB"'s."""
import pytest
import torch

from easy_gaussian_splatting_b200 import rendering, stages

C, N, W, H = 2, 12, 40, 24
SPLAT = stages.SPLAT_FLOATS
ACC_DEPTH = 2.0  # accumulated depth the stand-in blend returns at every ordinary pixel (alpha 0.5)


class DepthStages:
    def __init__(self):
        self.calls = []
        self.seen = {}

    def projection_fwd(self, means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d=0.3,
                       near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16, antialiased=False):
        self.calls.append("projection_fwd")
        C_, N_ = viewmats.shape[0], means.shape[0]
        vis = (torch.arange(C_ * N_).reshape(C_, N_) % 3) != 0
        out = {
            "radii": (vis.int() * 4),
            "means2d": (means.detach()[None, :, :2] + torch.arange(C_)[:, None, None]) * vis[..., None],
            "depths": (torch.arange(C_ * N_, dtype=torch.float32).reshape(C_, N_) + 1.0) * vis,
            "conics": torch.ones(C_, N_, 3) * vis[..., None],
            "colors": torch.full((C_, N_, 3), 0.5) * vis[..., None],
            "tiles_per_gauss": vis.int() * 2,
            "tight_rects": torch.zeros(C_, N_, 2, dtype=torch.int32),
            "splats": torch.zeros(C_, N_, SPLAT),
        }
        if antialiased:
            out["compensations"] = torch.full((C_, N_), 0.5) * vis
        return out

    def isect_tiles(self, means2d, radii, depths, tile_size, tw, th, sort=True, tiles_per_gauss=None, n_isects=None):
        flat = (radii.reshape(-1) > 0).nonzero(as_tuple=True)[0].int()
        return tiles_per_gauss, torch.arange(flat.numel(), dtype=torch.int64), flat

    def isect_offset_encode(self, isect_ids, C_, tw, th):
        return torch.zeros(C_, th, tw, dtype=torch.int32)

    def isect_sorted_async(self, means2d, radii, depths, tiles_per_gauss, tile_size, tw, th, capacity=None, tight_rects=None):
        self.calls.append("isect_sorted")
        flat = (radii.reshape(-1) > 0).nonzero(as_tuple=True)[0].int()
        return stages.ResolvedIsects(lambda: torch.arange(flat.numel(), dtype=torch.int64), flat,
                                     torch.zeros(radii.shape[0], th, tw, dtype=torch.int32))

    @staticmethod
    def _alphas(C_, height, width):
        a = torch.full((C_, height, width, 1), 0.5)
        a[0, 0, 0, 0] = 0.0     # nothing blended: accumulated depth 0, clamped alpha
        a[0, 0, 1, 0] = 1e-12   # below the clamp
        return a

    def _images(self, C_, width, height, D, depth_last):
        rc = torch.full((C_, height, width, D), 0.25)
        if depth_last:
            rc[..., -1] = ACC_DEPTH
            rc[0, 0, 0, -1] = 0.0
            rc[0, 0, 1, -1] = 3e-12
        return rc, self._alphas(C_, height, width), torch.zeros(C_, height, width, dtype=torch.int32)

    def rasterize_fwd(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, count_pairs=False,
                      n_isects=None, tile_order=None):
        self.calls.append("rasterize_fwd")
        return self._images(splats.shape[0], width, height, 3, False)

    def rasterize_fwd_checkpointed(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, segment,
                                   seg_min_len=0, n_isects=None, tile_order=None):
        self.calls.append("rasterize_fwd_checkpointed")
        return (*self._images(splats.shape[0], width, height, 3, False), torch.zeros(16))

    def rasterize_bwd(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_alphas, last_ids,
                      v_render_colors, v_render_alphas, n_isects=None, tile_order=None):
        self.calls.append("rasterize_bwd")
        return torch.ones_like(splats)

    def rasterize_bwd_segmented(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_colors,
                                render_alphas, last_ids, v_render_colors, v_render_alphas, checkpoints, segment,
                                seg_min_len=0, n_isects=None, tile_order=None):
        self.calls.append("rasterize_bwd_segmented")
        return torch.ones_like(splats)

    def rasterize_fwd_depth(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, n_isects=None,
                            tile_order=None):
        self.calls.append("rasterize_fwd_depth")
        self.seen["fwd_bg"] = backgrounds
        return self._images(splats.shape[0], width, height, 4, True)

    def rasterize_bwd_depth(self, splats, isect_offsets, flatten_ids, backgrounds, width, height, render_alphas,
                            last_ids, v_render_colors, v_render_alphas, n_isects=None, tile_order=None):
        self.calls.append("rasterize_bwd_depth")
        self.seen.update(bwd_bg=backgrounds, v_colors=v_render_colors, v_alphas=v_render_alphas)
        v = torch.ones_like(splats)
        v[..., 11] = 5.0
        return v

    def rasterize_fwd_features(self, splats, isect_offsets, flatten_ids, features, backgrounds, width, height,
                               n_isects=None, tile_order=None):
        self.calls.append("rasterize_fwd_features")
        self.seen.update(features=features, fwd_bg=backgrounds)
        return self._images(splats.shape[0], width, height, features.shape[-1], True)

    def rasterize_bwd_features(self, splats, isect_offsets, flatten_ids, features, backgrounds, width, height,
                               render_alphas, last_ids, v_render_colors, v_render_alphas, n_isects=None,
                               tile_order=None, want_features_grad=True):
        self.calls.append("rasterize_bwd_features")
        self.seen.update(bwd_features=features, bwd_bg=backgrounds, v_colors=v_render_colors, v_alphas=v_render_alphas,
                         want_features_grad=want_features_grad)
        v_feat = torch.arange(features.numel(), dtype=torch.float32).reshape(features.shape)
        return torch.ones_like(splats), v_feat

    def projection_bwd(self, means, quats, scales, colors, viewmats, Ks, width, height, sh_degree, eps2d, radii,
                       colors_rgb, v_splats, v_means2d_extra=None, want_absgrad=False, antialiased_opacities=None,
                       opacities=None, **kw):
        self.calls.append("projection_bwd")
        self.seen.update(proj_kw=kw, v_splats=v_splats.clone())
        C_, N_ = radii.shape
        outs = [stages._grad_buffer(t).fill_(float(i + 1)) for i, t in enumerate((means, quats, scales, opacities, colors))]
        outs = tuple(outs) + ((torch.zeros(C_, N_, 2),) if want_absgrad else ())
        if kw.get("want_viewmats_grad"):
            outs += (torch.full((C_, 4, 4), 9.0),)
        if kw.get("want_Ks_grad"):
            outs += (torch.full((C_, 3, 3), 8.0),)
        return outs


@pytest.fixture()
def fake(monkeypatch):
    f = DepthStages()
    for name in ("projection_fwd", "isect_sorted_async", "isect_tiles", "isect_offset_encode", "rasterize_fwd",
                 "rasterize_fwd_checkpointed", "rasterize_bwd", "rasterize_bwd_segmented", "rasterize_fwd_depth",
                 "rasterize_bwd_depth", "rasterize_fwd_features", "rasterize_bwd_features", "projection_bwd"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    monkeypatch.setenv("EGS_BWD_SEGMENT", "128")  # forces the checkpointed forward wherever it may be used
    return f


def _inputs(kind):
    g = torch.Generator().manual_seed(0)
    colors = {"sh": torch.randn(N, 16, 3, generator=g), "rgb": torch.rand(N, 3, generator=g),
              "feat": torch.rand(N, 5, generator=g), "feat_cam": torch.rand(C, N, 5, generator=g)}[kind]
    p = [torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
         torch.rand(N, generator=g), colors]
    return [t.requires_grad_(True) for t in p], torch.eye(4)[None].repeat(C, 1, 1), torch.eye(3)[None].repeat(C, 1, 1)


def _call(kind, mode, bg=True, **kw):
    p, vm, K = _inputs(kind)
    D = p[4].shape[-1]
    backgrounds = torch.rand(C, D, generator=torch.Generator().manual_seed(1)).requires_grad_(True) if bg else None
    sh = 3 if kind == "sh" else None
    out = rendering.rasterization(*p, vm, K, W, H, sh_degree=sh, packed=False, absgrad=True, backgrounds=backgrounds,
                                  render_mode=mode, **kw)
    return out, p, backgrounds


@pytest.mark.parametrize("mode", ["D", "RGB+D", "depth", "rgb", ""])
def test_other_modes_raise(fake, mode):
    p, vm, K = _inputs("sh")
    with pytest.raises(NotImplementedError, match="'RGB', 'ED' and 'RGB\\+ED'"):
        rendering.rasterization(*p, vm, K, W, H, sh_degree=3, render_mode=mode)
    assert fake.calls == []


@pytest.mark.parametrize("kind", ["sh", "rgb", "feat", "feat_cam"])
@pytest.mark.parametrize("mode", ["RGB", "ED", "RGB+ED"])
def test_stage_calls_and_shapes(fake, kind, mode):
    (rc, ra, meta), p, bg = _call(kind, mode)
    D = p[4].shape[-1]
    assert rc.shape == (C, H, W, {"RGB": D, "ED": 1, "RGB+ED": D + 1}[mode]) and ra.shape == (C, H, W, 1)
    (rc.sum() + ra.sum()).backward()
    feat = kind.startswith("feat")
    if mode == "RGB":
        blend = ["rasterize_fwd_features", "rasterize_bwd_features"] if feat else ["rasterize_fwd_checkpointed",
                                                                                    "rasterize_bwd_segmented"]
    else:  # never the checkpointed forward
        blend = ["rasterize_fwd_features", "rasterize_bwd_features"] if feat else ["rasterize_fwd_depth",
                                                                                    "rasterize_bwd_depth"]
    assert fake.calls == ["projection_fwd", "isect_sorted", blend[0], blend[1], "projection_bwd"]
    assert fake.seen["proj_kw"] == ({} if mode == "RGB" else {"depth_grad": True})


@pytest.mark.parametrize("kind", ["sh", "feat"])
def test_ed_division_clamp_and_alpha_gradient(fake, kind):
    (rc, ra, _), p, _ = _call(kind, "ED")
    ed = rc[..., 0]
    assert torch.all(ed[1] == ACC_DEPTH / 0.5)
    assert ed[0, 0, 0] == 0.0                                            # 0 / clamp(0)
    assert torch.isclose(ed[0, 0, 1], torch.tensor(3e-12 / 1e-10))       # divided by the clamp, not by 1e-12
    rc.sum().backward()
    va, vc = fake.seen["v_alphas"], fake.seen["v_colors"]
    assert torch.allclose(va[1], torch.full_like(va[1], -ACC_DEPTH / 0.25))  # d(acc / alpha) / d alpha
    assert va[0, 0, 0, 0] == 0.0 and va[0, 0, 1, 0] == 0.0                  # clamped: no alpha gradient
    assert torch.allclose(vc[1, ..., -1], torch.full_like(vc[1, ..., -1], 2.0))  # 1 / alpha on the depth channel
    if kind == "sh":
        assert torch.all(vc[..., :3] == 0)  # the RGB channels of the depth blend are not part of the output


@pytest.mark.parametrize("kind", ["sh", "rgb", "feat", "feat_cam"])
def test_ed_leaves_colour_and_background_gradients_none(fake, kind):
    (rc, ra, _), p, bg = _call(kind, "ED")
    assert fake.seen["fwd_bg"] is None
    (rc.sum() + ra.sum()).backward()
    assert p[4].grad is None and bg.grad is None
    assert all(t.grad is not None for t in p[:4])


@pytest.mark.parametrize("kind", ["sh", "feat", "feat_cam"])
def test_rgb_ed_backgrounds_get_the_colour_channels(fake, kind):
    (rc, ra, _), p, bg = _call(kind, "RGB+ED")
    D = p[4].shape[-1]
    (rc * torch.arange(D + 1, dtype=torch.float32)).sum().backward()
    assert bg.grad.shape == (C, D)
    ref = ((1.0 - ra.detach()) * torch.arange(D, dtype=torch.float32)).sum(dim=(1, 2))
    assert torch.allclose(bg.grad, ref)
    assert p[4].grad is not None and p[4].grad.shape == p[4].shape


def test_feature_blend_gets_the_depth_column(fake):
    (rc, ra, meta), p, bg = _call("feat", "RGB+ED")
    f, fbg = fake.seen["features"], fake.seen["fwd_bg"]
    assert f.shape == (C, N, 6) and fbg.shape == (C, 6)
    assert torch.equal(f[..., :5], p[4].detach()[None].expand(C, N, 5))
    assert torch.equal(f[..., 5], meta["depths"]) and torch.all(fbg[:, 5] == 0) and torch.equal(fbg[:, :5], bg.detach())
    rc.sum().backward()
    v_feat = torch.arange(C * N * 6, dtype=torch.float32).reshape(C, N, 6)
    assert torch.equal(fake.seen["v_splats"][..., 11], v_feat[..., 5])  # the depth column's gradient -> slot 11
    assert torch.equal(p[4].grad, v_feat[..., :5].sum(0))                 # shared rows: summed over the cameras
    fake.seen.clear()
    (rc, _, meta), p, _ = _call("feat_cam", "ED")
    assert fake.seen["features"].shape == (C, N, 1) and torch.equal(fake.seen["features"][..., 0], meta["depths"])
    rc.sum().backward()
    assert fake.seen["want_features_grad"] and torch.equal(fake.seen["v_splats"][..., 11],
                                                           torch.arange(C * N, dtype=torch.float32).reshape(C, N))


def test_rgb_depth_blend_backgrounds(fake):
    _call("sh", "RGB+ED")[0][0].sum().backward()
    assert fake.seen["fwd_bg"].shape == (C, 3) and fake.seen["bwd_bg"].shape == (C, 3)
    assert fake.seen["v_colors"].shape == (C, H, W, 4)
    assert torch.all(fake.seen["v_splats"][..., 11] == 5.0)  # what the depth blend wrote reaches the projection


@pytest.mark.parametrize("kind", ["sh", "feat"])
@pytest.mark.parametrize("packed", [False, True])
def test_meta_equals_rgb(fake, kind, packed):
    metas = {}
    for mode in ("RGB", "ED", "RGB+ED"):
        (_, ra, meta), _, _ = _call_packed(kind, mode, packed)
        metas[mode] = (dict(meta.items()), ra)
    ref, ra_ref = metas["RGB"]
    for mode in ("ED", "RGB+ED"):
        m, ra = metas[mode]
        assert torch.equal(ra, ra_ref)
        assert m.keys() == ref.keys()
        for k, v in ref.items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(m[k], v), (mode, k)
            else:
                assert m[k] == v, (mode, k)


def _call_packed(kind, mode, packed):
    p, vm, K = _inputs(kind)
    sh = 3 if kind == "sh" else None
    return rendering.rasterization(*p, vm, K, W, H, sh_degree=sh, packed=packed, render_mode=mode), p, None


def test_camera_gradients_in_depth_modes(fake):
    p, vm, K = _inputs("sh")
    vm.requires_grad_(True)
    K.requires_grad_(True)
    rc, _, _ = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False, render_mode="RGB+ED")
    rc.sum().backward()
    assert fake.seen["proj_kw"] == {"want_viewmats_grad": True, "want_Ks_grad": True, "depth_grad": True}
    assert torch.all(vm.grad == 9.0) and torch.all(K.grad == 8.0)


def test_no_grad_forward(fake):
    p, vm, K = _inputs("sh")
    with torch.no_grad():
        rc, ra, _ = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, render_mode="RGB+ED")
    assert rc.grad_fn is None and rc.shape == (C, H, W, 4)
    assert fake.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd_depth"]
