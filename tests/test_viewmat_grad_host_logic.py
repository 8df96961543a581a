"""CPU tests of the host logic of view-matrix gradients in rendering.py: which stage calls the backward pass makes and with
which keywords, where the [C,4,4] gradient lands (autograd input 5 of rasterization(), 6 of
rasterization_from_parameters()), and that a strided viewmats carries it back to its source — with the stage operators
replaced by CPU stand-ins that record their calls."""
import pytest
import torch

from easy_gaussian_splatting_b200 import rendering, stages

SPLAT = stages.SPLAT_FLOATS


class RecordingStages:
    """Shape-faithful stand-ins; the backward operators record their keyword names and return constants."""

    def __init__(self):
        self.calls = []
        self.bwd_kwargs = []

    def projection_fwd(self, means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d=0.3,
                       near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16, antialiased=False):
        self.calls.append("projection_fwd")
        return self._proj(viewmats.shape[0], means, antialiased)

    def projection_fwd_raw(self, means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width, height,
                           sh_degree, eps2d=0.3, near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16):
        self.calls.append("projection_fwd_raw")
        return self._proj(viewmats.shape[0], means, False)

    @staticmethod
    def _proj(C, means, antialiased):
        N = means.shape[0]
        vis = torch.ones(C, N, dtype=torch.bool)
        out = {
            "radii": torch.full((C, N), 4, dtype=torch.int32),
            "means2d": means.detach()[None, :, :2].expand(C, N, 2).contiguous(),
            "depths": torch.ones(C, N),
            "conics": torch.ones(C, N, 3),
            "colors": torch.full((C, N, 3), 0.5),
            "tiles_per_gauss": vis.int(),
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

    def projection_bwd(self, means, quats, scales, colors, viewmats, Ks, width, height, sh_degree, eps2d, radii,
                       colors_rgb, v_splats, v_means2d_extra=None, **kw):
        self.calls.append("projection_bwd")
        self.bwd_kwargs.append(sorted(kw))
        C, N = radii.shape
        outs = tuple(torch.full_like(t, float(i + 1)) for i, t in enumerate((means, quats, scales, means[:, 0], colors)))
        if kw.get("want_absgrad"):
            outs += (torch.zeros(C, N, 2),)
        if kw.get("want_viewmats_grad"):
            outs += (torch.arange(C * 16, dtype=torch.float32).reshape(C, 4, 4) + 100.0,)
        return outs

    def projection_bwd_raw(self, means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width, height,
                           sh_degree, eps2d, radii, colors_rgb, v_splats, v_means2d_extra=None, **kw):
        self.calls.append("projection_bwd_raw")
        self.bwd_kwargs.append(sorted(kw))
        C, N = radii.shape
        outs = tuple(torch.full_like(t, float(i + 1)) for i, t in
                     enumerate((means, quats, log_scales, logit_opacities, sh_0, sh_rest)))
        if kw.get("want_absgrad"):
            outs += (torch.zeros(C, N, 2),)
        if kw.get("want_viewmats_grad"):
            outs += (torch.arange(C * 16, dtype=torch.float32).reshape(C, 4, 4) - 50.0,)
        return outs


@pytest.fixture()
def rec(monkeypatch):
    f = RecordingStages()
    for name in ("projection_fwd", "projection_fwd_raw", "isect_sorted_async", "rasterize_fwd", "rasterize_bwd",
                 "projection_bwd", "projection_bwd_raw"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    monkeypatch.delenv("EGS_BWD_SEGMENT", raising=False)
    return f


def _params(N=10, C=2):
    g = torch.Generator().manual_seed(0)
    p = [torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
         torch.rand(N, generator=g), torch.randn(N, 16, 3, generator=g)]
    return [t.requires_grad_(True) for t in p], torch.eye(4)[None].repeat(C, 1, 1), torch.eye(3)[None].repeat(C, 1, 1)


EXPECTED_VM = torch.arange(32, dtype=torch.float32).reshape(2, 4, 4) + 100.0


@pytest.mark.parametrize("mode", ["classic", "antialiased"])
@pytest.mark.parametrize("absgrad", [False, True])
def test_viewmats_grad_arrives_at_input_5(rec, mode, absgrad):
    p, vm, K = _params()
    vm.requires_grad_(True)
    rc, ra, meta = rendering.rasterization(*p, vm, K, 32, 16, sh_degree=3, packed=False, absgrad=absgrad,
                                           rasterize_mode=mode)
    rc.sum().backward()
    assert vm.grad is not None and vm.grad.shape == (2, 4, 4)
    assert torch.equal(vm.grad, EXPECTED_VM)
    assert [t.grad.flatten()[0].item() for t in p] == [1.0, 2.0, 3.0, 4.0, 5.0]
    assert rec.calls[-1] == "projection_bwd" and "want_viewmats_grad" in rec.bwd_kwargs[-1]
    assert K.grad is None
    if absgrad:
        assert meta["means2d"].absgrad.shape == (2, 10, 2)  # absgrad still comes from out[5]


def test_without_viewmats_grad_the_backward_calls_are_unchanged(rec):
    """viewmats that do not require grad: the same stage calls with exactly the keywords the classic path passes."""
    p, vm, K = _params()
    for absgrad, mode in ((True, "classic"), (False, "classic"), (False, "antialiased")):
        rec.calls.clear()
        rec.bwd_kwargs.clear()
        rc, _, _ = rendering.rasterization(*p, vm, K, 32, 16, sh_degree=3, packed=False, absgrad=absgrad, rasterize_mode=mode)
        rc.sum().backward()
        assert rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd", "rasterize_bwd", "projection_bwd"]
        assert rec.bwd_kwargs == [["antialiased_opacities", "opacities", "want_absgrad"]]
    assert vm.grad is None
    rec.calls.clear()
    rec.bwd_kwargs.clear()
    rc = _raw_apply(p, vm, K, absgrad=False)[0]
    rc.sum().backward()
    assert rec.calls[-1] == "projection_bwd_raw" and rec.bwd_kwargs == [["want_absgrad"]]


def _raw_apply(p, vm, K, absgrad):
    """rasterization_from_parameters() refuses CPU tensors before anything else: drive its autograd node directly."""
    sh0, shr = p[4][:, :1].detach().requires_grad_(True), p[4][:, 1:].detach().requires_grad_(True)
    cfg = dict(width=32, height=16, sh_degree=3, eps2d=0.3, near_plane=0.01, far_plane=1e10, radius_clip=0.0,
               absgrad=absgrad, grad_enabled=True)
    outs = rendering._RasterizationRaw.apply(p[0], p[1], p[2], p[3], sh0, shr, vm, K, None, cfg)
    return outs[0], sh0, shr


def test_raw_entry_viewmats_grad_at_input_6(rec):
    p, vm, K = _params()
    vm.requires_grad_(True)
    rc, sh0, shr = _raw_apply(p, vm, K, absgrad=False)
    rc.sum().backward()
    assert rec.calls[-1] == "projection_bwd_raw" and "want_viewmats_grad" in rec.bwd_kwargs[-1]
    assert torch.equal(vm.grad, torch.arange(32, dtype=torch.float32).reshape(2, 4, 4) - 50.0)
    assert shr.grad is not None and float(shr.grad.flatten()[0]) == 6.0


def test_strided_viewmats_carry_the_gradient_to_their_source(rec):
    """viewmats = inverse(c2w) is a fresh, non-leaf tensor (and a transpose view is not even contiguous): autograd on
    the original carries the [C,4,4] gradient through the inverse to the c2w leaf."""
    p, _, K = _params()
    c2w = (torch.eye(4)[None].repeat(2, 1, 1) + 0.01 * torch.randn(2, 4, 4, generator=torch.Generator().manual_seed(1)))
    c2w[:, 3] = torch.tensor([0.0, 0.0, 0.0, 1.0])
    c2w.requires_grad_(True)
    vm = torch.linalg.inv(c2w).transpose(1, 2).transpose(1, 2)
    rc, _, _ = rendering.rasterization(*p, vm, K, 32, 16, sh_degree=3, packed=False)
    rc.sum().backward()
    inv = torch.linalg.inv(c2w.detach())
    expect = -(inv.transpose(1, 2) @ EXPECTED_VM @ inv.transpose(1, 2))  # VJP of the inverse
    assert c2w.grad is not None and torch.allclose(c2w.grad, expect, rtol=1e-5, atol=1e-4)


def test_no_grad_mode_ignores_requires_grad(rec):
    p, vm, K = _params()
    vm.requires_grad_(True)
    with torch.no_grad():
        rc, _, _ = rendering.rasterization(*p, vm, K, 32, 16, sh_degree=3, packed=False)
    assert rc.grad_fn is None and rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd"]
