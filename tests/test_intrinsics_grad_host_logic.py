"""CPU tests of the host logic of intrinsics gradients: which stage calls the backward pass makes and with which keywords,
where the [C,3,3] gradient lands (autograd input 6 of rasterization(), 7 of rasterization_from_parameters()), that an
expanded Ks carries it back to its source, which C entry the stages call, and the C entries' argument checks, which run
before any launch and need no GPU.  The stage operators are replaced by CPU stand-ins that record their calls."""
import contextlib
import ctypes

import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rendering, stages

SPLAT = stages.SPLAT_FLOATS
W, H = 32, 16
CALLS = ["projection_fwd", "isect_sorted", "rasterize_fwd", "rasterize_bwd", "projection_bwd"]


def _vks(C):
    return torch.arange(C * 9, dtype=torch.float32).reshape(C, 3, 3) + 200.0


def _vvm(C):
    return torch.arange(C * 16, dtype=torch.float32).reshape(C, 4, 4) + 100.0


class RecordingStages:
    """Shape-faithful stand-ins; the backward operators record their keyword names and return constants."""

    def __init__(self):
        self.calls = []
        self.bwd_kwargs = []

    def projection_fwd(self, means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d=0.3,
                       near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16, antialiased=False):
        self.calls.append("projection_fwd")
        self.fwd_Ks = Ks
        return self._proj(viewmats.shape[0], means, antialiased)

    def projection_fwd_raw(self, means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width, height,
                           sh_degree, eps2d=0.3, near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16):
        self.calls.append("projection_fwd_raw")
        return self._proj(viewmats.shape[0], means, False)

    @staticmethod
    def _proj(C, means, antialiased):
        N = means.shape[0]
        radii = torch.full((C, N), 4, dtype=torch.int32)
        radii[:, ::3] = 0  # some culled entries, so that packed=True has something to drop
        out = {
            "radii": radii,
            "means2d": means.detach()[None, :, :2].expand(C, N, 2).contiguous(),
            "depths": torch.ones(C, N),
            "conics": torch.ones(C, N, 3),
            "colors": torch.full((C, N, 3), 0.5),
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
        self.calls.append("rasterize_fwd")
        C, D = splats.shape[0], features.shape[-1]
        return (torch.full((C, height, width, D), 0.25), torch.full((C, height, width, 1), 0.5),
                torch.zeros(C, height, width, dtype=torch.int32))

    def rasterize_bwd_features(self, splats, isect_offsets, flatten_ids, features, backgrounds, width, height,
                               render_alphas, last_ids, v_render_colors, v_render_alphas, n_isects=None, tile_order=None,
                               want_features_grad=True):
        self.calls.append("rasterize_bwd")
        return torch.ones_like(splats), (torch.full_like(features, 7.0) if want_features_grad else None)

    @staticmethod
    def _camera_outs(C, kw):
        outs = ()
        if kw.get("want_viewmats_grad"):
            outs += (_vvm(C),)
        if kw.get("want_Ks_grad"):
            outs += (_vks(C),)
        return outs

    def projection_bwd(self, means, quats, scales, colors, viewmats, Ks, width, height, sh_degree, eps2d, radii,
                       colors_rgb, v_splats, v_means2d_extra=None, **kw):
        self.calls.append("projection_bwd")
        self.bwd_kwargs.append(sorted(kw))
        C, N = radii.shape
        outs = tuple(torch.full_like(t, float(i + 1)) for i, t in enumerate((means, quats, scales, means[:, 0], colors)))
        if kw.get("want_absgrad"):
            outs += (torch.zeros(C, N, 2),)
        return outs + self._camera_outs(C, kw)

    def projection_bwd_raw(self, means, quats, log_scales, logit_opacities, sh_0, sh_rest, viewmats, Ks, width, height,
                           sh_degree, eps2d, radii, colors_rgb, v_splats, v_means2d_extra=None, **kw):
        self.calls.append("projection_bwd_raw")
        self.bwd_kwargs.append(sorted(kw))
        C, N = radii.shape
        outs = tuple(torch.full_like(t, float(i + 1)) for i, t in
                     enumerate((means, quats, log_scales, logit_opacities, sh_0, sh_rest)))
        if kw.get("want_absgrad"):
            outs += (torch.zeros(C, N, 2),)
        return outs + self._camera_outs(C, kw)


@pytest.fixture()
def rec(monkeypatch):
    f = RecordingStages()
    for name in ("projection_fwd", "projection_fwd_raw", "isect_sorted_async", "rasterize_fwd", "rasterize_bwd",
                 "rasterize_fwd_features", "rasterize_bwd_features", "projection_bwd", "projection_bwd_raw"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    monkeypatch.delenv("EGS_BWD_SEGMENT", raising=False)
    return f


def _params(N=10, C=2, colors=None):
    g = torch.Generator().manual_seed(0)
    cols = torch.randn(N, 16, 3, generator=g) if colors is None else colors
    p = [torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
         torch.rand(N, generator=g), cols]
    return [t.requires_grad_(True) for t in p], torch.eye(4)[None].repeat(C, 1, 1), torch.eye(3)[None].repeat(C, 1, 1)


@pytest.mark.parametrize("mode", ["classic", "antialiased"])
@pytest.mark.parametrize("absgrad", [False, True])
def test_Ks_grad_arrives_at_input_6(rec, mode, absgrad):
    p, vm, K = _params()
    K.requires_grad_(True)
    rc, ra, meta = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False, absgrad=absgrad,
                                           rasterize_mode=mode, backgrounds=torch.zeros(2, 3))
    rc.sum().backward()
    assert K.grad is not None and K.grad.shape == (2, 3, 3)
    assert torch.equal(K.grad, _vks(2))
    assert [t.grad.flatten()[0].item() for t in p] == [1.0, 2.0, 3.0, 4.0, 5.0]
    assert rec.calls == CALLS
    assert "want_Ks_grad" in rec.bwd_kwargs[-1] and "want_viewmats_grad" not in rec.bwd_kwargs[-1]
    assert vm.grad is None
    if absgrad:
        assert meta["means2d"].absgrad.shape == (2, 10, 2)  # absgrad still comes from out[5]


def test_viewmats_and_Ks_together_make_one_backward_call(rec):
    p, vm, K = _params()
    vm.requires_grad_(True)
    K.requires_grad_(True)
    rc, _, _ = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False, absgrad=True)
    rc.sum().backward()
    assert rec.calls == CALLS  # one projection backward for both
    assert rec.bwd_kwargs[-1] == ["antialiased_opacities", "opacities", "want_Ks_grad", "want_absgrad",
                                  "want_viewmats_grad"]
    assert torch.equal(vm.grad, _vvm(2)) and torch.equal(K.grad, _vks(2))


def test_without_Ks_grad_the_backward_calls_are_unchanged(rec):
    """Ks that do not require grad: the same stage calls with exactly the keywords of today's calls."""
    p, vm, K = _params()
    for absgrad, mode in ((True, "classic"), (False, "classic"), (False, "antialiased")):
        rec.calls.clear()
        rec.bwd_kwargs.clear()
        rc, _, _ = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False, absgrad=absgrad, rasterize_mode=mode)
        rc.sum().backward()
        assert rec.calls == CALLS
        assert rec.bwd_kwargs == [["antialiased_opacities", "opacities", "want_absgrad"]]
    vm.requires_grad_(True)  # viewmats alone: today's single viewmat keyword
    rec.bwd_kwargs.clear()
    rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False)[0].sum().backward()
    assert rec.bwd_kwargs == [["antialiased_opacities", "opacities", "want_absgrad", "want_viewmats_grad"]]
    assert K.grad is None
    rec.bwd_kwargs.clear()
    rc = _raw_apply(p, vm.detach(), K, absgrad=False)[0]
    rc.sum().backward()
    assert rec.calls[-1] == "projection_bwd_raw" and rec.bwd_kwargs == [["want_absgrad"]]


def _raw_apply(p, vm, K, absgrad):
    """rasterization_from_parameters() refuses CPU tensors before anything else: drive its autograd node directly."""
    sh0, shr = p[4][:, :1].detach().requires_grad_(True), p[4][:, 1:].detach().requires_grad_(True)
    cfg = dict(width=W, height=H, sh_degree=3, eps2d=0.3, near_plane=0.01, far_plane=1e10, radius_clip=0.0,
               absgrad=absgrad, grad_enabled=True)
    outs = rendering._RasterizationRaw.apply(p[0], p[1], p[2], p[3], sh0, shr, vm, K, None, cfg)
    return outs[0], sh0, shr


@pytest.mark.parametrize("with_vm", [False, True])
def test_raw_entry_Ks_grad_at_input_7(rec, with_vm):
    p, vm, K = _params()
    K.requires_grad_(True)
    vm.requires_grad_(with_vm)
    rc, sh0, shr = _raw_apply(p, vm, K, absgrad=True)
    rc.sum().backward()
    assert rec.calls[-1] == "projection_bwd_raw" and "want_Ks_grad" in rec.bwd_kwargs[-1]
    assert ("want_viewmats_grad" in rec.bwd_kwargs[-1]) == with_vm
    assert rec.calls.count("projection_bwd_raw") == 1
    assert torch.equal(K.grad, _vks(2))
    assert (vm.grad is not None) == with_vm and (not with_vm or torch.equal(vm.grad, _vvm(2)))
    assert shr.grad is not None and float(shr.grad.flatten()[0]) == 6.0


def test_expanded_Ks_sum_the_gradient_into_their_source(rec):
    """One learned focal length for all cameras: Ks built from a shared [3,3] by expand is a stride-0 view; the forward
    gets a dense copy and autograd sums the per-camera gradients into the source."""
    p, vm, _ = _params(C=3)
    vm = vm[:1].expand(3, -1, -1)
    K0 = torch.tensor([[100.0, 0.0, 16.0], [0.0, 100.0, 8.0], [0.0, 0.0, 1.0]], requires_grad=True)
    Ks = K0[None].expand(3, -1, -1)
    rc, _, _ = rendering.rasterization(*p, vm, Ks, W, H, sh_degree=3, packed=False)
    assert rec.fwd_Ks.is_contiguous() and rec.fwd_Ks.shape == (3, 3, 3)
    rc.sum().backward()
    assert torch.equal(K0.grad, _vks(3).sum(0))
    f = torch.tensor(100.0, requires_grad=True)  # a non-leaf built from one scalar
    Kf = torch.stack([torch.stack([f, f * 0, f * 0 + 16]), torch.stack([f * 0, f, f * 0 + 8]),
                      torch.tensor([0.0, 0.0, 1.0])])[None].repeat(3, 1, 1)
    rendering.rasterization(*p, vm, Kf, W, H, sh_degree=3, packed=False)[0].sum().backward()
    v = _vks(3).sum(0)
    assert torch.equal(f.grad, v[0, 0] + v[1, 1])  # fx = fy = f; the other entries reach f only through f * 0


@pytest.mark.parametrize("D,per_camera", [(5, False), (5, True), (3, True), (40, False)])
def test_feature_colours(rec, D, per_camera):
    C, N = 2, 10
    g = torch.Generator().manual_seed(1)
    cols = torch.rand(C, N, D, generator=g) if per_camera else torch.rand(N, D, generator=g)
    p, vm, K = _params(N=N, C=C, colors=cols)
    K.requires_grad_(True)
    rc, _, _ = rendering.rasterization(*p, vm, K, W, H, packed=False, backgrounds=torch.zeros(C, D))
    assert rc.shape == (C, H, W, D)
    rc.sum().backward()
    assert rec.calls == CALLS and "want_Ks_grad" in rec.bwd_kwargs[-1]
    assert torch.equal(K.grad, _vks(C))


def test_per_camera_sh_and_packed(rec):
    C, N = 2, 10
    cols = torch.randn(C, N, 16, 3, generator=torch.Generator().manual_seed(2))
    p, vm, K = _params(N=N, C=C, colors=cols)
    K.requires_grad_(True)
    rc, _, meta = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=True, absgrad=True)
    (rc.sum() + meta["means2d"].sum()).backward()
    assert meta["means2d"].shape[0] == int((torch.arange(N) % 3 != 0).sum()) * C  # packed: the visible pairs
    assert rec.calls == CALLS and "want_Ks_grad" in rec.bwd_kwargs[-1]
    assert torch.equal(K.grad, _vks(C)) and p[4].grad.shape == (C, N, 16, 3)


def test_no_grad_mode_ignores_requires_grad(rec):
    p, vm, K = _params()
    K.requires_grad_(True)
    with torch.no_grad():
        rc, _, _ = rendering.rasterization(*p, vm, K, W, H, sh_degree=3, packed=False)
    assert rc.grad_fn is None and rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd"]


# ---- stages -> C entries ----------------------------------------------------------------------------------------------

class FakeLib:
    """Records the projection entries' arguments instead of launching."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("egs_projection"):
            raise AttributeError(name)

        def rec(*a):
            self.calls.append((name, a))
            return 0
        return rec

    def egs_projection_bwd_viewmats_workspace_bytes(self, C, N):
        return 64

    def egs_projection_bwd_intrinsics_workspace_bytes(self, C, N):
        return 80


@pytest.fixture()
def fake_lib(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(stages, "_stream", lambda dev: None)
    monkeypatch.setattr(stages, "_f32c", lambda t, name: t.contiguous())  # the real one refuses CPU tensors
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    return lib


def _scene(N=7, C=3):
    g = torch.Generator().manual_seed(0)
    return (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
            torch.rand(N, generator=g), torch.randn(N, 16, 3, generator=g), torch.eye(4)[None].repeat(C, 1, 1),
            torch.eye(3)[None].repeat(C, 1, 1))


@pytest.mark.parametrize("want_vm", [False, True])
@pytest.mark.parametrize("antialiased", [False, True])
def test_stage_calls_the_intrinsics_entry(fake_lib, want_vm, antialiased):
    means, quats, scales, opac, cols, vm, Ks = _scene()
    C, N = vm.shape[0], means.shape[0]
    radii = torch.ones(C, N, dtype=torch.int32)
    out = stages.projection_bwd(means, quats, scales, cols, vm, Ks, W, H, 3, 0.3, radii, torch.zeros(C, N, 3),
                                torch.zeros(C, N, SPLAT), want_absgrad=True,
                                antialiased_opacities=opac if antialiased else None, opacities=opac,
                                want_viewmats_grad=want_vm, want_Ks_grad=True)
    assert len(fake_lib.calls) == 1
    name, a = fake_lib.calls[0]
    assert name == "egs_projection_bwd_intrinsics"
    assert len(out) == 6 + want_vm + 1 and out[-1].shape == (C, 3, 3)
    assert a[25] == int(antialiased)
    assert (a[26] is None) == (not want_vm)  # v_viewmats nullable
    assert a[27].value == out[-1].data_ptr() and a[29] == 80
    if want_vm:
        assert out[-2].shape == (C, 4, 4) and a[26].value == out[-2].data_ptr()
    out = stages.projection_bwd_raw(means, quats, scales, opac, cols[:, :1], cols[:, 1:], vm, Ks, W, H, 3, 0.3, radii,
                                    torch.zeros(C, N, 3), torch.zeros(C, N, SPLAT), want_viewmats_grad=want_vm,
                                    want_Ks_grad=True)
    name, a = fake_lib.calls[-1]
    assert name == "egs_projection_bwd_raw_intrinsics" and len(out) == 6 + want_vm + 1
    assert (a[25] is None) == (not want_vm) and a[26].value == out[-1].data_ptr() and a[28] == 80


def test_stage_without_Ks_keeps_the_viewmat_entry(fake_lib):
    means, quats, scales, opac, cols, vm, Ks = _scene()
    C, N = vm.shape[0], means.shape[0]
    radii = torch.ones(C, N, dtype=torch.int32)
    args = (means, quats, scales, cols, vm, Ks, W, H, 3, 0.3, radii, torch.zeros(C, N, 3), torch.zeros(C, N, SPLAT))
    stages.projection_bwd(*args, want_viewmats_grad=True)
    stages.projection_bwd(*args)
    assert [n for n, _ in fake_lib.calls] == ["egs_projection_bwd_viewmats", "egs_projection_bwd"]


# ---- C entries: rejections before any launch ---------------------------------------------------------------------------

def test_entries_reject_bad_arguments_before_any_launch():
    lib = _lib.load()
    n0 = lib.egs_kernel_launch_count()
    fake = ctypes.c_void_p(0x1000)  # non-null pointers that are never touched
    ws_need = lib.egs_projection_bwd_intrinsics_workspace_bytes(1, 10)
    assert ws_need > lib.egs_projection_bwd_viewmats_workspace_bytes(1, 10) > 0
    assert lib.egs_projection_bwd_intrinsics_workspace_bytes(0, 10) == 0

    def bwd(C, v_Ks, ws, ws_bytes, v_vm=None):
        return lib.egs_projection_bwd_intrinsics(C, 10, None, None, None, None, None, 16, 3, 0, None, None, 64, 64, 0.3,
                                                 None, None, None, None, None, None, None, None, None, None, 0, v_vm, v_Ks,
                                                 ws, ws_bytes, None)

    def bwd_raw(C, v_Ks, ws, ws_bytes, v_vm=None):
        return lib.egs_projection_bwd_raw_intrinsics(C, 10, None, None, None, None, fake, fake, 3, None, None, 64, 64,
                                                     0.3, None, None, None, None, None, None, None, None, fake, fake, None,
                                                     v_vm, v_Ks, ws, ws_bytes, None)

    for call in (bwd, bwd_raw):
        assert call(1, None, fake, ws_need) == -1 and b"v_Ks" in lib.egs_last_error_string()
        assert call(1, None, fake, ws_need, fake) == -1 and b"v_Ks" in lib.egs_last_error_string()
        assert call(1, fake, fake, ws_need - 1) == -1 and b"workspace" in lib.egs_last_error_string()
        assert call(1, fake, None, ws_need) == -1 and b"workspace" in lib.egs_last_error_string()
        big = lib.egs_projection_bwd_intrinsics_workspace_bytes(65536, 10)
        assert call(65536, fake, fake, big) == -1 and b"65535" in lib.egs_last_error_string()
    assert lib.egs_kernel_launch_count() == n0
