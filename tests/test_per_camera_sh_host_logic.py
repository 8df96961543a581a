"""CPU tests of per-camera SH coefficients [C,N,K,3]: shape validation in rendering._check_inputs, the stage calls and
their C arguments (colors_per_camera = 1 and K, through a stand-in library that records the calls), gradient and meta
shapes through rasterization() with recording stand-in stages, and the C entries' argument checks, which run before
any launch and need no GPU."""
import contextlib
import ctypes

import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rendering, stages
from easy_gaussian_splatting_b200.rendering import _check_inputs

SPLAT = stages.SPLAT_FLOATS
W, H = 32, 16


def _base(N=5, C=2):
    f = lambda *s: torch.zeros(*s)
    return dict(means=f(N, 3), quats=f(N, 4), scales=f(N, 3), opacities=f(N), viewmats=f(C, 4, 4), Ks=f(C, 3, 3),
                backgrounds=None)


def test_shape_validation():
    N, C = 5, 2
    base = _base(N, C)
    for deg, cols in ((3, torch.zeros(C, N, 16, 3)), (1, torch.zeros(C, N, 4, 3)), (0, torch.zeros(C, N, 1, 3)),
                      (2, torch.zeros(C, N, 9, 3))):
        with pytest.raises(RuntimeError, match="CUDA-only"):  # shape accepted; the CPU tensors are refused next
            _check_inputs(**base, colors=cols, sh_degree=deg)
    for cols in (torch.zeros(C + 1, N, 16, 3), torch.zeros(1, N, 16, 3), torch.zeros(C, N + 1, 16, 3),  # leading dims
                 torch.zeros(C, N, 16, 4), torch.zeros(C, N, 16, 1),  # last dimension
                 torch.zeros(C, N, 9, 3), torch.zeros(C, N, 15, 3)):  # K too small for degree 3
        with pytest.raises(ValueError, match="colors|K >="):
            _check_inputs(**base, colors=cols, sh_degree=3)
    # without sh_degree a 4-D colour tensor stays an error
    with pytest.raises(ValueError, match="colors"):
        _check_inputs(**base, colors=torch.zeros(C, N, 16, 3), sh_degree=None)


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


@pytest.fixture()
def fake_lib(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(stages, "_stream", lambda dev: None)
    monkeypatch.setattr(stages, "_f32c", lambda t, name: t.contiguous())  # the real one refuses CPU tensors
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    return lib


def _scene(N=7, C=3, K=16):
    g = torch.Generator().manual_seed(0)
    return (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
            torch.rand(N, generator=g), torch.randn(C, N, K, 3, generator=g), torch.eye(4)[None].repeat(C, 1, 1),
            torch.eye(3)[None].repeat(C, 1, 1))


@pytest.mark.parametrize("K,deg", [(16, 3), (9, 2), (4, 1), (25, 3)])
@pytest.mark.parametrize("antialiased", [False, True])
def test_stage_calls_pass_per_camera_flag_and_K(fake_lib, K, deg, antialiased):
    means, quats, scales, opac, cols, vm, Ks = _scene(K=K)
    C, N = vm.shape[0], means.shape[0]
    stages.projection_fwd(means, quats, scales, opac, cols, vm, Ks, W, H, deg, antialiased=antialiased)
    name, a = fake_lib.calls[-1]
    assert name == ("egs_projection_fwd_antialiased" if antialiased else "egs_projection_fwd")
    assert a[:2] == (C, N) and a[7:10] == (K, deg, 1)  # K, sh_degree, colors_per_camera
    assert a[6].value == cols.data_ptr()
    radii = torch.ones(C, N, dtype=torch.int32)
    for want_vm in (False, True):
        out = stages.projection_bwd(means, quats, scales, cols, vm, Ks, W, H, deg, 0.3, radii, torch.zeros(C, N, 3),
                                    torch.zeros(C, N, SPLAT), antialiased_opacities=opac if antialiased else None,
                                    opacities=opac, want_viewmats_grad=want_vm)
        name, a = fake_lib.calls[-1]
        assert name == ("egs_projection_bwd_viewmats" if want_vm else
                        "egs_projection_bwd_antialiased" if antialiased else "egs_projection_bwd")
        tail = a[6:] if (want_vm or antialiased) else a[5:]  # after the opacities argument, if there is one
        assert tail[0].value == cols.data_ptr() and tail[1:4] == (K, deg, 1)
        assert out[4].shape == (C, N, K, 3)  # v_colors: one row per (camera, Gaussian)
        assert tail[17].value == out[4].data_ptr()


def test_shared_coefficients_still_pass_zero(fake_lib):
    means, quats, scales, opac, cols, vm, Ks = _scene()
    stages.projection_fwd(means, quats, scales, opac, cols[0], vm, Ks, W, H, 3)
    assert fake_lib.calls[-1][1][7:10] == (16, 3, 0)


class RecordingStages:
    """Shape-faithful stand-ins that record their calls and return constants."""

    def __init__(self):
        self.calls = []

    def projection_fwd(self, means, quats, scales, opacities, colors, viewmats, Ks, width, height, sh_degree, eps2d=0.3,
                       near_plane=0.01, far_plane=1e10, radius_clip=0.0, tile_size=16, antialiased=False):
        self.calls.append("projection_fwd")
        self.proj_colors = colors
        C, N = viewmats.shape[0], means.shape[0]
        radii = torch.full((C, N), 4, dtype=torch.int32)
        radii[:, ::3] = 0
        return {"radii": radii, "means2d": means.detach()[None, :, :2].expand(C, N, 2).contiguous(),
                "depths": torch.ones(C, N), "conics": torch.ones(C, N, 3),
                "colors": torch.arange(C * N * 3, dtype=torch.float32).reshape(C, N, 3),
                "tiles_per_gauss": (radii > 0).int(), "tight_rects": torch.zeros(C, N, 2, dtype=torch.int32),
                "splats": torch.zeros(C, N, SPLAT)}

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
    for name in ("projection_fwd", "isect_sorted_async", "rasterize_fwd", "rasterize_bwd", "projection_bwd"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    monkeypatch.delenv("EGS_BWD_SEGMENT", raising=False)
    return f


@pytest.mark.parametrize("packed", [False, True])
def test_gradient_and_meta_shapes(rec, packed):
    means, quats, scales, opac, cols, vm, Ks = _scene(N=10, C=2)
    p = [t.requires_grad_(True) for t in (means, quats, scales, opac, cols)]
    vm.requires_grad_(True)
    rc, ra, meta = rendering.rasterization(*p, vm, Ks, W, H, sh_degree=3, packed=packed, absgrad=True,
                                           backgrounds=torch.zeros(2, 3))
    assert rc.shape == (2, H, W, 3)
    assert rec.proj_colors.shape == (2, 10, 16, 3) and torch.equal(rec.proj_colors, cols.detach())
    vis = torch.ones(2, 10, dtype=torch.bool)
    vis[:, ::3] = False
    rgb = torch.arange(2 * 10 * 3, dtype=torch.float32).reshape(2, 10, 3)
    if packed:
        assert torch.equal(meta["colors"], rgb[vis])  # [nnz,3]
    else:
        assert torch.equal(meta["colors"], rgb)  # [C,N,3]
    rc.sum().backward()
    assert rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd", "rasterize_bwd", "projection_bwd"]
    assert rec.bwd_colors.shape == (2, 10, 16, 3)
    assert cols.grad.shape == (2, 10, 16, 3) and torch.all(cols.grad == 5.0)
    assert vm.grad.shape == (2, 4, 4)


def test_strided_per_camera_input_is_made_dense_once(rec):
    means, quats, scales, opac, cols, vm, Ks = _scene(N=10, C=3)
    shs = cols[0].clone().requires_grad_(True)
    expanded = shs[None].expand(3, -1, -1, -1)  # stride 0 over cameras
    rc, _, _ = rendering.rasterization(means, quats, scales, opac, expanded, vm, Ks, W, H, sh_degree=3, packed=False)
    assert rec.proj_colors.is_contiguous() and rec.proj_colors.shape == (3, 10, 16, 3)
    rc.sum().backward()
    assert rec.bwd_colors.data_ptr() == rec.proj_colors.data_ptr()  # the same dense copy feeds both passes
    assert torch.all(shs.grad == 3 * 5.0)  # autograd sums the per-camera rows of an expanded input


def test_no_grad_call(rec):
    means, quats, scales, opac, cols, vm, Ks = _scene(N=10, C=2)
    cols.requires_grad_(True)
    with torch.no_grad():
        rc, ra, meta = rendering.rasterization(means, quats, scales, opac, cols, vm, Ks, W, H, sh_degree=3, packed=False)
    assert rc.grad_fn is None and rec.calls == ["projection_fwd", "isect_sorted", "rasterize_fwd"]
    assert meta["colors"].shape == (2, 10, 3)


def test_entries_reject_bad_colors_per_camera_before_any_launch():
    lib = _lib.load()
    n0 = lib.egs_kernel_launch_count()
    fake = ctypes.c_void_p(0x1000)  # non-null pointers that are never touched

    def fwd(K, deg, pc, aa=False):
        args = (1, 10, None, None, None, None, None, K, deg, pc, None, None, 64, 64, 0.3, 0.01, 1e10, 0.0, 16, 4, 4,
                None, None, None, None, None, None, None, None)
        if aa:
            return lib.egs_projection_fwd_antialiased(*args, fake, None)
        return lib.egs_projection_fwd(*args, None)

    def bwd(K, deg, pc):
        return lib.egs_projection_bwd(1, 10, None, None, None, None, K, deg, pc, None, None, 64, 64, 0.3, None, None, None,
                                      None, None, None, None, None, None, None, None)

    def bwd_aa(K, deg, pc):
        return lib.egs_projection_bwd_antialiased(1, 10, None, None, None, None, None, K, deg, pc, None, None, 64, 64, 0.3,
                                                  None, None, None, None, None, None, None, None, None, None, None)

    def bwd_vm(K, deg, pc):
        return lib.egs_projection_bwd_viewmats(1, 10, None, None, None, None, None, K, deg, pc, None, None, 64, 64, 0.3,
                                               None, None, None, None, None, None, None, None, None, None, 0, fake, None, 0,
                                               None)

    for call in (fwd, lambda *a: fwd(*a, aa=True), bwd, bwd_aa, bwd_vm):
        for pc in (2, -1):
            assert call(16, 3, pc) == -1 and f"colors_per_camera={pc}".encode() in lib.egs_last_error_string()
        for K, deg in ((9, 3), (4, 2), (15, 3)):  # per-camera rows too short for the degree
            assert call(K, deg, 1) == -1 and f"K={K} too small".encode() in lib.egs_last_error_string()
    assert lib.egs_kernel_launch_count() == n0
