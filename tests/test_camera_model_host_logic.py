"""CPU tests of the host logic of rasterization_camera_model(): its signature (rasterization()'s plus camera_model), the
rejection of unknown models, pinhole calls that are exactly rasterization()'s, the camera_model keyword reaching both
projection stages for the other models in every render mode, and the ABI entries rejecting a bad camera_model or bad
sizes before any launch."""
import ctypes
import inspect

import pytest
import torch

from easy_gaussian_splatting_b200 import rasterization, rasterization_camera_model, rendering, stages
from tests.test_depth_host_logic import DepthStages

C, N, W, H = 2, 12, 40, 24


class CameraModelStages(DepthStages):
    def projection_fwd(self, *args, camera_model=None, **kw):
        self.seen.setdefault("fwd_camera_model", []).append(camera_model)
        return super().projection_fwd(*args, **kw)


@pytest.fixture()
def fake(monkeypatch):
    f = CameraModelStages()
    for name in ("projection_fwd", "isect_sorted_async", "isect_tiles", "isect_offset_encode", "rasterize_fwd",
                 "rasterize_fwd_checkpointed", "rasterize_bwd", "rasterize_bwd_segmented", "rasterize_fwd_depth",
                 "rasterize_bwd_depth", "rasterize_fwd_features", "rasterize_bwd_features", "projection_bwd"):
        monkeypatch.setattr(stages, name, getattr(f, name))
    monkeypatch.setattr(stages, "binning_hint", lambda *a, **k: None)
    monkeypatch.setattr(rendering, "_check_inputs", lambda *a, **k: None)  # the real one refuses CPU tensors
    return f


def _inputs(kind="sh"):
    g = torch.Generator().manual_seed(0)
    colors = {"sh": torch.randn(N, 16, 3, generator=g), "feat": torch.rand(N, 5, generator=g)}[kind]
    p = [torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.rand(N, 3, generator=g),
         torch.rand(N, generator=g), colors]
    vm = torch.eye(4)[None].repeat(C, 1, 1).requires_grad_(True)
    K = torch.eye(3)[None].repeat(C, 1, 1).requires_grad_(True)
    return [t.requires_grad_(True) for t in p], vm, K


def test_signature_is_rasterization_plus_camera_model():
    base = list(inspect.signature(rasterization).parameters.values())
    ext = list(inspect.signature(rasterization_camera_model).parameters.values())
    assert ext[:-1] == base
    assert ext[-1].name == "camera_model" and ext[-1].default == "pinhole"
    assert inspect.signature(rasterization_camera_model).return_annotation == inspect.signature(rasterization).return_annotation


@pytest.mark.parametrize("model", ["Pinhole", "orthographic", "equirect", "", None])
def test_unknown_model_raises(fake, model):
    p, vm, K = _inputs()
    with pytest.raises(ValueError, match="'pinhole', 'ortho', 'fisheye'"):
        rasterization_camera_model(*p, vm, K, W, H, sh_degree=3, camera_model=model)
    assert fake.calls == []


def _run(fn, kind, mode, **kw):
    p, vm, K = _inputs(kind)
    rc, ra, meta = fn(*p, vm, K, W, H, sh_degree=3 if kind == "sh" else None, packed=False, render_mode=mode, **kw)
    (rc.sum() + ra.sum()).backward()
    return rc, ra, meta, p, vm, K


@pytest.mark.parametrize("mode", ["RGB", "ED", "RGB+ED"])
def test_pinhole_is_exactly_rasterization(fake, mode):
    a = _run(rasterization, "sh", mode)
    calls, kw = list(fake.calls), fake.seen["proj_kw"]
    fake.calls.clear()
    b = _run(rasterization_camera_model, "sh", mode, camera_model="pinhole")
    assert fake.calls == calls and fake.seen["proj_kw"] == kw and "camera_model" not in kw
    assert fake.seen["fwd_camera_model"] == [None, None]  # no keyword: the pinhole entries
    for x, y in zip(a[:2], b[:2]):
        assert torch.equal(x, y)
    for x, y in zip(a[3] + [a[4], a[5]], b[3] + [b[4], b[5]]):  # (colors.grad is None in "ED")
        assert (x.grad is None and y.grad is None) or torch.equal(x.grad, y.grad)


@pytest.mark.parametrize("kind", ["sh", "feat"])
@pytest.mark.parametrize("mode", ["RGB", "ED", "RGB+ED"])
@pytest.mark.parametrize("model", ["ortho", "fisheye"])
def test_other_models_reach_both_projection_stages(fake, model, mode, kind):
    rc, ra, meta, p, vm, K = _run(rasterization_camera_model, kind, mode, camera_model=model)
    assert fake.seen["fwd_camera_model"] == [model]
    assert fake.seen["proj_kw"]["camera_model"] == model
    assert fake.seen["proj_kw"].get("want_viewmats_grad") and fake.seen["proj_kw"].get("want_Ks_grad")
    assert vm.grad is not None and K.grad is not None
    assert fake.calls[0] == "projection_fwd" and fake.calls[-1] == "projection_bwd"


def test_stages_reject_unknown_model():
    with pytest.raises(ValueError, match="camera_model"):
        stages.projection_fwd(*[None] * 7, 8, 8, None, camera_model="equirect")
    with pytest.raises(ValueError, match="camera_model"):
        stages.projection_bwd(*[None] * 6, 8, 8, None, 0.3, None, None, None, camera_model="equirect")


def test_abi_entries_reject_bad_camera_model_and_sizes_before_any_launch():
    from easy_gaussian_splatting_b200 import _lib
    lib = _lib.load()
    n0 = lib.egs_kernel_launch_count()
    fake = ctypes.c_void_p(0x1000)  # never touched

    def fwd(cm, C_=1, N_=10, K=16, deg=3, cpc=0, width=64):
        return lib.egs_projection_fwd_camera_model(cm, C_, N_, None, None, None, None, None, K, deg, cpc, None, None,
                                                   width, 64, 0.3, 0.01, 1e10, 0.0, 16, 4, 4, None, None, None, None,
                                                   None, None, None, None, None, None)

    def bwd(cm, C_=1, N_=10, K=16, deg=3, cpc=0, v_Ks=None, ws_bytes=0):
        return lib.egs_projection_bwd_camera_model(cm, C_, N_, None, None, None, None, None, K, deg, cpc, None, None, 64,
                                                   64, 0.3, None, None, None, None, None, None, None, None, None, None,
                                                   0, None, v_Ks, fake if v_Ks else None, ws_bytes, None)

    for cm in (0, 3, -1):
        assert fwd(cm) == -1 and b"camera_model" in lib.egs_last_error_string()
        assert bwd(cm) == -1 and b"camera_model" in lib.egs_last_error_string()
    for cm in (1, 2):
        assert fwd(cm, C_=-1) == -1 and b"negative sizes" in lib.egs_last_error_string()
        assert fwd(cm, C_=70000) == -1 and b"65535" in lib.egs_last_error_string()
        assert fwd(cm, deg=5) == -1 and b"sh_degree" in lib.egs_last_error_string()
        assert fwd(cm, K=9) == -1 and b"K=9 too small" in lib.egs_last_error_string()
        assert fwd(cm, cpc=2) == -1 and b"colors_per_camera" in lib.egs_last_error_string()
        assert fwd(cm, width=0) == -1 and b"width/height" in lib.egs_last_error_string()
        assert bwd(cm, N_=-1) == -1 and b"negative sizes" in lib.egs_last_error_string()
        assert bwd(cm, K=9) == -1 and b"K=9 too small" in lib.egs_last_error_string()
        assert bwd(cm, v_Ks=fake, ws_bytes=16) == -1 and b"workspace" in lib.egs_last_error_string()
    assert lib.egs_kernel_launch_count() == n0
