"""CPU tests of SH degree 4: validation in rendering._check_inputs and rasterization_from_parameters, the arguments the
projection stages pass to the C entries (through a stand-in library that records the calls), and the C entries'
degree / K checks, which run before any launch and need no GPU."""
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


@pytest.mark.parametrize("K", [25, 36])
@pytest.mark.parametrize("per_cam", [False, True])
def test_degree4_shapes_are_accepted(K, per_cam):
    N, C = 5, 2
    cols = torch.zeros(C, N, K, 3) if per_cam else torch.zeros(N, K, 3)
    with pytest.raises(RuntimeError, match="CUDA-only"):  # shape accepted; the CPU tensors are refused next
        _check_inputs(**_base(N, C), colors=cols, sh_degree=4)


@pytest.mark.parametrize("K", [16, 24])
@pytest.mark.parametrize("per_cam", [False, True])
def test_degree4_needs_25_bands(K, per_cam):
    N, C = 5, 2
    cols = torch.zeros(C, N, K, 3) if per_cam else torch.zeros(N, K, 3)
    with pytest.raises(ValueError, match="needs K >= 25"):
        _check_inputs(**_base(N, C), colors=cols, sh_degree=4)


def test_degree5_is_not_implemented():
    with pytest.raises(NotImplementedError, match="sh_degree=5"):
        _check_inputs(**_base(), colors=torch.zeros(5, 36, 3), sh_degree=5)


def test_raw_parameters_stay_at_16_bands():
    N, C = 5, 2
    b = _base(N, C)
    with pytest.raises(ValueError, match="needs K >= 25"):
        rendering.rasterization_from_parameters(b["means"], b["quats"], b["scales"], b["opacities"],
                                                torch.zeros(N, 1, 3), torch.zeros(N, 15, 3), b["viewmats"], b["Ks"],
                                                W, H, sh_degree=4)


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


@pytest.mark.parametrize("K", [25, 36])
@pytest.mark.parametrize("per_cam", [False, True])
@pytest.mark.parametrize("antialiased", [False, True])
def test_stage_calls_pass_degree_K_and_layout(fake_lib, K, per_cam, antialiased):
    N, C = 7, 3
    g = torch.Generator().manual_seed(0)
    means, quats, scales, opac = (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g),
                                  torch.rand(N, 3, generator=g), torch.rand(N, generator=g))
    cols = torch.randn(*((C,) if per_cam else ()), N, K, 3, generator=g)
    vm, Ks = torch.eye(4)[None].repeat(C, 1, 1), torch.eye(3)[None].repeat(C, 1, 1)
    stages.projection_fwd(means, quats, scales, opac, cols, vm, Ks, W, H, 4, antialiased=antialiased)
    name, a = fake_lib.calls[-1]
    assert name == ("egs_projection_fwd_antialiased" if antialiased else "egs_projection_fwd")
    assert a[:2] == (C, N) and a[7:10] == (K, 4, int(per_cam)) and a[6].value == cols.data_ptr()
    radii = torch.ones(C, N, dtype=torch.int32)
    for want_vm, want_ks in ((False, False), (True, False), (False, True), (True, True)):
        out = stages.projection_bwd(means, quats, scales, cols, vm, Ks, W, H, 4, 0.3, radii, torch.zeros(C, N, 3),
                                    torch.zeros(C, N, SPLAT), antialiased_opacities=opac if antialiased else None,
                                    opacities=opac, want_viewmats_grad=want_vm, want_Ks_grad=want_ks)
        name, a = fake_lib.calls[-1]
        assert name == ("egs_projection_bwd_intrinsics" if want_ks else "egs_projection_bwd_viewmats" if want_vm else
                        "egs_projection_bwd_antialiased" if antialiased else "egs_projection_bwd")
        tail = a[6:] if (want_vm or want_ks or antialiased) else a[5:]  # after the opacities argument, if any
        assert tail[0].value == cols.data_ptr() and tail[1:4] == (K, 4, int(per_cam))
        assert out[4].shape == cols.shape and tail[17].value == out[4].data_ptr()
        assert len(out) == 5 + want_vm + want_ks


def test_entries_reject_degree5_and_short_rows_before_any_launch():
    lib = _lib.load()
    n0 = lib.egs_kernel_launch_count()
    fake = ctypes.c_void_p(0x1000)  # non-null pointers that are never touched
    ws = lib.egs_projection_bwd_intrinsics_workspace_bytes(1, 10)

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
                                               None, None, None, None, None, None, None, None, None, None, 0, fake, fake,
                                               ws, None)

    def bwd_ks(K, deg, pc):
        return lib.egs_projection_bwd_intrinsics(1, 10, None, None, None, None, None, K, deg, pc, None, None, 64, 64, 0.3,
                                                 None, None, None, None, None, None, None, None, None, None, 0, None, fake,
                                                 fake, ws, None)

    for call in (fwd, lambda *a: fwd(*a, aa=True), bwd, bwd_aa, bwd_vm, bwd_ks):
        for pc in (0, 1):
            assert call(36, 5, pc) == -1 and b"sh_degree 5 > 4" in lib.egs_last_error_string()
            assert call(24, 4, pc) == -1 and b"K=24 too small" in lib.egs_last_error_string()
            assert call(16, 4, pc) == -1 and b"K=16 too small" in lib.egs_last_error_string()
    # the raw-parameter entries take K = 16: degree 4 is rejected there too
    raw_fwd = lib.egs_projection_fwd_raw(1, 10, None, None, None, None, fake, fake, 4, None, None, 64, 64, 0.3, 0.01,
                                         1e10, 0.0, 16, 4, 4, None, None, None, None, None, None, None, None, None)
    assert raw_fwd == -1 and b"K=16 too small" in lib.egs_last_error_string()
    raw_bwd = lib.egs_projection_bwd_raw(1, 10, None, None, None, None, fake, fake, 4, None, None, 64, 64, 0.3, None,
                                         None, None, None, None, None, None, None, fake, fake, None, None)
    assert raw_bwd == -1 and b"K=16 too small" in lib.egs_last_error_string()
    assert lib.egs_kernel_launch_count() == n0
