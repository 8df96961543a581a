"""CPU tests: the intrinsics gradient math of csrc/egs_math.cuh (project_bwd with v_K, ks_grad_finalize), compiled for
the host by tests/host_harness/intrinsics_harness.cpp, against fp64 autograd w.r.t. Ks through the oracle's projection
and SH colours."""
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from oracle import gsplat_oracle as O
from tests import host_harness as hh
from tests.host_harness import intrinsics as hi

CASES = [
    dict(kind="blob", N=6000, width=256, height=256, fx=274.5, seed=0, n_views=2),
    dict(kind="outdoor", N=40_000, width=979, height=546, fx=581.0, seed=2, n_views=2),
    dict(kind="object", N=20_000, width=800, height=800, fx=1111.11, seed=1, n_views=1),
    dict(kind="blob", N=3000, width=33, height=17, fx=15.0, seed=4, n_views=1),  # wide fov
    dict(kind="blob", N=3000, width=33, height=17, fx=60.0, seed=4, n_views=1),  # fov clamp active in x and y
]
NONZERO = torch.zeros(3, 3, dtype=torch.bool)
NONZERO[0, 0] = NONZERO[1, 1] = NONZERO[0, 2] = NONZERO[1, 2] = True  # fx, fy, cx, cy


def _reference(sc, deg, antialiased, seed):
    """fp64 autograd of a random linear functional of means2d, conics, colours (and compensations) w.r.t. Ks, and the
    same cotangents in fp32 for the harness."""
    V, N = sc.viewmats.shape[0], sc.means.shape[0]
    h = hh.projection_fwd(sc, max(deg, 0))
    Ks = sc.Ks.double().requires_grad_(True)
    m, q, s, vm = sc.means.double(), sc.quats.double(), sc.scales.double(), sc.viewmats.double()
    out = O.fully_fused_projection(m, q, s, vm, Ks, sc.width, sc.height, calc_compensations=antialiased)
    m2, con = out[1], out[3]
    vis = torch.from_numpy(h["radii"] > 0)
    visf = vis[..., None].double()
    g = torch.Generator().manual_seed(seed)
    v_m2 = torch.randn(V, N, 2, generator=g, dtype=torch.float64)
    v_con = torch.randn(V, N, 3, generator=g, dtype=torch.float64)
    v_col = torch.randn(V, N, 3, generator=g, dtype=torch.float64)
    v_comp = torch.randn(V, N, generator=g, dtype=torch.float64) if antialiased else None
    total = (m2 * v_m2 * visf).sum() + (con * v_con * visf).sum()
    if deg >= 0:  # the SH colours do not read Ks: their cotangents must not leak into it
        campos = torch.inverse(vm)[:, :3, 3]
        cols = torch.clamp_min(O.spherical_harmonics(deg, m[None] - campos[:, None],
                                                     sc.colors.double()[None].expand(V, -1, -1, -1), vis) + 0.5, 0)
        total = total + (cols * v_col * visf).sum()
    if antialiased:
        total = total + (out[4] * v_comp * vis.double()).sum()
    total.backward()
    got = hi.intrinsics_grad(sc, deg, h["radii"], h["colors"], v_m2.float(), v_con.float(), v_col.float(),
                             v_comps=None if v_comp is None else v_comp.float())
    return torch.from_numpy(got).double(), Ks.grad, h


def _check(got, ref):
    for c in range(ref.shape[0]):  # per camera: every camera's gradient must hold on its own
        rel = ((got[c] - ref[c]).norm() / ref[c].norm().clamp_min(1e-30)).item()
        assert rel <= 2e-5, (c, rel)
    assert torch.all(got[:, ~NONZERO] == 0.0)  # skew and last row: exactly 0
    assert torch.all(ref[:, ~NONZERO] == 0.0)


@pytest.mark.parametrize("cfg,deg,aa", [
    (CASES[0], 3, False), (CASES[0], 2, False), (CASES[0], 1, False), (CASES[0], 0, False), (CASES[0], -1, False),
    (CASES[1], 3, False), (CASES[2], 3, False), (CASES[3], 3, False), (CASES[3], -1, False),
    (CASES[0], 3, True), (CASES[3], 1, True), (CASES[4], 3, False), (CASES[4], -1, False), (CASES[4], 2, True),
])
def test_intrinsics_grad_vs_fp64_autograd(cfg, deg, aa):
    cfg = dict(cfg)
    cfg["N"] = min(cfg["N"], 5000)
    sc = make_scene(**cfg)
    got, ref, _ = _reference(sc, deg, aa, seed=7)
    _check(got, ref)
    assert torch.all(got[:, NONZERO] != 0.0)


def test_clamp_case_has_visible_gaussians_past_the_clamp():
    """CASES[4] puts visible Gaussians outside 1.3 x the half fov in x and in y, where J02 / J12 stop depending on
    fx / fy."""
    sc = make_scene(**CASES[4])
    h = hh.projection_fwd(sc, 3)
    vm, K = sc.viewmats[0], sc.Ks[0]
    pc = sc.means @ vm[:3, :3].T + vm[:3, 3]
    vis = torch.from_numpy(h["radii"][0] > 0)
    for axis, size in ((0, sc.width), (1, sc.height)):
        lim = 1.3 * 0.5 * size / K[axis, axis]
        assert int((((pc[:, axis] / pc[:, 2]).abs() > lim) & vis).sum()) > 0, axis


def test_intrinsics_grad_two_cameras_are_independent():
    """C = 2: each camera's gradient is that of the single-camera call with the same cotangents."""
    sc = make_scene(kind="blob", N=3000, width=256, height=256, fx=274.5, seed=3, n_views=2)
    got, ref, _ = _reference(sc, 3, False, seed=11)
    assert got.shape == (2, 3, 3)
    _check(got, ref)
    assert not torch.allclose(got[0], got[1])


def test_principal_point_gradient_is_the_sum_of_the_means2d_cotangents():
    """v_cx / v_cy take nothing but the means2d cotangents: with only those, they are their sums over visible pairs."""
    sc = make_scene(kind="blob", N=3000, width=256, height=256, fx=274.5, seed=5, n_views=2)
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    h = hh.projection_fwd(sc, 3)
    vis = torch.from_numpy(h["radii"] > 0)
    v_m2 = torch.randn(C, N, 2, generator=torch.Generator().manual_seed(2)) * vis[..., None]
    zero3 = torch.zeros(C, N, 3)
    got = torch.from_numpy(hi.intrinsics_grad(sc, 3, h["radii"], h["colors"], v_m2, zero3, zero3)).double()
    expect = v_m2.double().sum(dim=1)
    assert torch.allclose(got[:, 0, 2], expect[:, 0], rtol=1e-5, atol=1e-4)
    assert torch.allclose(got[:, 1, 2], expect[:, 1], rtol=1e-5, atol=1e-4)
