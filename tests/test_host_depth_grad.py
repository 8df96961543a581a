"""CPU tests: the depth cotangent of csrc/egs_math.cuh (project_bwd's v_depth, which the egs::depth projection backward
kernels take from gradient-record slot 11), compiled for the host by tests/host_harness/depth_harness.cpp, against fp64
autograd through the oracle's projection: v_means, v_viewmats and v_Ks, classic and antialiased, fov clamp included."""
import numpy as np
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from oracle import gsplat_oracle as O
from tests import host_harness as hh
from tests.host_harness import depth as hd

CASES = [
    dict(kind="blob", N=5000, width=256, height=256, fx=274.5, seed=0, n_views=2),
    dict(kind="outdoor", N=5000, width=979, height=546, fx=581.0, seed=2, n_views=2),
    dict(kind="blob", N=3000, width=33, height=17, fx=60.0, seed=4, n_views=1),  # fov clamp active in x and y
]


def _cotangents(sc, antialiased, seed, with_depth=True):
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    v_m2 = torch.randn(C, N, 2, generator=g, dtype=torch.float64)
    v_d = torch.randn(C, N, generator=g, dtype=torch.float64) * (1.0 if with_depth else 0.0)
    v_con = torch.randn(C, N, 3, generator=g, dtype=torch.float64)
    v_comp = torch.randn(C, N, generator=g, dtype=torch.float64) if antialiased else None
    return v_m2, v_d, v_con, v_comp


def _reference(sc, antialiased, seed):
    """fp64 autograd of a random linear functional of means2d, depths, conics (and compensations) of the visible pairs
    w.r.t. means, viewmats and Ks; the harness's answer for the same cotangents in fp32."""
    h = hh.projection_fwd(sc, 0)
    vis = torch.from_numpy(h["radii"] > 0)
    m = sc.means.double().requires_grad_(True)
    vm = sc.viewmats.double().requires_grad_(True)
    Ks = sc.Ks.double().requires_grad_(True)
    out = O.fully_fused_projection(m, sc.quats.double(), sc.scales.double(), vm, Ks, sc.width, sc.height,
                                   calc_compensations=antialiased)
    v_m2, v_d, v_con, v_comp = _cotangents(sc, antialiased, seed)
    visd = vis.double()
    total = (out[1] * v_m2 * visd[..., None]).sum() + (out[2] * v_d * visd).sum() + (out[3] * v_con * visd[..., None]).sum()
    if antialiased:
        total = total + (out[4] * v_comp * visd).sum()
    total.backward()
    got = hd.depth_grad(sc, h["radii"], v_m2.float(), v_d.float(), v_con.float(),
                        v_comps=None if v_comp is None else v_comp.float())
    return [torch.from_numpy(x).double() for x in got], (m.grad, vm.grad, Ks.grad), h


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("cfg,aa", [(CASES[0], False), (CASES[0], True), (CASES[1], False), (CASES[2], False),
                                    (CASES[2], True)])
def test_depth_cotangent_vs_fp64_autograd(cfg, aa):
    sc = make_scene(**cfg)
    (g_means, g_vm, g_ks), (r_means, r_vm, r_ks), _ = _reference(sc, aa, seed=3)
    assert _rel(g_means, r_means) <= 2e-5
    for c in range(r_vm.shape[0]):  # per camera
        assert _rel(g_vm[c], r_vm[c]) <= 2e-5, c
        assert _rel(g_ks[c], r_ks[c]) <= 2e-5, c


def test_clamp_case_has_visible_gaussians_past_the_clamp():
    sc = make_scene(**CASES[2])
    h = hh.projection_fwd(sc, 0)
    vm, K = sc.viewmats[0], sc.Ks[0]
    pc = sc.means @ vm[:3, :3].T + vm[:3, 3]
    vis = torch.from_numpy(h["radii"][0] > 0)
    for axis, size in ((0, sc.width), (1, sc.height)):
        lim = 1.3 * 0.5 * size / K[axis, axis]
        assert int((((pc[:, axis] / pc[:, 2]).abs() > lim) & vis).sum()) > 0, axis


@pytest.mark.parametrize("aa", [False, True])
def test_depth_cotangent_is_z_through_row_2(aa):
    """The depth cotangent alone: v_means = sum_c v_d R_c[2,:], v_viewmats[c] row 2 = sum_n v_d (m, 1), nothing else, and
    v_Ks is bit-identical to the call without it (z does not depend on K)."""
    sc = make_scene(**CASES[0])
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    h = hh.projection_fwd(sc, 0)
    vis = torch.from_numpy(h["radii"] > 0).double()
    v_m2, v_d, v_con, v_comp = _cotangents(sc, aa, seed=5)
    comps = None if v_comp is None else v_comp.float()
    with_d = hd.depth_grad(sc, h["radii"], v_m2.float(), v_d.float(), v_con.float(), v_comps=comps)
    without = hd.depth_grad(sc, h["radii"], v_m2.float(), torch.zeros(C, N), v_con.float(), v_comps=comps)
    assert np.array_equal(with_d[2], without[2])
    vd = v_d.float().double() * vis
    R = sc.viewmats[:, :3, :3].double()
    expect_means = torch.einsum("cn,cj->nj", vd, R[:, 2, :])
    d_means = torch.from_numpy(with_d[0]).double() - torch.from_numpy(without[0]).double()
    assert torch.allclose(d_means, expect_means, rtol=1e-4, atol=1e-4 * expect_means.abs().max().item())
    d_vm = torch.from_numpy(with_d[1]).double() - torch.from_numpy(without[1]).double()
    expect_row2 = torch.cat([vd @ sc.means.double(), vd.sum(1, keepdim=True)], 1)
    assert torch.allclose(d_vm[:, 2, :], expect_row2, rtol=1e-4, atol=1e-4 * expect_row2.abs().max().item())
    assert torch.allclose(d_vm[:, [0, 1, 3], :], torch.zeros(C, 3, 4, dtype=torch.float64),
                          atol=1e-4 * expect_row2.abs().max().item())
