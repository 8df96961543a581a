"""CPU tests: the view-matrix gradient math of csrc/egs_math.cuh (project_bwd / sh_color_bwd with a camera gradient and
viewmat_grad_finalize), compiled for the host by tests/host_harness/viewmat_harness.cpp, against fp64 autograd through
the oracle's projection and SH colours with campos = inverse(viewmats)[:, :3, 3], as gsplat 1.0.0 computes them."""
import numpy as np
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from oracle import gsplat_oracle as O
from tests import host_harness as hh
from tests.host_harness import viewmat as hv

CASES = [
    dict(kind="blob", N=6000, width=256, height=256, fx=274.5, seed=0, n_views=2),
    dict(kind="outdoor", N=40_000, width=979, height=546, fx=581.0, seed=2, n_views=2),
    dict(kind="object", N=20_000, width=800, height=800, fx=1111.11, seed=1, n_views=1),
    dict(kind="blob", N=3000, width=33, height=17, fx=15.0, seed=4, n_views=1),  # wide fov: clamp active
]


def _reference(sc, deg, antialiased, seed):
    """fp64 autograd of a random linear functional of means2d, conics, colours (and compensations) w.r.t. viewmats,
    and the same cotangents in fp32 for the harness."""
    V, N = sc.viewmats.shape[0], sc.means.shape[0]
    h = hh.projection_fwd(sc, max(deg, 0))
    vm = sc.viewmats.double().requires_grad_(True)
    m, q, s, Ks = sc.means.double(), sc.quats.double(), sc.scales.double(), sc.Ks.double()
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
    if deg >= 0:
        campos = torch.inverse(vm)[:, :3, 3]
        cols = torch.clamp_min(O.spherical_harmonics(deg, m[None] - campos[:, None],
                                                     sc.colors.double()[None].expand(V, -1, -1, -1), vis) + 0.5, 0)
        total = total + (cols * v_col * visf).sum()
    if antialiased:
        total = total + (out[4] * v_comp * vis.double()).sum()
    total.backward()
    got = hv.viewmat_grad(sc, deg, h["radii"], h["colors"], v_m2.float(), v_con.float(), v_col.float(),
                          v_comps=None if v_comp is None else v_comp.float())
    return torch.from_numpy(got).double(), vm.grad


@pytest.mark.parametrize("cfg,deg,aa", [
    (CASES[0], 3, False), (CASES[0], 2, False), (CASES[0], 1, False), (CASES[0], 0, False), (CASES[0], -1, False),
    (CASES[1], 3, False), (CASES[2], 3, False), (CASES[3], 3, False), (CASES[3], -1, False),
    (CASES[0], 3, True), (CASES[3], 1, True),
])
def test_viewmat_grad_vs_fp64_autograd(cfg, deg, aa):
    cfg = dict(cfg)
    cfg["N"] = min(cfg["N"], 5000)
    sc = make_scene(**cfg)
    got, ref = _reference(sc, deg, aa, seed=7)
    for c in range(ref.shape[0]):  # per camera: every camera's gradient must hold on its own
        rel = ((got[c] - ref[c]).norm() / ref[c].norm().clamp_min(1e-30)).item()
        assert rel <= 2e-5, (c, rel)
    bottom = got[:, 3].abs().max().item()
    if deg >= 1:
        assert bottom > 0.0 and ref[:, 3].abs().max().item() > 0.0  # the SH path reaches the bottom row
    else:
        assert bottom == 0.0  # without view-dependent colour, only the top 3x4 block carries gradient


def test_viewmat_grad_two_cameras_are_independent():
    """C = 2: each camera's gradient is that of the single-camera call with the same cotangents."""
    sc = make_scene(kind="blob", N=3000, width=256, height=256, fx=274.5, seed=3, n_views=2)
    got, ref = _reference(sc, 3, False, seed=11)
    assert got.shape == (2, 4, 4)
    for c in range(2):
        rel = ((got[c] - ref[c]).norm() / ref[c].norm()).item()
        assert rel <= 2e-5, (c, rel)
    assert not torch.allclose(got[0], got[1])
