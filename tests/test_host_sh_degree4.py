"""CPU tests: the degree-4 SH math of csrc/egs_math.cuh (sh_basis4, its VJP, sh4_color_fwd / sh4_color_bwd) with the
projection VJP, compiled for the host by tests/host_harness/sh4_harness.cpp, against fp64 autograd through the
degree-4 reference (tests/sh_degree4_reference.py): colours, coefficient gradients, v_means, v_viewmats and v_Ks."""
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from oracle import gsplat_oracle as O
from tests import host_harness as hh
from tests.host_harness import sh4
from tests.sh_degree4_reference import sh_colors4

BLOB = dict(kind="blob", N=3000, width=256, height=256, fx=274.5, seed=0, n_views=2)
OUTDOOR = dict(kind="outdoor", N=5000, width=979, height=546, fx=581.0, seed=2, n_views=2)
CLAMP = dict(kind="blob", N=3000, width=33, height=17, fx=60.0, seed=4, n_views=1)  # fov clamp active in x and y


def _coeffs(sc, K, per_cam, seed):
    """The scene's 16 bands, random band-4 rows and (K > 25) random rows past band 4; DC shifted so that a good share
    of the channels is clipped by clamp_min(+0.5, 0)."""
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    base = torch.cat([sc.colors, 0.3 * torch.randn(N, K - 16, 3, generator=g)], 1)
    base[:, 0] -= 1.2
    if per_cam:
        return (base[None] + 0.2 * torch.randn(C, N, K, 3, generator=g)).contiguous()
    return base.contiguous()


def _run(cfg, K, per_cam, aa, seed=7):
    sc = make_scene(**cfg)
    shs = _coeffs(sc, K, per_cam, seed)
    V, N = sc.viewmats.shape[0], sc.means.shape[0]
    radii = hh.projection_fwd(sc, 3)["radii"]
    vis = torch.from_numpy(radii > 0)
    visf = vis[..., None].double()
    g = torch.Generator().manual_seed(seed + 1)
    v_m2 = torch.randn(V, N, 2, generator=g, dtype=torch.float64)
    v_con = torch.randn(V, N, 3, generator=g, dtype=torch.float64)
    v_col = torch.randn(V, N, 3, generator=g, dtype=torch.float64)
    v_comp = torch.randn(V, N, generator=g, dtype=torch.float64) if aa else None
    m = sc.means.double().requires_grad_(True)
    vm = sc.viewmats.double().requires_grad_(True)
    Ks = sc.Ks.double().requires_grad_(True)
    sd = shs.double().requires_grad_(True)
    out = O.fully_fused_projection(m, sc.quats.double(), sc.scales.double(), vm, Ks, sc.width, sc.height,
                                   calc_compensations=aa)
    cols = sh_colors4(m, vm, sd, torch.from_numpy(radii))
    total = (out[1] * v_m2 * visf).sum() + (out[3] * v_con * visf).sum() + (cols * v_col * visf).sum()
    if aa:
        total = total + (out[4] * v_comp * vis.double()).sum()
    total.backward()
    got = sh4.sh4_grads(sc, shs, radii, v_m2.float(), v_con.float(), v_col.float(),
                        v_comps=None if v_comp is None else v_comp.float())
    ref = dict(colors=torch.where(vis[..., None], cols.detach(), torch.zeros((), dtype=torch.float64)), v_sh=sd.grad,
               v_means=m.grad, v_viewmats=vm.grad, v_Ks=Ks.grad)
    return {k: torch.from_numpy(v).double() for k, v in got.items()}, ref, vis


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


CASES = [(BLOB, 25, False, False), (BLOB, 25, True, False), (BLOB, 36, False, False), (BLOB, 36, True, True),
         (BLOB, 25, False, True), (OUTDOOR, 25, False, False), (CLAMP, 25, False, False), (CLAMP, 25, True, True)]


@pytest.mark.parametrize("cfg,K,per_cam,aa", CASES,
                         ids=[f"{c['kind']}{c['width']}-K{K}-pc{int(p)}-aa{int(a)}" for c, K, p, a in CASES])
def test_degree4_math_vs_fp64_autograd(cfg, K, per_cam, aa):
    got, ref, vis = _run(cfg, K, per_cam, aa)
    assert int(vis.sum()) > 100
    clipped = (ref["colors"] == 0) & vis[..., None]
    assert int(clipped.sum()) > 20  # clamp_min(+0.5, 0) clips channels of visible pairs
    assert _rel(got["colors"], ref["colors"]) <= 2e-5
    assert _rel(got["v_sh"], ref["v_sh"]) <= 2e-5
    assert _rel(got["v_means"], ref["v_means"]) <= 2e-5
    for c in range(vis.shape[0]):  # every camera's gradient must hold on its own
        assert _rel(got["v_viewmats"][c], ref["v_viewmats"][c]) <= 2e-5, c
        assert _rel(got["v_Ks"][c], ref["v_Ks"][c]) <= 2e-5, c
    # bands past 4 and rows nobody (per camera: that camera) sees get exactly 0
    assert torch.all(got["v_sh"][..., 25:, :] == 0)
    seen = vis if per_cam else vis.any(0)
    assert torch.all(got["v_sh"][~seen] == 0) and torch.all(ref["v_sh"][~seen] == 0)
    # band 4 takes part (channels that clamp_min clips get no gradient in any band)
    band4 = got["v_sh"][seen][:, 16:25]
    assert (band4 != 0).double().mean().item() > 0.3


def test_zero_band4_adds_nothing():
    """With zero band-4 rows the degree-4 math gives the degree-3 colours: the same bands, the same order."""
    sc = make_scene(**BLOB)
    shs = _coeffs(sc, 25, False, 3)
    shs[:, 16:] = 0
    radii = hh.projection_fwd(sc, 3)["radii"]
    V, N = radii.shape
    z2, z3 = torch.zeros(V, N, 2), torch.zeros(V, N, 3)
    got = sh4.sh4_grads(sc, shs, radii, z2, z3, z3)
    sc.colors = shs[:, :16].contiguous()
    ref = hh.projection_fwd(sc, 3)
    vis = radii > 0
    assert (got["colors"][vis] == ref["colors"][vis]).all()
