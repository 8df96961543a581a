"""-m gpu: per-camera SH coefficients [C,N,K,3] through rasterization() and the projection stages — the egs::percam
instantiations of the four projection kernels (projection_kernels.cuh) against the oracle, against the shared-coefficient
kernels on equal rows, gradient rows of culled pairs and inactive bands, viewmat gradients, a non-leaf input and the
launch count."""
import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rasterization, stages
from easy_gaussian_splatting_b200.synthetic import loss_weights, make_scene
from oracle import gsplat_oracle as O
from tests.util import PARAMS, cuda_run, image_report, oracle_run, rel_err

pytestmark = pytest.mark.gpu

C1 = dict(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1)
C3 = dict(kind="blob", N=2_000, width=131, height=77, fx=120.0, seed=7, n_views=3)  # ragged image, N % 32 != 0
C70 = dict(kind="blob", N=1500, width=24, height=16, fx=30.0, seed=6, n_views=70)  # more cameras than kMaxCamerasSmem


def _per_camera_colors(sc, K, seed=3, scale=0.2):
    """[C,N,K,3]: the scene's coefficients plus a different offset per camera."""
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    return (sc.colors[None, :, :K] + scale * torch.randn(C, N, K, 3, generator=g)).contiguous()


# ---- 1. oracle parity ------------------------------------------------------------------------------------------------

ORACLE_CASES = (
    [(C1, d, 16, "classic", True, False) for d in range(4)]
    + [(C3, d, 16, "classic", True, False) for d in range(4)]
    + [(C3, d, 9, "classic", True, False) for d in range(3)]
    + [(C1, 2, 9, "classic", True, False), (C3, 3, 16, "antialiased", True, False), (C1, 2, 9, "antialiased", True, False),
       (C3, 3, 16, "classic", False, False), (C3, 1, 9, "classic", False, False), (C3, 3, 16, "classic", True, True),
       (C3, 2, 9, "antialiased", True, True)]
)


@pytest.mark.parametrize("cfg,deg,K,mode,with_bg,packed", ORACLE_CASES,
                         ids=[f"C{c['n_views']}-d{d}-K{K}-{m}-bg{int(b)}-packed{int(p)}" for c, d, K, m, b, p in ORACLE_CASES])
def test_oracle_parity(cfg, deg, K, mode, with_bg, packed):
    sc = make_scene(**cfg)
    sc.colors = _per_camera_colors(sc, K)
    ref = oracle_run(sc, sh_degree=deg, with_bg=with_bg, rasterize_mode=mode)
    out = cuda_run(sc, sh_degree=deg, with_bg=with_bg, rasterize_mode=mode, packed=packed)
    border = ref["counters"]["borderline"]
    rep_c = image_report(out["colors"], ref["colors"], border)
    rep_a = image_report(out["alphas"], ref["alphas"], border)
    vis = ref["meta"]["radii"] > 0
    errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in PARAMS}
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"][vis] if packed else ref["absgrad"])  # packed: [nnz,2]
    print("colours", rep_c, "alphas", rep_a, "grads", errs)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    assert all(e <= 1e-3 for e in errs.values()), errs
    assert out["grads"]["colors"].shape == sc.colors.shape
    # meta["colors"] of visible pairs; the oracle's culled entries hold clamp_min(0 + 0.5, 0), the kernels' hold 0, as for
    # shared coefficients
    m = out["meta"]
    ref_cols = ref["meta"]["colors"].detach()[vis]
    if packed:
        assert m["colors"].shape == (int(vis.sum()), 3)
        torch.testing.assert_close(m["colors"].cpu(), ref_cols, rtol=1e-5, atol=1e-6)
    else:
        assert m["colors"].shape == (sc.viewmats.shape[0], sc.means.shape[0], 3)
        torch.testing.assert_close(m["colors"].cpu()[vis], ref_cols, rtol=1e-5, atol=1e-6)
        assert not m["colors"].cpu()[~vis].any()


def test_no_grad_forward_matches_the_grad_forward():
    sc = make_scene(**C3)
    sc.colors = _per_camera_colors(sc, 16)
    d = sc.to("cuda")
    with torch.no_grad():
        a = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width, sc.height,
                          sh_degree=3, packed=False)
    cols = d.colors.clone().requires_grad_(True)
    b = rasterization(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, sh_degree=3,
                      packed=False)
    assert a[0].grad_fn is None and torch.equal(a[0], b[0].detach()) and torch.equal(a[2]["colors"], b[2]["colors"])


# ---- 2. stage level: equal rows in every camera give the shared path's results -----------------------------------------

def _records(radii, seed):
    C, N = radii.shape
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(C, N, 12, generator=g)
    v[..., 9:11] = v[..., 0:2].abs()
    v[..., 11] = 0.0
    v *= (radii.cpu() > 0)[..., None]
    return v.cuda()


STAGE_CASES = [(K, deg, aa, vg) for K, deg in ((16, 3), (16, 1), (9, 2), (4, 1), (25, 3)) for aa in (False, True)
               for vg in (False, True)]


@pytest.mark.parametrize("K,deg,aa,vg", STAGE_CASES)
def test_stage_equivalence_with_equal_rows(K, deg, aa, vg):
    sc = make_scene(**C3)
    d = sc.to("cuda")
    C = sc.viewmats.shape[0]
    shared = d.colors[:, :K].contiguous() if K <= 16 else torch.cat(
        [d.colors, 0.1 * torch.ones(sc.means.shape[0], K - 16, 3, device="cuda")], 1).contiguous()
    percam = shared[None].expand(C, -1, -1, -1).contiguous()
    kw = dict(antialiased=aa)
    fa = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, shared, d.viewmats, d.Ks, sc.width, sc.height, deg, **kw)
    fb = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, percam, d.viewmats, d.Ks, sc.width, sc.height, deg, **kw)
    vis = fa["radii"] > 0
    for k in fa:  # radii, means2d, depths, conics, colours, splat records, ... bit-identical
        if k == "splats":  # records are written for visible pairs only
            assert torch.equal(fa[k][vis], fb[k][vis]), k
        else:
            assert torch.equal(fa[k], fb[k]), k
    v_splats = _records(fa["radii"], 11)
    extra = torch.randn(C, sc.means.shape[0], 2, device="cuda") * (fa["radii"] > 0)[..., None]
    bkw = dict(want_absgrad=True, antialiased_opacities=d.opacities if aa else None, want_viewmats_grad=vg)
    ba = stages.projection_bwd(d.means, d.quats, d.scales, shared, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3,
                               fa["radii"], fa["colors"], v_splats, extra, **bkw)
    bb = stages.projection_bwd(d.means, d.quats, d.scales, percam, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3,
                               fb["radii"], fb["colors"], v_splats, extra, **bkw)
    for i, name in enumerate(("v_means", "v_quats", "v_scales", "v_opacities")):
        assert torch.equal(ba[i], bb[i]), name
    assert torch.equal(ba[5], bb[5])  # absgrad
    assert bb[4].shape == (C, sc.means.shape[0], K, 3)
    assert rel_err(bb[4].sum(0), ba[4]) <= 1e-6
    if vg:
        assert rel_err(bb[-1], ba[-1]) <= 1e-6  # same terms; only the SH row each camera reads differs in address


# ---- 3. every gradient element written: zeros for culled pairs and inactive bands --------------------------------------

@pytest.mark.parametrize("K,deg", [(16, 1), (16, 3), (9, 0), (9, 2), (4, 1), (25, 3)])
@pytest.mark.parametrize("vg", [False, True])
def test_culled_rows_and_inactive_bands_are_zero(monkeypatch, K, deg, vg):
    sc = make_scene(**C3)
    d = sc.to("cuda")
    cols = _per_camera_colors(sc, min(K, 16)).cuda()
    if K > 16:
        cols = torch.cat([cols, torch.ones(*cols.shape[:2], K - 16, 3, device="cuda")], 2).contiguous()
    f = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, deg)
    monkeypatch.setattr(stages, "_grad_buffer", lambda t: torch.full(t.shape, float("nan"), dtype=t.dtype, device=t.device))
    out = stages.projection_bwd(d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3, f["radii"],
                                f["colors"], _records(f["radii"], 5), want_viewmats_grad=vg)
    v = out[4]
    assert not torch.isnan(v).any()
    culled = f["radii"] <= 0
    assert culled.any() and (~culled).any()
    assert not v[culled].any()
    nb = (deg + 1) ** 2
    assert not v[:, :, nb:].any()
    assert v[~culled][:, :nb].abs().sum() > 0


# ---- 4. viewmat gradients: each camera's own coefficients in the SH direction term -------------------------------------

def _oracle_viewmat_grad(sc, sh_degree, colors, radii, v_splats, aa_opacities=None):
    vm = sc.viewmats.double().requires_grad_(True)
    m, q, s, Ks = sc.means.double(), sc.quats.double(), sc.scales.double(), sc.Ks.double()
    out = O.fully_fused_projection(m, q, s, vm, Ks, sc.width, sc.height, calc_compensations=aa_opacities is not None)
    v = v_splats.double().cpu()
    vis = radii.cpu() > 0
    total = (out[1] * v[..., 0:2] * vis[..., None]).sum() + (out[3] * v[..., 2:5]).sum()
    campos = torch.inverse(vm)[:, :3, 3]
    cols = torch.clamp_min(O.spherical_harmonics(sh_degree, m[None] - campos[:, None], colors.double().cpu(), vis) + 0.5, 0)
    total = total + (cols * v[..., 6:9] * vis[..., None]).sum()
    if aa_opacities is not None:
        total = total + (out[4] * v[..., 5] * aa_opacities.double().cpu()[None]).sum()
    total.backward()
    return vm.grad


def _per_camera_rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return [((a[c] - b[c]).norm() / b[c].norm().clamp_min(1e-30)).item() for c in range(b.shape[0])]


@pytest.mark.parametrize("cfg", [C3, C70], ids=["C3", "C70"])
@pytest.mark.parametrize("K,deg", [(16, 3), (9, 2)])
@pytest.mark.parametrize("aa", [False, True])
def test_stage_viewmat_grad_vs_oracle(cfg, K, deg, aa):
    sc = make_scene(**cfg)
    d = sc.to("cuda")
    cols = _per_camera_colors(sc, K).cuda()
    f = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, deg,
                              antialiased=aa)
    v_splats = _records(f["radii"], 9)
    out = stages.projection_bwd(d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3, f["radii"],
                                f["colors"], v_splats, antialiased_opacities=d.opacities if aa else None,
                                want_viewmats_grad=True)
    ref = _oracle_viewmat_grad(sc, deg, cols, f["radii"], v_splats, aa_opacities=sc.opacities if aa else None)
    rel = _per_camera_rel(out[-1], ref)
    print("per-camera rel err", max(rel))
    assert max(rel) <= 1e-4, rel


@pytest.mark.parametrize("cfg", [C3, C70], ids=["C3", "C70"])
def test_end_to_end_viewmat_grad_vs_oracle(cfg):
    sc = make_scene(**cfg)
    cols = _per_camera_colors(sc, 16)
    C = sc.viewmats.shape[0]
    bg = sc.background[None].expand(C, 3).contiguous()
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    leaves = [t.detach().clone().requires_grad_(True) for t in (sc.means, sc.quats, sc.scales, sc.opacities, cols, sc.viewmats)]
    rc, ra, _ = O.rasterization(*leaves[:5], leaves[5], sc.Ks, sc.width, sc.height, sh_degree=3, packed=False, backgrounds=bg)
    ((rc * Wc).sum() + (ra * Wa).sum()).backward()
    gl = [t.detach().clone().cuda().requires_grad_(True) for t in (sc.means, sc.quats, sc.scales, sc.opacities, cols, sc.viewmats)]
    rc, ra, _ = rasterization(*gl[:5], gl[5], sc.Ks.cuda(), sc.width, sc.height, sh_degree=3, packed=False, backgrounds=bg.cuda())
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    rel = _per_camera_rel(gl[5].grad, leaves[5].grad)
    errs = [rel_err(a.grad.cpu(), b.grad) for a, b in zip(gl[:5], leaves[:5])]
    print("viewmat per-camera rel err", max(rel), "param grads", errs)
    assert max(rel) <= 1e-3, rel
    assert all(e <= 1e-3 for e in errs), errs


# ---- 5. a non-leaf input: shared coefficients plus a per-camera offset -------------------------------------------------

def test_shared_plus_per_camera_offset():
    sc = make_scene(**C3)
    d = sc.to("cuda")
    C = sc.viewmats.shape[0]
    shs = d.colors.clone().requires_grad_(True)
    delta = (0.05 * torch.randn(C, *shs.shape, device="cuda")).requires_grad_(True)
    rc, ra, _ = rasterization(d.means, d.quats, d.scales, d.opacities, shs[None] + delta, d.viewmats, d.Ks, sc.width,
                              sc.height, sh_degree=3, packed=False)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    assert shs.grad is not None and delta.grad is not None and delta.grad.shape == (C, *shs.shape)
    assert delta.grad.abs().sum() > 0
    torch.testing.assert_close(shs.grad, delta.grad.sum(0), rtol=1e-6, atol=1e-7)
    # a stride-0 expand of the shared coefficients renders what the shared coefficients render
    rc2, _, _ = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors[None].expand(C, -1, -1, -1), d.viewmats,
                              d.Ks, sc.width, sc.height, sh_degree=3, packed=False)
    rc3, _, _ = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width, sc.height,
                              sh_degree=3, packed=False)
    assert torch.equal(rc2, rc3)


# ---- 6. launches ----------------------------------------------------------------------------------------------------

def test_same_launch_count_as_shared_coefficients():
    lib = _lib.load()
    sc = make_scene(**C3)
    d = sc.to("cuda")
    C = sc.viewmats.shape[0]

    def count(colors, vm_grad):
        cols = colors.clone().requires_grad_(True)
        vm = d.viewmats.clone().requires_grad_(vm_grad)
        torch.cuda.synchronize()
        n0 = lib.egs_kernel_launch_count()
        rc, ra, _ = rasterization(d.means, d.quats, d.scales, d.opacities, cols, vm, d.Ks, sc.width, sc.height, sh_degree=3,
                                  packed=False)
        (rc.sum() + ra.sum()).backward()
        torch.cuda.synchronize()
        return lib.egs_kernel_launch_count() - n0

    for vm_grad in (False, True):
        count(d.colors, vm_grad)  # warm the binning size hints of this shape
        shared = count(d.colors, vm_grad)
        percam = count(d.colors[None].expand(C, -1, -1, -1).contiguous(), vm_grad)
        assert shared == percam, (vm_grad, shared, percam)
