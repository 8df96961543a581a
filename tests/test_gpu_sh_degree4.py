"""-m gpu: SH degree 4 ([N,K,3] / [C,N,K,3], K >= 25) through rasterization() and the projection stages — the
projection_fwd_sh4_kernel / projection_bwd_sh4_kernel instantiations against the degree-4 reference
(tests/sh_degree4_reference.py), camera gradients against fp64 autograd, degree 4 with zero band-4 rows against
degree 3, gradient buffers written once, and the launch count."""
import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rasterization, stages
from easy_gaussian_splatting_b200.synthetic import loss_weights, make_scene
from oracle import gsplat_oracle as O
from tests.sh_degree4_reference import rasterization4, sh_basis4, sh_colors4
from tests.util import image_report, rel_err

pytestmark = pytest.mark.gpu

S1 = dict(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1)
S3 = dict(kind="blob", N=2_001, width=131, height=77, fx=120.0, seed=7, n_views=3)  # N % 4 != 0, ragged image
S70 = dict(kind="blob", N=1_501, width=24, height=16, fx=30.0, seed=6, n_views=70)  # more cameras than kMaxCamerasSmem
GEOM = ("means", "quats", "scales", "opacities")


def _coeffs(sc, K, per_cam, seed=3):
    """The scene's 16 bands, random band-4 rows and random rows past band 4 (which must not matter); per camera, a
    different offset per camera."""
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    base = torch.cat([sc.colors, 0.15 * torch.randn(N, 9, 3, generator=g), torch.randn(N, K - 25, 3, generator=g)], 1)
    if per_cam:
        return (base[None] + 0.1 * torch.randn(C, N, K, 3, generator=g)).contiguous()
    return base.contiguous()


# ---- 1. parity with the degree-4 reference --------------------------------------------------------------------------

def _ref_run(sc, shs, mode, with_bg):
    leaves = {k: getattr(sc, k).detach().clone().requires_grad_(True) for k in GEOM}
    leaves["colors"] = shs.detach().clone().requires_grad_(True)
    C = sc.viewmats.shape[0]
    bg = sc.background[None].expand(C, 3).contiguous() if with_bg else None
    counters = {}
    rc, ra, meta = rasterization4(*[leaves[k] for k in (*GEOM, "colors")], sc.viewmats, sc.Ks, sc.width, sc.height,
                                  rasterize_mode=mode, packed=False, absgrad=True, backgrounds=bg, counters=counters)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc).sum() + (ra * Wa).sum()).backward()
    return dict(colors=rc.detach(), alphas=ra.detach(), border=counters["borderline"], radii=meta["radii"],
                grads={k: v.grad for k, v in leaves.items()}, absgrad=meta["means2d"].absgrad)


def _cuda_run(sc, shs, mode, with_bg, packed, offset):
    d = sc.to("cuda")
    leaves = {k: getattr(d, k).detach().clone().requires_grad_(True) for k in GEOM}
    if offset:  # a coefficient tensor with a storage offset of one float
        buf = torch.zeros(shs.numel() + 1, device="cuda")
        buf[1:] = shs.reshape(-1).cuda()
        buf.requires_grad_(True)
        cols = buf[1:].view(shs.shape)
        assert cols.storage_offset() == 1
    else:
        cols = shs.cuda().requires_grad_(True)
    C = sc.viewmats.shape[0]
    bg = d.background[None].expand(C, 3).contiguous() if with_bg else None
    rc, ra, meta = rasterization(*[leaves[k] for k in GEOM], cols, d.viewmats, d.Ks, sc.width, sc.height, sh_degree=4,
                                 packed=packed, absgrad=True, backgrounds=bg, rasterize_mode=mode)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    grads = {k: v.grad.cpu() for k, v in leaves.items()}
    if offset:
        assert buf.grad[0].item() == 0.0
        grads["colors"] = buf.grad[1:].view(shs.shape).cpu()
    else:
        grads["colors"] = cols.grad.cpu()
    return dict(colors=rc.detach().cpu(), alphas=ra.detach().cpu(), grads=grads, meta=meta,
                absgrad=meta["means2d"].absgrad.detach().cpu())


PARITY = [  # (scene, K, per-camera, mode, background, packed, storage offset)
    (S1, 25, False, "classic", True, False, False),
    (S1, 25, False, "antialiased", False, False, False),
    (S1, 36, True, "classic", True, False, False),
    (S3, 25, True, "classic", True, False, False),
    (S3, 25, True, "antialiased", False, True, True),
    (S3, 36, False, "antialiased", True, True, False),
    (S3, 25, False, "classic", False, False, True),
    (S70, 25, False, "classic", True, False, False),
    (S70, 25, True, "antialiased", True, False, False),
    (S70, 36, True, "classic", False, True, False),
]


@pytest.mark.parametrize("cfg,K,per_cam,mode,with_bg,packed,offset", PARITY,
                         ids=[f"C{c['n_views']}-K{K}-pc{int(p)}-{m}-bg{int(b)}-packed{int(pk)}-off{int(o)}"
                              for c, K, p, m, b, pk, o in PARITY])
def test_oracle_parity(cfg, K, per_cam, mode, with_bg, packed, offset):
    sc = make_scene(**cfg)
    shs = _coeffs(sc, K, per_cam)
    ref = _ref_run(sc, shs, mode, with_bg)
    out = _cuda_run(sc, shs, mode, with_bg, packed, offset)
    rep_c = image_report(out["colors"], ref["colors"], ref["border"])
    rep_a = image_report(out["alphas"], ref["alphas"], ref["border"])
    vis = ref["radii"] > 0
    errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in ref["grads"]}
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"][vis] if packed else ref["absgrad"])
    print("colours", rep_c, "alphas", rep_a, "grads", errs)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    assert all(e <= 1e-3 for e in errs.values()), errs
    g = out["grads"]["colors"]
    assert g.shape == shs.shape and not g[..., 25:, :].any()  # bands past 4
    assert g[..., 16:25, :].abs().sum() > 0  # band 4 is trained


def test_no_grad_forward_matches_the_grad_forward():
    sc = make_scene(**S3)
    d = sc.to("cuda")
    shs = _coeffs(sc, 25, True).cuda()
    with torch.no_grad():
        a = rasterization(d.means, d.quats, d.scales, d.opacities, shs, d.viewmats, d.Ks, sc.width, sc.height,
                          sh_degree=4, packed=False)
    cols = shs.clone().requires_grad_(True)
    b = rasterization(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, sh_degree=4,
                      packed=False)
    assert a[0].grad_fn is None and torch.equal(a[0], b[0].detach()) and torch.equal(a[2]["colors"], b[2]["colors"])


# ---- 2. camera gradients against fp64 autograd ------------------------------------------------------------------------

def _records(radii, seed):
    """Random gradient records {v_x,v_y,v_ca,v_cb | v_cc,v_opacity,v_r,v_g | v_b,|v_x|,|v_y|,0}, zero where culled."""
    C, N = radii.shape
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(C, N, 12, generator=g)
    v[..., 9:11] = v[..., 0:2].abs()
    v[..., 11] = 0.0
    v *= (radii.cpu() > 0)[..., None]
    return v.cuda()


def _oracle_camera_grads(sc, shs, radii, v_splats, v_extra, aa_opacities):
    vm = sc.viewmats.double().requires_grad_(True)
    Ks = sc.Ks.double().requires_grad_(True)
    m, q, s = sc.means.double(), sc.quats.double(), sc.scales.double()
    out = O.fully_fused_projection(m, q, s, vm, Ks, sc.width, sc.height, calc_compensations=aa_opacities is not None)
    v = v_splats.double().cpu()
    vis = (radii.cpu() > 0)[..., None]
    cols = sh_colors4(m, vm, shs.double(), radii.cpu())
    total = ((out[1] * (v[..., 0:2] + v_extra.double().cpu()) * vis).sum() + (out[3] * v[..., 2:5]).sum()
             + (cols * v[..., 6:9] * vis).sum())
    if aa_opacities is not None:
        total = total + (out[4] * v[..., 5] * aa_opacities.double().cpu()[None]).sum()
    total.backward()
    return vm.grad, Ks.grad


def _per_camera_rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return [((a[c] - b[c]).norm() / b[c].norm().clamp_min(1e-30)).item() for c in range(b.shape[0])]


CAM_CASES = [(S3, 25, False, False), (S3, 25, True, True), (S3, 36, False, True), (S70, 25, False, False),
             (S70, 25, True, True)]


@pytest.mark.parametrize("cfg,K,per_cam,aa", CAM_CASES,
                         ids=[f"C{c['n_views']}-K{K}-pc{int(p)}-aa{int(a)}" for c, K, p, a in CAM_CASES])
def test_camera_gradients_vs_fp64(cfg, K, per_cam, aa):
    sc = make_scene(**cfg)
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    d = sc.to("cuda")
    shs = _coeffs(sc, K, per_cam)
    cols = shs.cuda()
    proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, 4,
                                 antialiased=aa)
    v_splats = _records(proj["radii"], 3)
    v_extra = 0.1 * torch.randn(C, N, 2, generator=torch.Generator().manual_seed(4)).cuda()
    args = (d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, 4, 0.3, proj["radii"],
            proj["colors"], v_splats, v_extra)
    kw = dict(want_absgrad=True, antialiased_opacities=d.opacities if aa else None)
    old = stages.projection_bwd(*args, **kw)
    vm_only = stages.projection_bwd(*args, **kw, want_viewmats_grad=True)
    both = stages.projection_bwd(*args, **kw, want_viewmats_grad=True, want_Ks_grad=True)
    again = stages.projection_bwd(*args, **kw, want_viewmats_grad=True, want_Ks_grad=True)
    for i, a in enumerate(old):  # v_means, v_quats, v_scales, v_opacities, v_colors, absgrad
        assert torch.equal(a, vm_only[i]) and torch.equal(a, both[i]), i
    assert torch.equal(both[-2], vm_only[-1])  # v_viewmats with or without v_Ks
    assert torch.equal(both[-2], again[-2]) and torch.equal(both[-1], again[-1])  # deterministic
    ref_vm, ref_ks = _oracle_camera_grads(sc, shs, proj["radii"], v_splats, v_extra, d.opacities if aa else None)
    rel_vm, rel_ks = _per_camera_rel(both[-2], ref_vm), _per_camera_rel(both[-1], ref_ks)
    print("per-camera rel err: viewmats", max(rel_vm), "Ks", max(rel_ks))
    assert max(rel_vm) <= 1e-4, rel_vm
    assert max(rel_ks) <= 1e-4, rel_ks


def test_end_to_end_camera_gradients():
    """viewmats.grad and Ks.grad through rasterization() at degree 4, per-camera coefficients, against fp64 autograd
    through the reference."""
    sc = make_scene(**S3)
    C = sc.viewmats.shape[0]
    shs = _coeffs(sc, 25, True)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    bg = sc.background[None].expand(C, 3).contiguous()

    def run(dev, dt):
        p = [getattr(sc, k).detach().to(dev, dt) for k in GEOM] + [shs.to(dev, dt)]
        vm = sc.viewmats.detach().to(dev, dt).requires_grad_(True)
        Ks = sc.Ks.detach().to(dev, dt).requires_grad_(True)
        f = rasterization if dev == "cuda" else rasterization4
        kw = dict(sh_degree=4) if dev == "cuda" else {}
        rc, ra, _ = f(*p, vm, Ks, sc.width, sc.height, packed=False, backgrounds=bg.to(dev, dt), **kw)
        ((rc * Wc.to(dev, dt)).sum() + (ra * Wa.to(dev, dt)).sum()).backward()
        return vm.grad.cpu(), Ks.grad.cpu()

    got, ref = run("cuda", torch.float32), run("cpu", torch.float64)
    rel_vm, rel_ks = _per_camera_rel(got[0], ref[0]), _per_camera_rel(got[1], ref[1])
    print("end-to-end per-camera rel err: viewmats", max(rel_vm), "Ks", max(rel_ks))
    assert max(rel_vm) <= 1e-3 and max(rel_ks) <= 1e-3, (rel_vm, rel_ks)


# ---- 3. zero band-4 rows: degree 4 against degree 3 on the same tensor -------------------------------------------------

@pytest.mark.parametrize("per_cam", [False, True])
@pytest.mark.parametrize("aa", [False, True])
def test_zero_band4_matches_degree3(per_cam, aa):
    sc = make_scene(**S3)
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    d = sc.to("cuda")
    shs = _coeffs(sc, 25, per_cam)
    shs[..., 16:, :] = 0
    cols = shs.cuda()
    fwd = [stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height,
                                 deg, antialiased=aa) for deg in (3, 4)]
    vis = fwd[0]["radii"] > 0
    assert vis.any() and (~vis).any()
    for k in fwd[0]:  # radii, means2d, depths, conics, colours, tile counts, rectangles, splat records
        a, b = (fwd[0][k][vis], fwd[1][k][vis]) if k == "splats" else (fwd[0][k], fwd[1][k])
        assert torch.equal(a, b), k
    v_splats = _records(fwd[0]["radii"], 5)
    v_extra = 0.1 * torch.randn(C, N, 2, generator=torch.Generator().manual_seed(6)).cuda()
    for cam in (False, True):
        kw = dict(want_absgrad=True, antialiased_opacities=d.opacities if aa else None, want_viewmats_grad=cam,
                  want_Ks_grad=cam)
        b3, b4 = [stages.projection_bwd(d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3,
                                        fwd[0]["radii"], fwd[0]["colors"], v_splats, v_extra, **kw) for deg in (3, 4)]
        for i in range(len(b3)):  # geometry gradients, absgrad and (cam) v_viewmats, v_Ks: bit-identical
            if i != 4:
                assert torch.equal(b3[i], b4[i]), (cam, i)
        assert torch.equal(b3[4][..., :16, :], b4[4][..., :16, :])  # bands 0..3
        assert not b3[4][..., 16:, :].any()
    # band 4 = basis x the colour cotangent where the colour is not clipped, summed over cameras for shared rows
    campos = torch.inverse(sc.viewmats.double())[:, :3, 3]
    Y4 = sh_basis4(sc.means.double()[None] - campos[:, None])[..., 16:]  # [C,N,9]
    v_rgb = v_splats.double().cpu()[..., 6:9] * (fwd[0]["colors"].cpu() > 0) * vis.cpu()[..., None]
    expect = Y4[..., :, None] * v_rgb[..., None, :]  # [C,N,9,3]
    if not per_cam:
        expect = expect.sum(0)
    got = b4[4][..., 16:, :].double().cpu()
    # (fp32 basis: near a root of a band-4 polynomial, e.g. z (-4.68 z^2 + 2.01), its error is absolute, ~1e-7 |terms|)
    torch.testing.assert_close(got, expect, rtol=1e-5, atol=5e-6)
    # and the images of the whole path
    outs = [rasterization(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height,
                          sh_degree=deg, packed=False, rasterize_mode="antialiased" if aa else "classic")
            for deg in (3, 4)]
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# ---- 4. every gradient element written once ---------------------------------------------------------------------------

@pytest.mark.parametrize("K", [25, 36])
@pytest.mark.parametrize("per_cam", [False, True])
@pytest.mark.parametrize("cam", [False, True])
def test_gradient_buffers_are_written_once(monkeypatch, K, per_cam, cam):
    sc = make_scene(**S3)
    d = sc.to("cuda")
    cols = _coeffs(sc, K, per_cam).cuda()
    f = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height, 4)
    monkeypatch.setattr(stages, "_grad_buffer", lambda t: torch.full(t.shape, float("nan"), dtype=t.dtype, device=t.device))
    out = stages.projection_bwd(d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, 4, 0.3,
                                f["radii"], f["colors"], _records(f["radii"], 5), want_viewmats_grad=cam,
                                want_Ks_grad=cam)
    for i, t in enumerate(out):
        assert not torch.isnan(t).any(), i
    v = out[4]
    culled = (f["radii"] <= 0) if per_cam else (f["radii"] <= 0).all(0)
    assert culled.any() and (~culled).any()
    assert not v[culled].any()
    assert not v[..., 25:, :].any()
    assert v[~culled][:, :25].abs().sum() > 0
    unseen = (f["radii"] <= 0).all(0)
    for t in out[:4]:  # v_means, v_quats, v_scales, v_opacities of Gaussians no camera sees
        assert not t[unseen].any()


# ---- 5. launches ----------------------------------------------------------------------------------------------------

def test_same_launch_count_as_degree3():
    lib = _lib.load()
    sc = make_scene(**S3)
    d = sc.to("cuda")
    C = sc.viewmats.shape[0]

    def count(colors, deg, cam_grad):
        cols = colors.clone().requires_grad_(True)
        vm = d.viewmats.clone().requires_grad_(cam_grad)
        Ks = d.Ks.clone().requires_grad_(cam_grad)
        torch.cuda.synchronize()
        n0 = lib.egs_kernel_launch_count()
        rc, ra, _ = rasterization(d.means, d.quats, d.scales, d.opacities, cols, vm, Ks, sc.width, sc.height,
                                  sh_degree=deg, packed=False)
        (rc.sum() + ra.sum()).backward()
        torch.cuda.synchronize()
        return lib.egs_kernel_launch_count() - n0

    sh16 = d.colors
    sh25 = _coeffs(sc, 25, False).cuda()
    for cam_grad in (False, True):
        count(sh16, 3, cam_grad)  # warm the binning size hints of this shape
        deg3 = count(sh16, 3, cam_grad)
        deg4 = count(sh25, 4, cam_grad)
        deg4_pc = count(sh25[None].expand(C, -1, -1, -1).contiguous(), 4, cam_grad)
        assert deg3 == deg4 == deg4_pc, (cam_grad, deg3, deg4, deg4_pc)
