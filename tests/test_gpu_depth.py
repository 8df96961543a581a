"""-m gpu: the expected-depth render modes ("ED", "RGB+ED") through rasterization() against the reference of
tests/depth_reference.py (every colour kind, antialiased mode, backgrounds, packed, camera gradients, C = 65, N = 0,
no-grad), the DEPTH blend kernels against the RGB ones at stage level, the depth cotangent in the egs::depth projection
backward kernels, and a few Adam steps on an L1 depth loss."""
import pytest
import torch

from easy_gaussian_splatting_b200 import rasterization, stages
from easy_gaussian_splatting_b200.synthetic import make_scene
from tests.depth_reference import rasterization_depth
from tests.util import image_report, rel_err

pytestmark = pytest.mark.gpu

S1 = dict(kind="blob", N=4_000, width=128, height=96, fx=120.0, seed=0, n_views=1)
S3 = dict(kind="blob", N=2_001, width=131, height=77, fx=120.0, seed=7, n_views=3)  # N % 4 != 0, ragged image
S65 = dict(kind="blob", N=801, width=24, height=16, fx=30.0, seed=6, n_views=65)   # more cameras than shared memory holds
GEOM = ("means", "quats", "scales", "opacities")


def _colors(sc, kind, seed=3):
    """-> (colours, sh_degree) of a colour kind: "sh<d>" / "shcam<d>" (shared / per-camera SH of degree d), "rgb",
    "rgbcam", "feat<D>" / "featcam<D>"."""
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    if kind.startswith("sh"):
        deg = int(kind[-1])
        base = sc.colors if deg < 4 else torch.cat([sc.colors, 0.15 * torch.randn(N, 9, 3, generator=g)], 1)
        if "cam" in kind:
            base = base[None] + 0.1 * torch.randn(C, *base.shape, generator=g)
        return base.contiguous(), deg
    if kind.startswith("rgb"):
        return (torch.rand(C, N, 3, generator=g) if "cam" in kind else torch.rand(N, 3, generator=g)), None
    D = int(kind.lstrip("featcm"))
    return (torch.rand(C, N, D, generator=g) if "cam" in kind else torch.rand(N, D, generator=g)), None


def _weights(C, H, W, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(C, H, W, D, generator=g), torch.rand(C, H, W, 1, generator=g)


def _run(sc, colors, sh, mode, aa, with_bg, cam_grads, packed, device):
    """One forward + backward of a random linear functional; the reference on the CPU, ours on the GPU."""
    C = sc.viewmats.shape[0]
    dev = torch.device(device)
    leaves = {k: getattr(sc, k).detach().clone().to(dev).requires_grad_(True) for k in GEOM}
    leaves["colors"] = colors.detach().clone().to(dev).requires_grad_(True)
    D = colors.shape[-1]
    bg = None
    if with_bg:
        bg = (sc.background[None].expand(C, 3) if D == 3 else torch.rand(C, D, generator=torch.Generator().manual_seed(9)))
        bg = bg.contiguous().to(dev).requires_grad_(True)
    vm, Ks = sc.viewmats.clone().to(dev), sc.Ks.clone().to(dev)
    if cam_grads:
        vm.requires_grad_(True)
        Ks.requires_grad_(True)
    kw = dict(sh_degree=sh, backgrounds=bg, absgrad=True, render_mode=mode,
              rasterize_mode="antialiased" if aa else "classic")
    counters = {}
    if device == "cpu":
        rc, ra, meta = rasterization_depth(*[leaves[k] for k in (*GEOM, "colors")], vm, Ks, sc.width, sc.height,
                                           counters=counters, **kw)
    else:
        rc, ra, meta = rasterization(*[leaves[k] for k in (*GEOM, "colors")], vm, Ks, sc.width, sc.height,
                                     packed=packed, **kw)
    Wc, Wa = _weights(C, sc.height, sc.width, rc.shape[-1], sc.seed + 1000)
    ((rc * Wc.to(dev)).sum() + (ra * Wa.to(dev)).sum()).backward()
    grads = {k: (None if v.grad is None else v.grad.cpu()) for k, v in leaves.items()}
    grads["backgrounds"] = None if bg is None or bg.grad is None else bg.grad.cpu()
    if cam_grads:
        grads["viewmats"], grads["Ks"] = vm.grad.cpu(), Ks.grad.cpu()
    return dict(colors=rc.detach().cpu(), alphas=ra.detach().cpu(), grads=grads, radii=meta["radii"].cpu(),
                absgrad=meta["means2d"].absgrad.cpu(), border=counters.get("borderline"), meta=meta)


CASES = [  # (scene, colour kind, mode, antialiased, background, camera gradients, packed)
    (S1, "sh3", "RGB+ED", False, True, True, False),
    (S1, "sh3", "ED", True, True, False, True),
    (S3, "sh0", "RGB+ED", False, False, False, False),
    (S3, "shcam4", "RGB+ED", True, True, False, True),
    (S3, "sh4", "ED", False, False, True, False),
    (S3, "shcam3", "RGB+ED", False, True, True, False),
    (S3, "rgb", "RGB+ED", False, True, False, False),
    (S3, "feat1", "RGB+ED", False, True, False, False),
    (S3, "featcam5", "RGB+ED", True, True, False, True),
    (S3, "feat5", "ED", False, True, False, False),
    (S3, "feat32", "RGB+ED", False, True, True, False),
    (S65, "sh3", "RGB+ED", False, True, False, False),
    (S65, "rgbcam", "ED", False, False, False, False),
]


@pytest.mark.parametrize("cfg,kind,mode,aa,with_bg,cam,packed", CASES,
                         ids=[f"C{c['n_views']}-{k}-{m}-aa{int(a)}-bg{int(b)}-cam{int(v)}-packed{int(p)}"
                              for c, k, m, a, b, v, p in CASES])
def test_reference_parity(cfg, kind, mode, aa, with_bg, cam, packed):
    sc = make_scene(**cfg)
    colors, sh = _colors(sc, kind)
    ref = _run(sc, colors, sh, mode, aa, with_bg, cam, packed, "cpu")
    out = _run(sc, colors, sh, mode, aa, with_bg, cam, packed, "cuda")
    assert out["colors"].shape == ref["colors"].shape
    rep_c = image_report(out["colors"], ref["colors"], ref["border"])
    rep_a = image_report(out["alphas"], ref["alphas"], ref["border"])
    errs = {}
    for k, r in ref["grads"].items():
        g = out["grads"][k]
        assert (g is None) == (r is None), k
        if r is not None:
            assert g.shape == r.shape, k
            errs[k] = rel_err(g, r)
    vis = ref["radii"] > 0
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"][vis] if packed else ref["absgrad"])
    print("colours", rep_c, "alphas", rep_a, "grads", errs)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    assert all(e <= 1e-3 for e in errs.values()), errs
    if mode == "ED":
        assert out["grads"]["colors"] is None and out["grads"]["backgrounds"] is None
    elif with_bg:
        assert out["grads"]["backgrounds"].shape == (sc.viewmats.shape[0], colors.shape[-1])


def test_meta_and_alphas_equal_rgb_and_no_grad_forward():
    sc = make_scene(**S3)
    d = sc.to("cuda")
    outs = {}
    for mode in ("RGB", "ED", "RGB+ED"):
        with torch.no_grad():
            outs[mode] = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width,
                                       sc.height, sh_degree=3, packed=False, render_mode=mode)
    rgb_c, rgb_a, rgb_m = outs["RGB"]
    for mode in ("ED", "RGB+ED"):
        rc, ra, meta = outs[mode]
        assert rc.grad_fn is None and torch.equal(ra, rgb_a)
        for k in ("radii", "means2d", "depths", "conics", "opacities", "colors", "isect_ids", "flatten_ids"):
            assert torch.equal(meta[k], rgb_m[k]), (mode, k)
    assert torch.equal(outs["RGB+ED"][0][..., :3], rgb_c)  # the DEPTH kernel's RGB channels are the RGB kernel's
    assert torch.equal(outs["RGB+ED"][0][..., 3:], outs["ED"][0])


def test_zero_gaussians():
    sc = make_scene(**S3)
    d = sc.to("cuda")
    e = lambda *s: torch.zeros(*s, device="cuda", requires_grad=True)
    means, quats, scales, opac, cols = e(0, 3), e(0, 4), e(0, 3), e(0), e(0, 16, 3)
    rc, ra, _ = rasterization(means, quats, scales, opac, cols, d.viewmats, d.Ks, sc.width, sc.height, sh_degree=3,
                              render_mode="RGB+ED", backgrounds=d.background[None].expand(3, 3).contiguous())
    assert rc.shape == (3, sc.height, sc.width, 4)
    assert torch.all(rc[..., 3] == 0) and torch.all(ra == 0)
    rc.sum().backward()
    assert means.grad.shape == (0, 3)


# ---- stage level ------------------------------------------------------------------------------------------------------

def _stage_setup(cfg, seed=5):
    sc = make_scene(**cfg)
    d = sc.to("cuda")
    proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width,
                                 sc.height, 3)
    tw, th = stages.tile_grid(sc.width, sc.height)
    _, flat, offs = stages.isect_sorted(proj["means2d"], proj["radii"], proj["depths"], proj["tiles_per_gauss"], 16, tw, th)
    C = sc.viewmats.shape[0]
    bg = torch.rand(C, 3, generator=torch.Generator().manual_seed(seed)).cuda()
    return sc, d, proj, flat, offs, bg


STAGE = dict(kind="blob", N=100_000, width=256, height=192, fx=200.0, seed=0, n_views=2)  # long lists


def test_depth_blend_forward_matches_rgb_and_reference():
    sc, d, proj, flat, offs, bg = _stage_setup(STAGE)
    splats = proj["splats"]
    rc, ra, last = stages.rasterize_fwd(splats, offs, flat, bg, sc.width, sc.height)
    dc, da, dlast = stages.rasterize_fwd_depth(splats, offs, flat, bg, sc.width, sc.height)
    assert torch.equal(dc[..., :3], rc) and torch.equal(da, ra) and torch.equal(dlast, last)
    # the depth channel: the same blend of proj["depths"] through the feature kernel (one channel, background 0)
    fc, fa, _ = stages.rasterize_fwd_features(splats, offs, flat, proj["depths"][..., None].contiguous(), None,
                                              sc.width, sc.height)
    assert torch.equal(fa, ra)
    assert (dc[..., 3:] - fc).abs().max().item() <= 1e-5 * max(1.0, fc.abs().max().item())


def test_depth_blend_backward_slots():
    sc, d, proj, flat, offs, bg = _stage_setup(STAGE)
    splats = proj["splats"]
    C = sc.viewmats.shape[0]
    dc, ra, last = stages.rasterize_fwd_depth(splats, offs, flat, bg, sc.width, sc.height)
    g = torch.Generator().manual_seed(2)
    v_c4 = torch.randn(C, sc.height, sc.width, 4, generator=g).cuda()
    v_a = torch.randn(C, sc.height, sc.width, 1, generator=g).cuda()
    # zero depth cotangent: slots 0-10 are the RGB kernel's (up to the order of the atomic adds), slot 11 is 0
    v_zero = v_c4.clone()
    v_zero[..., 3] = 0
    v_rgb = stages.rasterize_bwd(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_zero[..., :3].contiguous(), v_a)
    v_dep = stages.rasterize_bwd_depth(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_zero, v_a)
    for k in range(11):
        assert rel_err(v_dep[..., k].cpu(), v_rgb[..., k].cpu()) <= 1e-6, k
    assert not v_dep[..., 11].any()
    # non-zero cotangent: slot 11 is the depth gradient of the one-channel feature blend of the depths, and the geometry
    # slots are those of the 4-channel feature blend of (r, g, b, depth)
    v_dep = stages.rasterize_bwd_depth(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_c4, v_a)
    feats = torch.cat([proj["colors"], proj["depths"][..., None]], -1).contiguous()
    bg4 = torch.cat([bg, torch.zeros(C, 1, device="cuda")], -1)
    v_geo, v_feat = stages.rasterize_bwd_features(splats, offs, flat, feats, bg4, sc.width, sc.height, ra, last, v_c4, v_a)
    assert v_dep[..., 11].abs().sum() > 0
    assert rel_err(v_dep[..., 11].cpu(), v_feat[..., 3].cpu()) <= 1e-5
    assert rel_err(v_dep[..., 6:9].cpu(), v_feat[..., :3].cpu()) <= 1e-5
    for k in (0, 1, 2, 3, 4, 5, 9, 10):
        assert rel_err(v_dep[..., k].cpu(), v_geo[..., k].cpu()) <= 1e-5, k


def test_projection_backward_takes_the_depth_cotangent():
    """Records that differ only in slot 11: every output but v_means is identical, and v_means differs by
    sum_c v_depth R_c[2,:]; with v_viewmats, row 2 differs by sum_n v_depth (m, 1)."""
    sc, d, proj, flat, offs, bg = _stage_setup(dict(kind="blob", N=5_000, width=128, height=96, fx=120.0, seed=1,
                                                    n_views=3))
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    radii = proj["radii"]
    g = torch.Generator().manual_seed(4)
    rec = torch.randn(C, N, 12, generator=g).cuda() * (radii > 0)[..., None]
    rec[..., 11] = 0
    rec_d = rec.clone()
    v_depth = torch.randn(C, N, generator=g).cuda() * (radii > 0)
    rec_d[..., 11] = v_depth
    args = (d.means, d.quats, d.scales, d.colors, d.viewmats, d.Ks, sc.width, sc.height, 3, 0.3, radii, proj["colors"])
    for aa in (False, True):
        kw = dict(want_absgrad=True, want_viewmats_grad=True, want_Ks_grad=True,
                  antialiased_opacities=d.opacities if aa else None, opacities=d.opacities)
        base = stages.projection_bwd(*args, rec, **kw)
        plain = stages.projection_bwd(*args, rec, depth_grad=True, **kw)  # slot 11 = 0
        dep = stages.projection_bwd(*args, rec_d, depth_grad=True, **kw)
        for i in range(len(base)):  # the egs::depth kernels compute what the others do when slot 11 is 0
            assert rel_err(plain[i].cpu(), base[i].cpu()) <= 1e-6, (aa, i)
        for i in (1, 2, 3, 4, 5, 7):  # v_quats, v_scales, v_opacities, v_colors, absgrad, v_Ks
            assert torch.equal(dep[i], plain[i]), (aa, i)
        base = plain
        R = d.viewmats[:, :3, :3].double()
        expect = torch.einsum("cn,cj->nj", v_depth.double(), R[:, 2, :])
        diff = dep[0].double() - base[0].double()
        assert (diff - expect).abs().max().item() <= 1e-4 * max(1.0, base[0].abs().max().item()), aa
        row2 = torch.cat([v_depth.double() @ d.means.double(), v_depth.double().sum(1, keepdim=True)], 1)
        dvm = dep[6].double() - base[6].double()
        assert (dvm[:, 2, :] - row2).abs().max().item() <= 1e-4 * max(1.0, base[6].abs().max().item()), aa
        assert (dvm[:, [0, 1, 3], :]).abs().max().item() <= 1e-4 * max(1.0, base[6].abs().max().item()), aa


# ---- training sanity ----------------------------------------------------------------------------------------------------

def test_adam_on_an_l1_depth_loss_lowers_it():
    sc = make_scene(**S1)
    d = sc.to("cuda")
    with torch.no_grad():  # the depth map of the scene as it is; the optimisation starts from perturbed means
        target, _, _ = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width,
                                     sc.height, sh_degree=3, render_mode="RGB+ED")
        target = target[..., 3:]
    scale = d.means.std().item()
    noise = torch.randn(d.means.shape, generator=torch.Generator().manual_seed(0)).cuda()
    means = (d.means + 0.05 * scale * noise).requires_grad_(True)
    opt = torch.optim.Adam([means], lr=0.005 * scale)
    losses = []
    for _ in range(30):
        rc, ra, _ = rasterization(means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width,
                                  sc.height, sh_degree=3, render_mode="RGB+ED")
        loss = ((rc[..., 3:] - target).abs() * (ra > 0.5)).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print(losses)
    assert losses[-1] < 0.9 * losses[0], losses
