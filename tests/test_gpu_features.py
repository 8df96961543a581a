"""-m gpu: colours with any number of channels — the feature blend kernels against the D-channel oracle
(tests/features_oracle.py) end to end, against the RGB blend kernels at stage level, the viewmat gradient through them,
their launch count, and the 32-channel chunking."""
import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rasterization, stages
from easy_gaussian_splatting_b200.synthetic import make_scene
from tests import features_oracle as FO
from tests.util import image_report, rel_err

pytestmark = pytest.mark.gpu

GEOM = ("means", "quats", "scales", "opacities")
BLOB = dict(kind="blob", N=2_000, width=131, height=77, fx=120.0, seed=7, n_views=3)
OUTDOOR = dict(kind="outdoor", N=12_000, width=160, height=96, fx=95.0, seed=2, n_views=1)

# (scene, D, per-camera colours, backgrounds, rasterize_mode): every D of the chunk widths and both sides of a chunk
# boundary, [N,D] and [C,N,D], C = 1 and 3, with and without backgrounds, classic and antialiased
PARITY = [
    (BLOB, 1, False, True, "classic"),
    (BLOB, 2, True, False, "antialiased"),
    (OUTDOOR, 4, False, False, "classic"),
    (BLOB, 5, True, True, "classic"),
    (OUTDOOR, 8, True, True, "antialiased"),
    (BLOB, 16, False, True, "antialiased"),
    (OUTDOOR, 32, False, True, "classic"),
    (BLOB, 33, True, True, "classic"),
    (BLOB, 64, False, False, "antialiased"),
    (OUTDOOR, 64, True, True, "classic"),
]


def _inputs(sc, D, per_camera, with_bg, seed=11):
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(seed)
    feats = torch.rand(*((C, N, D) if per_camera else (N, D)), generator=g) * 2.0 - 0.5
    bg = torch.rand(C, D, generator=g) if with_bg else None
    Wc = torch.rand(C, sc.height, sc.width, D, generator=g)
    Wa = torch.rand(C, sc.height, sc.width, 1, generator=g)
    return feats, bg, Wc, Wa


def _run(fn, sc, feats, bg, Wc, Wa, device, mode="classic", viewmats_grad=False, counters=None):
    leaves = {k: getattr(sc, k).detach().clone().to(device).requires_grad_(True) for k in GEOM}
    cols = feats.detach().clone().to(device).requires_grad_(True)
    bgs = None if bg is None else bg.detach().clone().to(device).requires_grad_(True)
    vm = sc.viewmats.detach().clone().to(device).requires_grad_(viewmats_grad)
    kw = dict(counters=counters) if counters is not None else {}
    rc, ra, meta = fn(*[leaves[k] for k in GEOM], cols, vm, sc.Ks.to(device), sc.width, sc.height, sh_degree=None,
                      packed=False, backgrounds=bgs, absgrad=True, rasterize_mode=mode, **kw)
    ((rc * Wc.to(device)).sum() + (ra * Wa.to(device)).sum()).backward()
    grads = {k: v.grad.detach().cpu() for k, v in leaves.items()}
    grads["colors"] = cols.grad.detach().cpu()
    if bgs is not None:
        grads["backgrounds"] = bgs.grad.detach().cpu()
    grads["absgrad"] = meta["means2d"].absgrad.detach().cpu()
    if viewmats_grad:
        grads["viewmats"] = vm.grad.detach().cpu()
    return rc.detach().cpu(), ra.detach().cpu(), grads


@pytest.mark.parametrize("cfg,D,per_camera,with_bg,mode", PARITY)
def test_parity_with_oracle(cfg, D, per_camera, with_bg, mode):
    sc = make_scene(**cfg)
    feats, bg, Wc, Wa = _inputs(sc, D, per_camera, with_bg)
    counters = {}
    rc_o, ra_o, g_o = _run(FO.rasterization_features, sc, feats, bg, Wc, Wa, "cpu", mode, counters=counters)
    rc, ra, g = _run(rasterization, sc, feats, bg, Wc, Wa, "cuda", mode)
    assert rc.shape == (sc.viewmats.shape[0], sc.height, sc.width, D)
    border = counters["borderline"]
    rep_c, rep_a = image_report(rc, rc_o, border), image_report(ra, ra_o, border)
    print(D, per_camera, with_bg, mode, rep_c, rep_a)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    errs = {k: rel_err(g[k], g_o[k]) for k in g_o}
    print("grad rel err", errs)
    assert set(errs) == set(g)
    assert all(e <= 1e-3 for e in errs.values()), errs


def _stage_setup(cfg, seed=5):
    sc = make_scene(**cfg)
    d = sc.to("cuda")
    N = sc.means.shape[0]
    rgb = torch.rand(N, 3, generator=torch.Generator().manual_seed(seed)).cuda()
    proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, rgb, d.viewmats, d.Ks, sc.width, sc.height, None)
    tw, th = stages.tile_grid(sc.width, sc.height)
    _, flat, offs = stages.isect_sorted(proj["means2d"], proj["radii"], proj["depths"], proj["tiles_per_gauss"], 16, tw, th)
    return sc, d, rgb, proj, flat, offs


def test_feature_kernels_match_the_rgb_kernels():
    """D = 3 through the feature entries (CH = 4, one zero pad channel) on the RGB path's records and lists, at a size
    with thousands of entries per tile."""
    sc, d, rgb, proj, flat, offs = _stage_setup(dict(kind="blob", N=200_000, width=256, height=256, fx=274.5, seed=0,
                                                     n_views=2))
    longest = int((offs.reshape(-1)[1:] - offs.reshape(-1)[:-1]).max())
    assert longest >= 2000, longest
    C = sc.viewmats.shape[0]
    bg = torch.rand(C, 3, generator=torch.Generator().manual_seed(1)).cuda()
    splats = proj["splats"]
    rc, ra, last = stages.rasterize_fwd(splats, offs, flat, bg, sc.width, sc.height)
    fc, fa, flast = stages.rasterize_fwd_features(splats, offs, flat, rgb, bg, sc.width, sc.height)
    assert torch.equal(fa, ra) and torch.equal(flast, last)
    assert (fc - rc).abs().max().item() <= 1e-6
    g = torch.Generator().manual_seed(2)
    v_c = torch.randn(C, sc.height, sc.width, 3, generator=g).cuda()
    v_a = torch.randn(C, sc.height, sc.width, 1, generator=g).cuda()
    v_rgb = stages.rasterize_bwd(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_c, v_a)
    v_geo, v_feat = stages.rasterize_bwd_features(splats, offs, flat, rgb, bg, sc.width, sc.height, ra, last, v_c, v_a)
    geo = [0, 1, 2, 3, 4, 5, 9, 10]
    for k in geo:
        e = rel_err(v_geo[..., k].cpu(), v_rgb[..., k].cpu())
        assert e <= 1e-5, (k, e)
    assert not v_geo[..., 6:9].any() and not v_geo[..., 11].any()
    assert v_feat.shape == (sc.means.shape[0], 3)
    assert rel_err(v_feat.cpu(), v_rgb[..., 6:9].sum(0).cpu()) <= 1e-5  # [N,D] rows: summed over the cameras
    # [C,N,D] rows: one gradient row per (camera, Gaussian)
    per_cam = rgb[None].expand(C, -1, -1).contiguous()
    _, v_feat_c = stages.rasterize_bwd_features(splats, offs, flat, per_cam, bg, sc.width, sc.height, ra, last, v_c, v_a)
    assert rel_err(v_feat_c.cpu(), v_rgb[..., 6:9].cpu()) <= 1e-5


def test_viewmat_gradient_with_eight_channels():
    sc = make_scene(**BLOB)
    feats, bg, Wc, Wa = _inputs(sc, 8, False, True, seed=3)
    _, _, g_o = _run(FO.rasterization_features, sc, feats, bg, Wc, Wa, "cpu", viewmats_grad=True)
    _, _, g = _run(rasterization, sc, feats, bg, Wc, Wa, "cuda", viewmats_grad=True)
    a, b = g["viewmats"].double(), g_o["viewmats"].double()
    rel = [((a[c] - b[c]).norm() / b[c].norm()).item() for c in range(b.shape[0])]
    print("per-camera rel err", rel)
    assert max(rel) <= 1e-4, rel


def test_launch_count():
    lib = _lib.load()
    sc = make_scene(**BLOB).to("cuda")

    def launches(D):
        p = {k: getattr(sc, k).clone().requires_grad_(True) for k in GEOM}
        cols = torch.rand(sc.means.shape[0], D, device="cuda").requires_grad_(True)
        torch.cuda.synchronize()
        n0 = lib.egs_kernel_launch_count()
        rc, ra, _ = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], cols, sc.viewmats, sc.Ks,
                                  sc.width, sc.height, packed=False)
        torch.cuda.synchronize()
        n1 = lib.egs_kernel_launch_count()
        (rc.sum() + ra.sum()).backward()
        torch.cuda.synchronize()
        return n1 - n0, lib.egs_kernel_launch_count() - n1

    for D in (3, 1, 8, 32, 64):
        launches(D)  # warm-up: the binning hints of this shape
    rgb = launches(3)
    for D in (1, 5, 8, 16, 32):
        assert launches(D) == rgb, D
    assert launches(64) == (rgb[0] + 1, rgb[1] + 1)


def test_forty_channels_equal_the_32_and_8_channel_calls():
    sc = make_scene(**BLOB).to("cuda")
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(9)
    feats = torch.rand(C, N, 40, generator=g).cuda()
    bg = torch.rand(C, 40, generator=g).cuda()

    def render(cols, b):
        return rasterization(sc.means, sc.quats, sc.scales, sc.opacities, cols, sc.viewmats, sc.Ks, sc.width, sc.height,
                             packed=False, backgrounds=b)

    rc, ra, meta = render(feats, bg)
    r32, a32, _ = render(feats[..., :32].contiguous(), bg[:, :32].contiguous())
    r8, a8, _ = render(feats[..., 32:].contiguous(), bg[:, 32:].contiguous())
    assert torch.equal(rc, torch.cat([r32, r8], -1))
    assert torch.equal(ra, a32)
    # the 8-channel call blends in the 4-pixels-per-lane layout, the 32-channel one in the one-pixel-per-lane layout
    d = (ra - a8).abs()
    print("alpha difference between layouts: max", d.max().item(), "pixels", int((d > 0).sum()), "of", d.numel())
    assert d.max().item() <= 1e-6
    assert meta["colors"].shape == (C, N, 40)
