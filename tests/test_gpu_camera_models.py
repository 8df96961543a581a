"""-m gpu: rasterization_camera_model(camera_model="ortho" | "fisheye") against tests/camera_model_reference.py: radii,
means2d, depths, conics and meta's isect_ids / flatten_ids bit for bit, images on clean pixels, every gradient and
absgrad, over a case table of colour kinds, render modes, antialiased mode, packed, camera gradients, a wide-angle
fisheye view, near_plane < 0 with Gaussians behind the camera, a ragged C = 3 view and C = 65; N = 0 and the no-grad forward; camera_model="pinhole" equal to
rasterization() (forward bit for bit); and a few Adam steps on a fisheye L1 loss."""
import pytest
import torch

from easy_gaussian_splatting_b200 import rasterization, rasterization_camera_model
from easy_gaussian_splatting_b200.synthetic import look_at, make_scene
from tests.camera_model_reference import rasterization_camera_model as reference
from tests.test_gpu_depth import GEOM, _colors, _weights
from tests.util import image_report, rel_err

pytestmark = pytest.mark.gpu

S1 = dict(kind="blob", N=4_000, width=128, height=96, fx=120.0, seed=0, n_views=1)
S3 = dict(kind="blob", N=2_001, width=131, height=77, fx=120.0, seed=7, n_views=3)  # N % 4 != 0, ragged image
S65 = dict(kind="blob", N=801, width=24, height=16, fx=30.0, seed=6, n_views=65)   # more cameras than shared memory holds
SW = dict(kind="blob", N=3_000, width=160, height=120, fx=50.0, seed=1, n_views=1, wide=True)  # fisheye inside the blob
# near_plane < 0: the camera inside the blob sees Gaussians behind it (fisheye theta past 90 degrees, ortho z < 0)
SB = dict(kind="blob", N=3_000, width=160, height=120, fx=40.0, seed=2, n_views=1, wide=True, near=-10.0)


def _scene(cfg, model):
    """make_scene(cfg) with the camera for the model: "ortho" at a quarter of fx (pixels per world unit, the blob fills
    the image); the wide view puts a fisheye camera inside the blob (angles up to ~90 degrees, Gaussians behind it)."""
    cfg = dict(cfg)
    wide = cfg.pop("wide", False)
    cfg.pop("near", None)
    sc = make_scene(**cfg)
    if model == "ortho":
        sc.Ks = sc.Ks.clone()
        sc.Ks[:, 0, 0] = sc.Ks[:, 1, 1] = cfg["fx"] / 4.0
    if wide:
        sc.viewmats = look_at(torch.tensor([0.3, -0.2, -1.2]), torch.zeros(3), up_world=(0.0, -1.0, 0.0))[None].contiguous()
    return sc


def _run(sc, model, colors, sh, mode, aa, with_bg, cam_grads, packed, device, near_plane=0.01):
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
    kw = dict(sh_degree=sh, backgrounds=bg, absgrad=True, render_mode=mode, rasterize_mode="antialiased" if aa else "classic",
              near_plane=near_plane)
    args = [leaves[k] for k in (*GEOM, "colors")] + [vm, Ks, sc.width, sc.height]
    counters = {}
    if device == "cpu":
        rc, ra, meta = reference(*args, camera_model=model, counters=counters, **kw)
    else:
        rc, ra, meta = rasterization_camera_model(*args, packed=packed, camera_model=model, **kw)
    Wc, Wa = _weights(C, sc.height, sc.width, rc.shape[-1], sc.seed + 1000)
    ((rc * Wc.to(dev)).sum() + (ra * Wa.to(dev)).sum()).backward()
    grads = {k: (None if v.grad is None else v.grad.cpu()) for k, v in leaves.items()}
    grads["backgrounds"] = None if bg is None or bg.grad is None else bg.grad.cpu()
    if cam_grads:
        grads["viewmats"], grads["Ks"] = vm.grad.cpu(), Ks.grad.cpu()
    m = {k: meta[k].detach().cpu() for k in ("radii", "means2d", "depths", "conics", "isect_ids", "flatten_ids")}
    return dict(colors=rc.detach().cpu(), alphas=ra.detach().cpu(), grads=grads, meta=m,
                absgrad=meta["means2d"].absgrad.cpu(), border=counters.get("borderline"))


CASES = [  # (scene, model, colour kind, mode, antialiased, background, camera gradients, packed)
    (S1, "fisheye", "sh3", "RGB", False, True, True, False),
    (S1, "ortho", "sh3", "RGB", False, True, True, False),
    (SW, "fisheye", "sh3", "RGB+ED", False, True, True, False),
    (SW, "fisheye", "feat5", "RGB", True, True, True, False),
    (SB, "fisheye", "sh3", "RGB+ED", False, True, True, False),
    (SB, "fisheye", "feat5", "RGB", True, True, True, False),
    (SB, "ortho", "sh3", "RGB", True, True, True, False),
    (S3, "ortho", "sh0", "RGB", True, False, False, True),
    (S3, "fisheye", "shcam4", "RGB+ED", True, True, False, True),
    (S3, "ortho", "sh4", "ED", False, False, True, False),
    (S3, "fisheye", "shcam3", "RGB", False, True, True, False),
    (S3, "ortho", "rgb", "RGB", False, True, False, False),
    (S3, "fisheye", "feat1", "RGB", False, True, True, False),
    (S3, "ortho", "featcam5", "RGB+ED", True, True, False, True),
    (S3, "fisheye", "feat5", "ED", False, True, False, False),
    (S3, "fisheye", "feat32", "RGB", False, True, True, False),
    (S65, "ortho", "sh3", "RGB+ED", False, True, True, False),
    (S65, "fisheye", "rgbcam", "RGB", False, False, True, False),
]


@pytest.mark.parametrize("cfg,model,kind,mode,aa,with_bg,cam,packed", CASES,
                         ids=[f"C{c['n_views']}{'w' if c.get('wide') else ''}{'b' if c.get('near', 1) < 0 else ''}-{m}-{k}-{md}-aa{int(a)}-bg{int(b)}-cam{int(v)}"
                              f"-packed{int(p)}" for c, m, k, md, a, b, v, p in CASES])
def test_reference_parity(cfg, model, kind, mode, aa, with_bg, cam, packed):
    sc = _scene(cfg, model)
    colors, sh = _colors(sc, kind)
    near = cfg.get("near", 0.01)
    ref = _run(sc, model, colors, sh, mode, aa, with_bg, cam, packed, "cpu", near)
    out = _run(sc, model, colors, sh, mode, aa, with_bg, cam, packed, "cuda", near)
    vis = ref["meta"]["radii"] > 0
    assert vis.sum() > 0
    if near < 0:  # pairs behind the camera are visible, and their gradients are checked below
        assert (vis & (ref["meta"]["depths"] < 0)).sum() > 50
    for k in ("radii", "means2d", "depths", "conics"):
        r = ref["meta"][k][vis] if packed else ref["meta"][k]
        assert torch.equal(out["meta"][k], r), k
    if not packed:  # (packed flatten_ids index the packed list)
        for k in ("isect_ids", "flatten_ids"):
            assert torch.equal(out["meta"][k], ref["meta"][k].to(out["meta"][k].dtype)), k
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
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"][vis] if packed else ref["absgrad"])
    print("colours", rep_c, "alphas", rep_a, "grads", errs)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    assert all(e <= 1e-3 for e in errs.values()), errs


@pytest.mark.parametrize("model", ["ortho", "fisheye"])
def test_zero_gaussians_and_no_grad_forward(model):
    sc = _scene(S3, model)
    d = sc.to("cuda")
    e = lambda *s: torch.zeros(*s, device="cuda", requires_grad=True)
    means, quats, scales, opac, cols = e(0, 3), e(0, 4), e(0, 3), e(0), e(0, 16, 3)
    Ks = d.Ks.clone().requires_grad_(True)
    rc, ra, _ = rasterization_camera_model(means, quats, scales, opac, cols, d.viewmats, Ks, sc.width, sc.height,
                                           sh_degree=3, render_mode="RGB+ED", camera_model=model)
    assert rc.shape == (3, sc.height, sc.width, 4) and torch.all(ra == 0)
    rc.sum().backward()
    assert means.grad.shape == (0, 3) and torch.all(Ks.grad == 0)
    with torch.no_grad():
        rc, ra, meta = rasterization_camera_model(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks,
                                                  sc.width, sc.height, sh_degree=3, packed=False, camera_model=model)
    assert rc.grad_fn is None and (meta["radii"] > 0).any()
    rc2, ra2, meta2 = rasterization_camera_model(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks,
                                                 sc.width, sc.height, sh_degree=3, packed=False, camera_model=model)
    assert torch.equal(rc, rc2.detach()) and torch.equal(ra, ra2.detach())


def test_pinhole_is_rasterization():
    """The same kernels: the forward outputs are bit-identical.  The gradients agree to the rounding of the blend
    backward's float atomics, whose order varies from run to run (two rasterization() calls differ the same way)."""
    sc = make_scene(**S3)
    outs = []
    for fn, kw in ((rasterization, {}), (rasterization_camera_model, {"camera_model": "pinhole"})):
        d = sc.to("cuda")
        leaves = [t.clone().requires_grad_(True) for t in (d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats,
                                                            d.Ks)]
        rc, ra, meta = fn(*leaves, sc.width, sc.height, sh_degree=3, absgrad=True, packed=False, render_mode="RGB+ED",
                          **kw)
        Wc, Wa = _weights(3, sc.height, sc.width, 4, 11)
        ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
        outs.append([rc, ra, meta["means2d"], meta["conics"], meta["radii"], meta["means2d"].absgrad] +
                    [t.grad for t in leaves])
    for i, (a, b) in enumerate(zip(*outs)):
        if i < 5:
            assert torch.equal(a, b), i
        else:
            assert rel_err(b.cpu(), a.cpu()) <= 1e-6, i


def test_adam_on_a_fisheye_l1_loss_lowers_it():
    sc = _scene(S1, "fisheye")
    d = sc.to("cuda")
    kw = dict(sh_degree=3, camera_model="fisheye")
    with torch.no_grad():
        target, _, _ = rasterization_camera_model(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks,
                                                  sc.width, sc.height, **kw)
    scale = d.means.std().item()
    noise = torch.randn(d.means.shape, generator=torch.Generator().manual_seed(0)).cuda()
    means = (d.means + 0.05 * scale * noise).requires_grad_(True)
    opt = torch.optim.Adam([means], lr=0.005 * scale)
    losses = []
    for _ in range(30):
        rc, _, _ = rasterization_camera_model(means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks,
                                              sc.width, sc.height, **kw)
        loss = (rc - target).abs().mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print(losses)
    assert losses[-1] < 0.9 * losses[0], losses
