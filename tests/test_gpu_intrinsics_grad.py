"""-m gpu: gradients w.r.t. Ks (camera intrinsics refinement) — the egs::ksgrad instantiations of the projection backward
kernels and intrinsics_grad_finalize_kernel against fp64 autograd through the oracle, end to end through rasterization()
and rasterization_from_parameters(), the launch count, and a small intrinsics-recovery run."""
import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rasterization, rasterization_from_parameters, stages
from easy_gaussian_splatting_b200.synthetic import loss_weights, make_scene
from oracle import gsplat_oracle as O
from tests import features_oracle as FO
from tests.util import PARAMS

pytestmark = pytest.mark.gpu

CASES = [  # those of test_gpu_rasterization.py
    dict(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1),
    dict(kind="blob", N=2_000, width=131, height=77, fx=120.0, seed=7, n_views=3),
    dict(kind="object", N=20_000, width=400, height=400, fx=555.0, seed=1, n_views=1, white_background=True),
    dict(kind="outdoor", N=60_000, width=489, height=273, fx=290.0, seed=2, n_views=1),
]
OFF = torch.ones(3, 3, dtype=torch.bool)
OFF[0, 0] = OFF[1, 1] = OFF[0, 2] = OFF[1, 2] = False  # the entries the projection does not read


def _per_camera_rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return [((a[c] - b[c]).norm() / b[c].norm().clamp_min(1e-30)).item() for c in range(b.shape[0])]


# ---- stage level ----------------------------------------------------------------------------------------------------

def _records(radii, seed):
    """Random gradient records {v_x,v_y,v_ca,v_cb | v_cc,v_opacity,v_r,v_g | v_b,|v_x|,|v_y|,0}, zero where culled."""
    C, N = radii.shape
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(C, N, 12, generator=g)
    v[..., 9:11] = v[..., 0:2].abs()
    v[..., 11] = 0.0
    v *= (radii.cpu() > 0)[..., None]
    return v.cuda()


def _oracle_Ks_grad(sc, radii, v_splats, v_extra=None, aa_opacities=None):
    """fp64 autograd w.r.t. Ks of the functional whose cotangents the records hold (the colours do not read Ks)."""
    Ks = sc.Ks.double().requires_grad_(True)
    m, q, s, vm = sc.means.double(), sc.quats.double(), sc.scales.double(), sc.viewmats.double()
    out = O.fully_fused_projection(m, q, s, vm, Ks, sc.width, sc.height, calc_compensations=aa_opacities is not None)
    v = v_splats.double().cpu()
    vis = radii.cpu() > 0
    v_xy = v[..., 0:2] + (0 if v_extra is None else v_extra.double().cpu())
    total = (out[1] * v_xy * vis[..., None]).sum() + (out[3] * v[..., 2:5]).sum()
    if aa_opacities is not None:
        total = total + (out[4] * v[..., 5] * aa_opacities.double().cpu()[None]).sum()
    total.backward()
    return Ks.grad


STAGE_CASES = [
    # (scene, sh_degree, K, per-camera colours, antialiased): the dispatch family in the id
    pytest.param(dict(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2), 3, 16, False, False,
                 id="sh16"),
    pytest.param(dict(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2), 3, 16, False, True,
                 id="sh16-aa"),
    pytest.param(dict(kind="blob", N=6_000, width=33, height=17, fx=60.0, seed=4, n_views=1), 1, 16, False, False,
                 id="sh16-fov-clamp"),
    pytest.param(dict(kind="outdoor", N=30_000, width=489, height=273, fx=290.0, seed=2, n_views=3), 2, 9, False, False,
                 id="generic"),
    pytest.param(dict(kind="outdoor", N=30_000, width=489, height=273, fx=290.0, seed=2, n_views=3), 1, 4, False, True,
                 id="vec4-aa"),
    pytest.param(dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=2), None, 1, False, False,
                 id="direct-colours"),
    pytest.param(dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=2), None, 1, True, True,
                 id="direct-colours-per-camera-aa"),
    pytest.param(dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=3), 3, 16, True, False,
                 id="per-camera-sh16"),
    pytest.param(dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=3), 2, 9, True, True,
                 id="per-camera-generic-aa"),
    pytest.param(dict(kind="blob", N=3_001, width=24, height=16, fx=30.0, seed=5, n_views=70), 3, 16, False, False,
                 id="sh16-C70"),
    pytest.param(dict(kind="blob", N=3_001, width=24, height=16, fx=30.0, seed=5, n_views=70), 2, 9, False, False,
                 id="generic-C70"),
]


@pytest.mark.parametrize("cfg,deg,K,per_cam,aa", STAGE_CASES)
def test_stage_Ks_grad(cfg, deg, K, per_cam, aa):
    sc = make_scene(**cfg)
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(2)
    if deg is not None:
        colors = sc.colors[:, :K].contiguous()
        if per_cam:
            colors = (colors[None] + 0.1 * torch.randn(C, N, K, 3, generator=g)).contiguous()
    else:
        colors = torch.rand(*((C, N, 3) if per_cam else (N, 3)), generator=g)
    d = sc.to("cuda")
    cols = colors.cuda()
    proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols, d.viewmats, d.Ks, sc.width, sc.height,
                                 deg, antialiased=aa)
    v_splats = _records(proj["radii"], seed=3)
    v_extra = 0.1 * torch.randn(C, N, 2, generator=torch.Generator().manual_seed(4)).cuda()
    args = (d.means, d.quats, d.scales, cols, d.viewmats, d.Ks, sc.width, sc.height, deg, 0.3, proj["radii"],
            proj["colors"], v_splats, v_extra)
    kw = dict(want_absgrad=True, antialiased_opacities=d.opacities if aa else None)
    old = stages.projection_bwd(*args, **kw)
    vm_only = stages.projection_bwd(*args, **kw, want_viewmats_grad=True)
    ks_only = stages.projection_bwd(*args, **kw, want_Ks_grad=True)
    both = stages.projection_bwd(*args, **kw, want_viewmats_grad=True, want_Ks_grad=True)
    again = stages.projection_bwd(*args, **kw, want_viewmats_grad=True, want_Ks_grad=True)
    assert len(ks_only) == len(old) + 1 and len(both) == len(old) + 2
    for i, a in enumerate(old):  # v_means, v_quats, v_scales, v_opacities, v_colors, absgrad
        assert torch.equal(a, ks_only[i]) and torch.equal(a, both[i]), i
    assert torch.equal(both[-2], vm_only[-1])  # v_viewmats: bit-identical with or without v_Ks
    assert torch.equal(both[-1], ks_only[-1]) and torch.equal(both[-1], again[-1])  # deterministic
    v_Ks = both[-1].cpu()
    assert v_Ks.shape == (C, 3, 3) and torch.all(v_Ks[:, OFF] == 0.0)
    ref = _oracle_Ks_grad(sc, proj["radii"], v_splats, v_extra, d.opacities if aa else None)
    rel = _per_camera_rel(v_Ks, ref)
    print("per-camera rel err", max(rel))
    assert max(rel) <= 1e-4, rel


@pytest.mark.parametrize("with_vm", [False, True])
def test_stage_raw_entry_Ks_grad(with_vm):
    sc = make_scene(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2)
    d = sc.to("cuda")
    raw = (d.means, d.quats, d.scales.log(), torch.logit(d.opacities), d.colors[:, :1].contiguous(), d.colors[:, 1:].contiguous())
    proj = stages.projection_fwd_raw(*raw, d.viewmats, d.Ks, sc.width, sc.height, 3)
    v_splats = _records(proj["radii"], seed=8)
    args = (*raw, d.viewmats, d.Ks, sc.width, sc.height, 3, 0.3, proj["radii"], proj["colors"], v_splats)
    old = stages.projection_bwd_raw(*args, want_absgrad=True, want_viewmats_grad=with_vm)
    new = stages.projection_bwd_raw(*args, want_absgrad=True, want_viewmats_grad=with_vm, want_Ks_grad=True)
    assert len(new) == len(old) + 1
    for a, b in zip(old, new[:-1]):  # including v_viewmats
        assert torch.equal(a, b)
    assert torch.equal(new[-1], stages.projection_bwd_raw(*args, want_Ks_grad=True)[-1])
    sc_act = make_scene(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2)
    sc_act.scales = raw[2].exp().cpu()  # what the folded exp computes
    rel = _per_camera_rel(new[-1], _oracle_Ks_grad(sc_act, proj["radii"], v_splats))
    print("raw per-camera rel err", max(rel))
    assert max(rel) <= 1e-4, rel


def test_stage_no_gaussians_gives_zeros():
    sc = make_scene(kind="blob", N=100, width=64, height=64, fx=70.0, seed=0, n_views=2).to("cuda")
    z = torch.zeros(0, 3, device="cuda")
    out = stages.projection_bwd(z, torch.zeros(0, 4, device="cuda"), z, torch.zeros(0, 16, 3, device="cuda"), sc.viewmats,
                                sc.Ks, 64, 64, 3, 0.3, torch.zeros(2, 0, dtype=torch.int32, device="cuda"),
                                torch.zeros(2, 0, 3, device="cuda"), torch.zeros(2, 0, 12, device="cuda"),
                                want_viewmats_grad=True, want_Ks_grad=True)
    assert out[-1].shape == (2, 3, 3) and float(out[-1].abs().max()) == 0.0
    assert out[-2].shape == (2, 4, 4) and float(out[-2].abs().max()) == 0.0


# ---- end to end -----------------------------------------------------------------------------------------------------

def _oracle_e2e(sc, rasterize_mode="classic", with_bg=True, colors=None, sh_degree=3):
    """fp64 oracle: Ks.grad of the bench functional."""
    leaves = [getattr(sc, k).double() for k in PARAMS]
    if colors is not None:
        leaves[4] = colors.double()
    Ks = sc.Ks.double().requires_grad_(True)
    C = Ks.shape[0]
    D = leaves[4].shape[-1]
    bg = _background(sc, D).double() if with_bg else None
    fn = O.rasterization if sh_degree is not None else FO.rasterization_features
    rc, ra, _ = fn(*leaves, sc.viewmats.double(), Ks, sc.width, sc.height, sh_degree=sh_degree, packed=False,
                   backgrounds=bg, rasterize_mode=rasterize_mode)
    Wc, Wa = _weights(sc, D)
    ((rc * Wc.double()).sum() + (ra * Wa.double()).sum()).backward()
    return Ks.grad


def _background(sc, D):
    C = sc.viewmats.shape[0]
    if D == 3:
        return sc.background[None].expand(C, 3).contiguous()
    return torch.rand(C, D, generator=torch.Generator().manual_seed(12))


def _weights(sc, D):
    C = sc.viewmats.shape[0]
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    if D != 3:
        Wc = torch.rand(C, sc.height, sc.width, D, generator=torch.Generator().manual_seed(13))
    return Wc, Wa


def _cuda_e2e(sc, rasterize_mode="classic", with_bg=True, packed=False, colors=None, sh_degree=3, vm_grad=False):
    leaves = [getattr(sc, k).detach().clone().cuda().requires_grad_(True) for k in PARAMS]
    if colors is not None:
        leaves[4] = colors.detach().clone().cuda().requires_grad_(True)
    D = leaves[4].shape[-1]
    Ks = sc.Ks.detach().clone().cuda().requires_grad_(True)
    vm = sc.viewmats.detach().clone().cuda().requires_grad_(vm_grad)
    bg = _background(sc, D).cuda() if with_bg else None
    rc, ra, meta = rasterization(*leaves, vm, Ks, sc.width, sc.height, sh_degree=sh_degree, packed=packed,
                                 backgrounds=bg, rasterize_mode=rasterize_mode, absgrad=True)
    Wc, Wa = _weights(sc, D)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    return Ks.grad.cpu(), meta


def _check_e2e(got, ref, what):
    rel = _per_camera_rel(got, ref)
    print(what, "Ks per-camera rel err", rel)
    assert torch.all(got[:, OFF] == 0.0)
    assert max(rel) <= 1e-3, rel
    return max(rel)


@pytest.mark.parametrize("with_bg", [True, False])
@pytest.mark.parametrize("mode", ["classic", "antialiased"])
@pytest.mark.parametrize("cfg", CASES)
def test_end_to_end_Ks_grad_vs_oracle(cfg, mode, with_bg):
    sc = make_scene(**cfg)
    got, _ = _cuda_e2e(sc, mode, with_bg)
    _check_e2e(got, _oracle_e2e(sc, mode, with_bg), f"{cfg['kind']} {mode} bg={with_bg}")


@pytest.mark.parametrize("per_camera", [False, True])
def test_end_to_end_feature_colours(per_camera):
    sc = make_scene(**CASES[1])
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator().manual_seed(11)
    feats = torch.rand(*((C, N, 5) if per_camera else (N, 5)), generator=g) * 2.0 - 0.5
    got, _ = _cuda_e2e(sc, colors=feats, sh_degree=None)
    _check_e2e(got, _oracle_e2e(sc, colors=feats, sh_degree=None), f"D=5 per_camera={per_camera}")


@pytest.mark.parametrize("mode", ["classic", "antialiased"])
def test_end_to_end_per_camera_sh(mode):
    sc = make_scene(**CASES[1])
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    shs = (sc.colors[None] + 0.1 * torch.randn(C, N, 16, 3, generator=torch.Generator().manual_seed(3))).contiguous()
    got, _ = _cuda_e2e(sc, mode, colors=shs)
    _check_e2e(got, _oracle_e2e(sc, mode, colors=shs), f"per-camera SH {mode}")


def test_end_to_end_raw_parameters_and_packed():
    sc = make_scene(**CASES[1])
    ref = _oracle_e2e(sc)
    a, _ = _cuda_e2e(sc, packed=False, vm_grad=True)
    b, meta = _cuda_e2e(sc, packed=True)
    assert meta["camera_ids"] is not None
    _check_e2e(a, ref, "dense with viewmats")
    _check_e2e(b, ref, "packed")
    d = sc.to("cuda")
    raw = [d.means.clone(), d.quats.clone(), d.scales.log(), torch.logit(d.opacities), d.colors[:, :1].contiguous(),
           d.colors[:, 1:].contiguous()]
    raw = [t.requires_grad_(True) for t in raw]
    Ks = d.Ks.clone().requires_grad_(True)
    C = Ks.shape[0]
    rc, ra, _ = rasterization_from_parameters(*raw, d.viewmats, Ks, sc.width, sc.height, 3,
                                              backgrounds=d.background[None].expand(C, 3).contiguous())
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    _check_e2e(Ks.grad.cpu(), ref, "raw entry")


def test_many_cameras_tiny_image():
    """C = 70 > the 64 cameras of the kernels' shared-memory table: the per-camera loads of the cam_local path."""
    sc = make_scene(kind="blob", N=1500, width=24, height=16, fx=30.0, seed=6, n_views=70)
    got, _ = _cuda_e2e(sc)
    _check_e2e(got, _oracle_e2e(sc), "C=70")


def test_loss_on_means2d_only():
    """A loss placed only on meta["means2d"]: v_cx / v_cy are the sums of its gradient over the visible Gaussians."""
    sc = make_scene(**CASES[1]).to("cuda")
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    Ks = sc.Ks.clone().requires_grad_(True)
    _, _, meta = rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, sc.viewmats, Ks, sc.width,
                               sc.height, sh_degree=3, packed=False)
    G = torch.randn(C, N, 2, generator=torch.Generator().manual_seed(5)).cuda()
    (meta["means2d"] * G).sum().backward()
    vis = (meta["radii"] > 0)[..., None]
    expect = (G.double() * vis).sum(dim=1).cpu()
    got = Ks.grad.double().cpu()
    err = (got[:, :2, 2] - expect).abs().max().item()
    print("means2d-only: max |(v_cx, v_cy) - sum|", err, "of", expect.abs().max().item())
    assert torch.allclose(got[:, :2, 2], expect, rtol=1e-5, atol=1e-3)
    # fx / fy take the means2d path alone here: against fp64 autograd through the oracle's projection
    d = sc.to("cpu")
    Kd = d.Ks.double().requires_grad_(True)
    out = O.fully_fused_projection(d.means.double(), d.quats.double(), d.scales.double(), d.viewmats.double(), Kd,
                                   sc.width, sc.height)
    (out[1] * G.double().cpu() * vis.cpu()).sum().backward()
    assert max(_per_camera_rel(got, Kd.grad)) <= 1e-4


def test_launch_count_grows_by_the_finalize_launch():
    lib = _lib.load()
    sc = make_scene(**CASES[0]).to("cuda")

    def launches(vg, kg):
        p = {k: getattr(sc, k).clone().requires_grad_(True) for k in PARAMS}
        vm = sc.viewmats.clone().requires_grad_(vg)
        Ks = sc.Ks.clone().requires_grad_(kg)
        rc, ra, _ = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], p["colors"], vm, Ks, sc.width,
                                  sc.height, sh_degree=3, packed=False, backgrounds=sc.background[None])
        loss = rc.sum() + ra.sum()
        torch.cuda.synchronize()
        n0 = lib.egs_kernel_launch_count()
        loss.backward()
        torch.cuda.synchronize()
        return lib.egs_kernel_launch_count() - n0

    for flags in ((False, False), (False, True), (True, True)):  # warm-up: the binning hints of this shape
        launches(*flags)
    plain = launches(False, False)
    assert launches(False, True) == plain + 1
    assert launches(True, True) == plain + 1


# ---- intrinsics recovery --------------------------------------------------------------------------------------------

RECOVERY_STEPS = 200


def test_intrinsics_recovery():
    """Frozen Gaussians, 4 views sharing one K.  Start from fx, fy x 1.05 and the principal point off by (+4, -3) px;
    Adam on the L1 distance to the images rendered with the true K brings both the relative focal error and the
    principal-point error down by at least 10x within RECOVERY_STEPS steps."""
    sc = make_scene(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=4).to("cuda")
    C = sc.viewmats.shape[0]
    K_true = sc.Ks[0].clone()
    bg = sc.background[None].expand(C, 3).contiguous()

    def render(K):
        rc, _, _ = rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, sc.viewmats,
                                 K[None].expand(C, 3, 3), sc.width, sc.height, sh_degree=3, packed=False, backgrounds=bg)
        return rc

    with torch.no_grad():
        target = render(K_true)
    f0 = K_true[[0, 1], [0, 1]] * 1.05
    c0 = K_true[[0, 1], [2, 2]] + torch.tensor([4.0, -3.0], device="cuda")
    theta = torch.zeros(4, device="cuda", requires_grad=True)  # log focal factors, principal point offset / 10 px

    def intrinsics(th):
        f = f0 * torch.exp(th[:2])
        c = c0 + 10.0 * th[2:]
        z = torch.zeros((), device="cuda")
        one = torch.ones((), device="cuda")
        return torch.stack([torch.stack([f[0], z, c[0]]), torch.stack([z, f[1], c[1]]), torch.stack([z, z, one])])

    def errors(K):
        f_err = ((K[[0, 1], [0, 1]] - K_true[[0, 1], [0, 1]]).abs() / K_true[[0, 1], [0, 1]]).max().item()
        c_err = (K[[0, 1], [2, 2]] - K_true[[0, 1], [2, 2]]).norm().item()
        return f_err, c_err

    opt = torch.optim.Adam([theta], lr=1e-2)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=0.985)
    fe0, ce0 = errors(intrinsics(theta.detach()))
    for _ in range(RECOVERY_STEPS):
        opt.zero_grad()
        loss = (render(intrinsics(theta)) - target).abs().mean()
        loss.backward()
        opt.step()
        sched.step()
    fe1, ce1 = errors(intrinsics(theta.detach()))
    print(f"relative focal error {fe0:.4g} -> {fe1:.4g}, principal point error {ce0:.4g} -> {ce1:.4g} px "
          f"after {RECOVERY_STEPS} steps")
    assert fe1 <= 0.1 * fe0 and ce1 <= 0.1 * ce0
