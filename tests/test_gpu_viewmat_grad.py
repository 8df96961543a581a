"""-m gpu: gradients w.r.t. viewmats (camera pose refinement) — the VG instantiations of the projection backward kernels
and viewmat_grad_finalize_kernel against fp64 autograd through the oracle, end to end through rasterization() and
rasterization_from_parameters(), and a small pose-recovery run."""
import math

import pytest
import torch

from easy_gaussian_splatting_b200 import _lib, rasterization, rasterization_from_parameters, stages
from easy_gaussian_splatting_b200.synthetic import loss_weights, make_scene
from oracle import gsplat_oracle as O
from tests.util import PARAMS, rel_err

pytestmark = pytest.mark.gpu

CASES = [  # those of test_gpu_rasterization.py
    dict(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1),
    dict(kind="blob", N=2_000, width=131, height=77, fx=120.0, seed=7, n_views=3),
    dict(kind="object", N=20_000, width=400, height=400, fx=555.0, seed=1, n_views=1, white_background=True),
    dict(kind="outdoor", N=60_000, width=489, height=273, fx=290.0, seed=2, n_views=1),
]


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


def _oracle_viewmat_grad(sc, sh_degree, colors, radii, v_splats, v_extra=None, aa_opacities=None):
    """fp64 autograd of the functional whose cotangents the records hold, w.r.t. viewmats."""
    vm = sc.viewmats.double().requires_grad_(True)
    m, q, s, Ks = sc.means.double(), sc.quats.double(), sc.scales.double(), sc.Ks.double()
    out = O.fully_fused_projection(m, q, s, vm, Ks, sc.width, sc.height, calc_compensations=aa_opacities is not None)
    v = v_splats.double().cpu()
    vis = radii.cpu() > 0
    v_xy = v[..., 0:2] + (0 if v_extra is None else v_extra.double().cpu())
    total = (out[1] * v_xy * vis[..., None]).sum() + (out[3] * v[..., 2:5]).sum()
    if sh_degree is not None:
        C = vm.shape[0]
        campos = torch.inverse(vm)[:, :3, 3]
        cols = torch.clamp_min(O.spherical_harmonics(sh_degree, m[None] - campos[:, None],
                                                     colors.double().cpu()[None].expand(C, -1, -1, -1), vis) + 0.5, 0)
        total = total + (cols * v[..., 6:9] * vis[..., None]).sum()
    if aa_opacities is not None:
        total = total + (out[4] * v[..., 5] * aa_opacities.double().cpu()[None]).sum()
    total.backward()
    return vm.grad


STAGE_CASES = [
    # (scene, sh_degree, K, antialiased): K = 16 runs projection_bwd_sh16_kernel, the others projection_bwd_kernel
    (dict(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2), 3, 16, False),
    (dict(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2), 3, 16, True),
    (dict(kind="blob", N=6_000, width=33, height=17, fx=15.0, seed=4, n_views=1), 1, 16, False),  # fov clamp active
    (dict(kind="outdoor", N=30_000, width=489, height=273, fx=290.0, seed=2, n_views=3), 2, 9, False),
    (dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=2), None, 1, False),  # direct colours
    (dict(kind="blob", N=8_000, width=131, height=77, fx=120.0, seed=7, n_views=2), None, 1, True),
    (dict(kind="blob", N=3_001, width=24, height=16, fx=30.0, seed=5, n_views=70), 3, 16, False),  # C > 64 cameras
    (dict(kind="blob", N=3_001, width=24, height=16, fx=30.0, seed=5, n_views=70), None, 1, False),
]


@pytest.mark.parametrize("cfg,deg,K,aa", STAGE_CASES)
def test_stage_viewmat_grad(cfg, deg, K, aa):
    sc = make_scene(**cfg)
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    colors = sc.colors[:, :K].contiguous() if deg is not None else torch.rand(N, 3, generator=torch.Generator().manual_seed(2))
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
    new = stages.projection_bwd(*args, **kw, want_viewmats_grad=True)
    again = stages.projection_bwd(*args, **kw, want_viewmats_grad=True)
    assert len(new) == len(old) + 1
    for a, b in zip(old, new[:-1]):  # v_means, v_quats, v_scales, v_opacities, v_colors, absgrad
        assert torch.equal(a, b)
    assert torch.equal(new[-1], again[-1])  # deterministic
    ref = _oracle_viewmat_grad(sc, deg, colors, proj["radii"], v_splats, v_extra, d.opacities if aa else None)
    rel = _per_camera_rel(new[-1], ref)
    print("per-camera rel err", max(rel))
    assert max(rel) <= 1e-4, rel
    if deg is not None and deg >= 1:
        assert new[-1][:, 3].abs().max() > 0  # SH directions reach the bottom row
    else:
        assert float(new[-1][:, 3].abs().max()) == 0.0


def test_stage_raw_entry_viewmat_grad():
    sc = make_scene(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2)
    d = sc.to("cuda")
    raw = (d.means, d.quats, d.scales.log(), torch.logit(d.opacities), d.colors[:, :1].contiguous(), d.colors[:, 1:].contiguous())
    proj = stages.projection_fwd_raw(*raw, d.viewmats, d.Ks, sc.width, sc.height, 3)
    v_splats = _records(proj["radii"], seed=8)
    args = (*raw, d.viewmats, d.Ks, sc.width, sc.height, 3, 0.3, proj["radii"], proj["colors"], v_splats)
    old = stages.projection_bwd_raw(*args, want_absgrad=True)
    new = stages.projection_bwd_raw(*args, want_absgrad=True, want_viewmats_grad=True)
    for a, b in zip(old, new[:-1]):
        assert torch.equal(a, b)
    assert torch.equal(new[-1], stages.projection_bwd_raw(*args, want_viewmats_grad=True)[-1])
    sc_act = make_scene(kind="blob", N=20_000, width=256, height=256, fx=274.5, seed=0, n_views=2)
    sc_act.scales = raw[2].exp().cpu()  # what the folded exp computes
    ref = _oracle_viewmat_grad(sc_act, 3, sc.colors, proj["radii"], v_splats)
    assert max(_per_camera_rel(new[-1], ref)) <= 1e-4


# ---- end to end -----------------------------------------------------------------------------------------------------

def _oracle_e2e(sc, sh_degree, rasterize_mode="classic"):
    leaves = {k: getattr(sc, k).detach().clone().requires_grad_(True) for k in PARAMS}
    vm = sc.viewmats.detach().clone().requires_grad_(True)
    C = vm.shape[0]
    bg = sc.background[None].expand(C, 3).contiguous()
    rc, ra, meta = O.rasterization(leaves["means"], leaves["quats"], leaves["scales"], leaves["opacities"], leaves["colors"],
                                   vm, sc.Ks, sc.width, sc.height, sh_degree=sh_degree, packed=False, backgrounds=bg,
                                   rasterize_mode=rasterize_mode)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc).sum() + (ra * Wa).sum()).backward()
    return {k: v.grad for k, v in leaves.items()}, vm.grad


def _cuda_e2e(sc, sh_degree, rasterize_mode="classic", packed=False, viewmats_grad=True):
    leaves = {k: getattr(sc, k).detach().clone().cuda().requires_grad_(True) for k in PARAMS}
    vm = sc.viewmats.detach().clone().cuda().requires_grad_(viewmats_grad)
    C = vm.shape[0]
    bg = sc.background[None].expand(C, 3).contiguous().cuda()
    rc, ra, meta = rasterization(leaves["means"], leaves["quats"], leaves["scales"], leaves["opacities"], leaves["colors"],
                                 vm, sc.Ks.cuda(), sc.width, sc.height, sh_degree=sh_degree, packed=packed, backgrounds=bg,
                                 rasterize_mode=rasterize_mode, absgrad=True)
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    return {k: v.grad.cpu() for k, v in leaves.items()}, (vm.grad.cpu() if viewmats_grad else None), meta


@pytest.mark.parametrize("mode", ["classic", "antialiased"])
@pytest.mark.parametrize("cfg", CASES)
def test_end_to_end_viewmat_grad_vs_oracle(cfg, mode):
    sc = make_scene(**cfg)
    ref_g, ref_vm = _oracle_e2e(sc, 3, mode)
    g, vm_grad, _ = _cuda_e2e(sc, 3, mode)
    g_plain, _, _ = _cuda_e2e(sc, 3, mode, viewmats_grad=False)
    errs = {k: rel_err(g[k], ref_g[k]) for k in PARAMS}
    rel = _per_camera_rel(vm_grad, ref_vm)
    print(cfg["kind"], mode, "viewmat per-camera rel err", rel, "param grads", errs)
    assert all(e <= 1e-3 for e in errs.values()), errs
    # asking for the camera gradient changes no other gradient: the projection backward outputs are bit-identical for the
    # same gradient records (test_stage_viewmat_grad); two separate calls differ only by the order of the blend
    # backward's atomic adds
    for k in PARAMS:
        assert rel_err(g[k], g_plain[k]) <= 5e-5, k
    assert max(rel) <= 1e-3, rel


def test_end_to_end_raw_parameters():
    sc = make_scene(**CASES[1])
    ref_g, ref_vm = _oracle_e2e(sc, 3)
    d = sc.to("cuda")
    raw = [d.means.clone(), d.quats.clone(), d.scales.log(), torch.logit(d.opacities), d.colors[:, :1].contiguous(),
           d.colors[:, 1:].contiguous()]
    raw = [t.requires_grad_(True) for t in raw]
    vm = d.viewmats.clone().requires_grad_(True)
    C = vm.shape[0]
    rc, ra, _ = rasterization_from_parameters(*raw, vm, d.Ks, sc.width, sc.height, 3,
                                              backgrounds=d.background[None].expand(C, 3).contiguous())
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    rel = _per_camera_rel(vm.grad, ref_vm)
    print("raw entry viewmat per-camera rel err", rel)
    assert max(rel) <= 1e-3, rel
    assert rel_err(raw[0].grad.cpu(), ref_g["means"]) <= 1e-3


def test_packed_gives_the_same_viewmat_grad():
    sc = make_scene(**CASES[1])
    _, a, _ = _cuda_e2e(sc, 3, packed=False)
    _, b, meta = _cuda_e2e(sc, 3, packed=True)
    assert meta["camera_ids"] is not None
    assert max(_per_camera_rel(b, a)) <= 5e-5  # (run-to-run order of the blend backward's atomic adds only)


def test_many_cameras_tiny_image():
    """C = 70 > the 64 cameras of the kernels' shared-memory table: the per-camera loads of the cam_local path."""
    sc = make_scene(kind="blob", N=1500, width=24, height=16, fx=30.0, seed=6, n_views=70)
    _, ref_vm = _oracle_e2e(sc, 3)
    _, vm_grad, _ = _cuda_e2e(sc, 3)
    rel = _per_camera_rel(vm_grad, ref_vm)
    print("C=70 max per-camera rel err", max(rel))
    assert max(rel) <= 1e-3, rel


def test_inverse_of_camera_to_world_reaches_the_leaf():
    """viewmats = inverse(c2w): a strided, non-leaf input; the gradient must arrive on the c2w leaf."""
    sc = make_scene(**CASES[1])
    c2w_cpu = torch.inverse(sc.viewmats.double()).float()
    c2w_o = c2w_cpu.double().requires_grad_(True)
    C = c2w_o.shape[0]
    leaves = {k: getattr(sc, k).double() for k in PARAMS}
    rc, ra, _ = O.rasterization(*[leaves[k] for k in PARAMS], torch.linalg.inv(c2w_o), sc.Ks.double(), sc.width, sc.height,
                                sh_degree=3, packed=False, backgrounds=sc.background[None].expand(C, 3).double())
    Wc, Wa = loss_weights(sc.seed, C, sc.height, sc.width)
    ((rc * Wc.double()).sum() + (ra * Wa.double()).sum()).backward()
    d = sc.to("cuda")
    c2w = c2w_cpu.cuda().requires_grad_(True)
    vm = torch.linalg.inv(c2w).transpose(1, 2).contiguous().transpose(1, 2)  # strided on purpose
    assert not vm.is_contiguous()
    rc, ra, _ = rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, vm, d.Ks, sc.width, sc.height, sh_degree=3,
                              packed=False, backgrounds=d.background[None].expand(C, 3).contiguous())
    ((rc * Wc.cuda()).sum() + (ra * Wa.cuda()).sum()).backward()
    rel = _per_camera_rel(c2w.grad, c2w_o.grad)
    print("c2w per-camera rel err", rel)
    assert max(rel) <= 1e-3, rel


def test_launch_count_grows_by_the_finalize_launch():
    lib = _lib.load()
    sc = make_scene(**CASES[0]).to("cuda")

    def launches(vg):
        p = {k: getattr(sc, k).clone().requires_grad_(True) for k in PARAMS}
        vm = sc.viewmats.clone().requires_grad_(vg)
        rc, ra, _ = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], p["colors"], vm, sc.Ks, sc.width,
                                  sc.height, sh_degree=3, packed=False, backgrounds=sc.background[None])
        loss = rc.sum() + ra.sum()
        torch.cuda.synchronize()
        n0 = lib.egs_kernel_launch_count()
        loss.backward()
        torch.cuda.synchronize()
        return lib.egs_kernel_launch_count() - n0

    launches(False), launches(True)  # warm-up: the binning hints of this shape
    assert launches(True) == launches(False) + 1


# ---- pose recovery --------------------------------------------------------------------------------------------------

def _hat(w):
    z = torch.zeros_like(w[0])
    return torch.stack([torch.stack([z, -w[2], w[1]]), torch.stack([w[2], z, -w[0]]), torch.stack([-w[1], w[0], z])])


def _se3_exp(xi):
    """4x4 exp of the twist xi = (rho, omega) (differentiable, via the matrix exponential of the 4x4 generator)."""
    G = torch.zeros(4, 4, dtype=xi.dtype, device=xi.device)
    G = G + torch.nn.functional.pad(_hat(xi[3:]), (0, 1, 0, 1))
    G = G + torch.nn.functional.pad(xi[:3, None], (3, 0, 0, 1))
    return torch.linalg.matrix_exp(G)


POSE_STEPS = 150


def test_pose_recovery_smoke():
    """One camera of a 10 k-Gaussian blob scene, perturbed by 1 degree and 1 % of the scene scale (exp(xi^) V), is pulled
    back by Adam on the L1 distance to the image rendered from the true pose: after POSE_STEPS steps the pose error is
    below a fifth of the initial one."""
    sc = make_scene(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1).to("cuda")
    V_true = sc.viewmats.clone()
    scale = float((sc.means - sc.means.mean(0)).norm(dim=-1).mean())
    bg = sc.background[None]

    def render(vm):
        rc, _, _ = rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, vm, sc.Ks, sc.width, sc.height,
                                 sh_degree=3, packed=False, backgrounds=bg)
        return rc

    with torch.no_grad():
        target = render(V_true)
    axis = torch.tensor([0.3, -0.8, 0.5], device="cuda")
    axis = axis / axis.norm()
    tdir = torch.tensor([0.6, 0.2, -0.77], device="cuda")
    tdir = tdir / tdir.norm()
    xi0 = torch.cat([tdir * 0.01 * scale, axis * math.radians(1.0)])
    V_pert = (_se3_exp(xi0) @ V_true[0])[None]

    def pose_err(V):
        dR = V[0, :3, :3] @ V_true[0, :3, :3].T
        ang = torch.arccos(((torch.trace(dR) - 1) / 2).clamp(-1, 1)).item()
        return ang / math.radians(1.0) + (V[0, :3, 3] - V_true[0, :3, 3]).norm().item() / (0.01 * scale)

    xi = torch.zeros(6, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([xi], lr=2e-3)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=0.98)
    e0 = pose_err(V_pert)
    for _ in range(POSE_STEPS):
        opt.zero_grad()
        vm = (_se3_exp(xi) @ V_pert[0])[None]
        loss = (render(vm) - target).abs().mean()
        loss.backward()
        opt.step()
        sched.step()
    with torch.no_grad():
        e1 = pose_err((_se3_exp(xi) @ V_pert[0])[None])
    print(f"pose error {e0:.4f} -> {e1:.4f} after {POSE_STEPS} steps")
    assert e1 < 0.2 * e0
