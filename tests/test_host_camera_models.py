"""CPU tests: project_fwd / project_bwd of csrc/egs_math.cuh for the orthographic and fisheye camera models, compiled for
the host by tests/host_harness/camera_model_harness.cpp, against tests/camera_model_reference.py: the fp32 forward bit
for bit, the backward against fp64 autograd (v_means, quats, scales, v_viewmats, v_Ks; classic and antialiased, with a
non-zero depth cotangent), the polynomial theta / r against fp64 over the whole range, and the fisheye model's first
order agreement with the pinhole one at the optical axis."""
import math

import numpy as np
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import look_at, make_scene
from tests import camera_model_reference as R
from tests.host_harness import camera_model as hc

f32 = torch.float32


def _identity_views(C=1):
    return torch.eye(4, dtype=f32)[None].repeat(C, 1, 1).contiguous()


def _K(fx, fy, cx, cy):
    return torch.tensor([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]], dtype=f32)


def _gaussians(means, seed):
    g = torch.Generator().manual_seed(seed)
    N = means.shape[0]
    quats = torch.randn(N, 4, generator=g, dtype=f32)
    scales = torch.exp(math.log(0.03) + 0.5 * torch.randn(N, 3, generator=g, dtype=f32))
    return means.contiguous(), quats, scales


def _blob(model):
    sc = make_scene(kind="blob", N=3000, width=128, height=96, fx=120.0, seed=0, n_views=2)
    Ks = sc.Ks.clone()
    if model == "ortho":  # ~2 world units across the image: the blob fills it
        Ks[:, 0, 0] = Ks[:, 1, 1] = 30.0
    return dict(means=sc.means, quats=sc.quats, scales=sc.scales, viewmats=sc.viewmats, Ks=Ks, width=128, height=96)


def _wide_fisheye():
    """A camera inside the blob with a 180-degree-wide image: angles up to ~90 degrees, some Gaussians behind it."""
    sc = make_scene(kind="blob", N=3000, width=160, height=120, fx=120.0, seed=1, n_views=1)
    vm = look_at(torch.tensor([0.3, -0.2, -1.2], dtype=f32), torch.zeros(3, dtype=f32), up_world=(0.0, -1.0, 0.0))
    return dict(means=sc.means, quats=sc.quats, scales=sc.scales, viewmats=vm[None].contiguous(),
                Ks=_K(50.0, 50.0, 80.0, 60.0)[None].contiguous(), width=160, height=120)


def _axis():
    """Gaussians exactly on the optical axis and at r / z = 1e-6 and 1e-8 (identity view: camera space = world)."""
    z = torch.tensor([0.5, 1.0, 3.0, 7.0], dtype=f32)
    pts = [torch.stack([0 * z, 0 * z, z], -1)]
    for rel in (1e-6, 1e-8):
        pts.append(torch.stack([rel * z, 0 * z, z], -1))
        pts.append(torch.stack([0 * z, -rel * z, z], -1))
        pts.append(torch.stack([0.6 * rel * z, 0.8 * rel * z, z], -1))
    means, quats, scales = _gaussians(torch.cat(pts), seed=5)
    return dict(means=means, quats=quats, scales=scales, viewmats=_identity_views(),
                Ks=_K(100.0, 90.0, 64.0, 48.0)[None].contiguous(), width=128, height=96)


def _ortho_decades():
    """Orthographic view of Gaussians with z from 0.1 to 100 (three decades)."""
    g = torch.Generator().manual_seed(9)
    N = 2000
    z = 10.0 ** (-1.0 + 3.0 * torch.rand(N, generator=g, dtype=f32))
    xy = 2.0 * torch.rand(N, 2, generator=g, dtype=f32) - 1.0
    means, quats, scales = _gaussians(torch.cat([xy, z[:, None]], -1), seed=9)
    return dict(means=means, quats=quats, scales=scales, viewmats=_identity_views(),
                Ks=_K(60.0, 50.0, 64.0, 48.0)[None].contiguous(), width=128, height=96)


def _behind():
    """near_plane < 0: Gaussians all around the camera, z <= 0 included (fisheye theta up to ~150 degrees on screen),
    and one at theta ~ 112 degrees on the image's x axis (identity view: camera space = world)."""
    g = torch.Generator().manual_seed(11)
    N = 3000
    d = torch.randn(N, 3, generator=g, dtype=f32)
    d = d / d.norm(dim=-1, keepdim=True) * (0.5 + 2.5 * torch.rand(N, 1, generator=g, dtype=f32))
    means, quats, scales = _gaussians(torch.cat([d, torch.tensor([[0.5, 0.1, -0.2]])]), seed=11)
    return dict(means=means, quats=quats, scales=scales, viewmats=_identity_views(),
                Ks=_K(30.0, 30.0, 80.0, 60.0)[None].contiguous(), width=160, height=120, near=-10.0)


CASES = {
    "blob": _blob,
    "behind": lambda model: _behind(),
    "wide": lambda model: _wide_fisheye(),
    "axis": lambda model: _axis(),
    "decades": lambda model: _ortho_decades(),
}
MODEL_CASES = [("ortho", "blob"), ("ortho", "decades"), ("ortho", "axis"), ("ortho", "behind"), ("fisheye", "blob"),
               ("fisheye", "wide"), ("fisheye", "axis"), ("fisheye", "behind")]


def _fwd(model, s):
    return hc.projection_fwd(model, s["means"], s["quats"], s["scales"], s["viewmats"], s["Ks"], s["width"], s["height"],
                             near=s.get("near", 0.01))


def _ref_fwd(model, s, dtype=f32, aa=True, grad=False):
    t = {k: (v.to(dtype).requires_grad_(grad) if isinstance(v, torch.Tensor) else v) for k, v in s.items()}
    out = R.fully_fused_projection(t["means"], t["quats"], t["scales"], t["viewmats"], t["Ks"], s["width"], s["height"],
                                   near_plane=s.get("near", 0.01), calc_compensations=aa, camera_model=model)
    return t, out


@pytest.mark.parametrize("model,case", MODEL_CASES)
def test_forward_bit_exact(model, case):
    s = CASES[case](model)
    h = _fwd(model, s)
    _, (radii, means2d, depths, conics, comp) = _ref_fwd(model, s)
    assert (h["radii"] > 0).sum() > 0
    np.testing.assert_array_equal(h["radii"], radii.numpy())
    for name, ref in (("means2d", means2d), ("depths", depths), ("conics", conics), ("compensations", comp)):
        np.testing.assert_array_equal(h[name].view(np.int32), ref.detach().numpy().view(np.int32), err_msg=name)


def test_wide_fisheye_reaches_85_degrees():
    s = _wide_fisheye()
    h = hc.projection_fwd("fisheye", s["means"], s["quats"], s["scales"], s["viewmats"], s["Ks"], s["width"], s["height"])
    vm = s["viewmats"][0]
    pc = s["means"] @ vm[:3, :3].T + vm[:3, 3]
    theta = torch.atan2(pc[:, :2].norm(dim=-1), pc[:, 2])
    vis = torch.from_numpy(h["radii"][0] > 0)
    assert theta[vis].max().item() > math.radians(85.0)


def test_axis_case_is_visible():
    s = _axis()
    for model in ("ortho", "fisheye"):
        h = hc.projection_fwd(model, s["means"], s["quats"], s["scales"], s["viewmats"], s["Ks"], s["width"], s["height"])
        assert (h["radii"] > 0).all(), model


@pytest.mark.parametrize("model", ["ortho", "fisheye"])
def test_behind_case_has_visible_gaussians_behind_the_camera(model):
    s = _behind()
    h = _fwd(model, s)
    z = s["means"][:, 2].numpy()
    vis = h["radii"][0] > 0
    assert (vis & (z < 0)).sum() > 100 and vis[-1], model
    if model == "fisheye":  # the Gaussian at theta ~ 112 degrees
        assert math.degrees(math.atan2(math.hypot(0.5, 0.1), -0.2)) > 110


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("aa", [False, True])
@pytest.mark.parametrize("model,case", MODEL_CASES)
def test_backward_vs_fp64_autograd(model, case, aa):
    s = CASES[case](model)
    h = _fwd(model, s)
    vis = torch.from_numpy(h["radii"] > 0).double()
    C, N = vis.shape
    g = torch.Generator().manual_seed(3)
    v_m2 = torch.randn(C, N, 2, generator=g, dtype=torch.float64)
    v_d = torch.randn(C, N, generator=g, dtype=torch.float64)
    v_con = torch.randn(C, N, 3, generator=g, dtype=torch.float64)
    v_comp = torch.randn(C, N, generator=g, dtype=torch.float64)
    t, out = _ref_fwd(model, s, torch.float64, aa=aa, grad=True)
    total = (out[1] * v_m2 * vis[..., None]).sum() + (out[2] * v_d * vis).sum() + (out[3] * v_con * vis[..., None]).sum()
    if aa:
        total = total + (out[4] * v_comp * vis).sum()
    total.backward()
    got = hc.projection_bwd(model, s["means"], s["quats"], s["scales"], s["viewmats"], s["Ks"], s["width"], s["height"],
                            h["radii"], v_m2.float(), v_d.float(), v_con.float(),
                            v_comps=v_comp.float() if aa else None)
    for name, key in (("v_means", "means"), ("v_quats", "quats"), ("v_scales", "scales")):
        assert _rel(torch.from_numpy(got[name]).double(), t[key].grad) <= 2e-5, name
    for c in range(C):
        assert _rel(torch.from_numpy(got["v_viewmats"][c]).double(), t["viewmats"].grad[c]) <= 2e-5, c
        assert _rel(torch.from_numpy(got["v_Ks"][c]).double(), t["Ks"].grad[c]) <= 2e-5, c
    assert np.all(got["v_Ks"][:, [0, 1, 2], [1, 0, 0]] == 0) and np.all(got["v_Ks"][:, 2, :] == 0)


def test_theta_over_r_within_2_ulp_of_fp64():
    """s = atan2(r, z) / r over theta in [0, pi), five decades of scale, r / z down to 1e-8 and r = 0 exactly."""
    g = np.random.default_rng(0)
    n = 200_000
    theta = np.concatenate([g.uniform(0.0, np.pi * 0.999, n), g.uniform(0.0, 0.05, n // 4),
                            g.uniform(np.pi * 0.75, np.pi * 0.999, n // 4)])
    rho = 10.0 ** g.uniform(-2.0, 3.0, theta.size)
    r = (rho * np.sin(theta)).astype(np.float32)
    z = (rho * np.cos(theta)).astype(np.float32)
    zs = (10.0 ** g.uniform(-2.0, 3.0, 4000)).astype(np.float32)
    tiny = np.concatenate([np.zeros(1000), 10.0 ** g.uniform(-8.0, -5.0, 3000)])
    r = np.concatenate([r, (zs * tiny).astype(np.float32)])
    z = np.concatenate([z, zs])
    keep = r > 0
    s, gg = hc.theta_over_r(r, z)
    exact = np.where(keep, np.arctan2(r.astype(np.float64), z) / np.where(keep, r, 1.0), 1.0 / z.astype(np.float64))
    ulp = np.spacing(np.abs(exact).astype(np.float32)).astype(np.float64)
    err = np.abs(s.astype(np.float64) - exact) / ulp
    assert np.all(np.isfinite(s)) and err.max() <= 2.0, err.max()
    # g = (z / (r^2 + z^2) - s) / r^2 in fp64 where it does not cancel, and its limit -2 / (3 z^3) on the axis
    r64, z64 = r.astype(np.float64), z.astype(np.float64)
    direct = r64 > 0.3 * np.abs(z64)
    g_ref = (z64 / (r64 ** 2 + z64 ** 2) - exact) / np.where(direct, r64 ** 2, 1.0)
    scale = 1.0 / (r64 ** 2 + z64 ** 2) ** 1.5
    assert np.max(np.abs(gg[direct] - g_ref[direct]) / (np.abs(g_ref[direct]) + scale[direct])) < 1e-5
    axis = r == 0
    np.testing.assert_allclose(gg[axis], -2.0 / (3.0 * z64[axis] ** 3), rtol=1e-6)


def test_fisheye_matches_pinhole_to_first_order_at_the_axis():
    """On the optical axis theta / r = 1 / z and the fisheye Jacobian is the pinhole one; close to it the two models'
    means2d differ only at third order in r / z, and conics at second."""
    s = _axis()
    out = {m: hc.projection_fwd(m, s["means"], s["quats"], s["scales"], s["viewmats"], s["Ks"], s["width"], s["height"])
           for m in ("pinhole", "fisheye")}
    for key in ("radii", "depths"):
        np.testing.assert_array_equal(out["fisheye"][key], out["pinhole"][key])
    np.testing.assert_allclose(out["fisheye"]["means2d"], out["pinhole"]["means2d"], rtol=1e-6, atol=1e-5)
    np.testing.assert_allclose(out["fisheye"]["conics"], out["pinhole"]["conics"], rtol=1e-5)
