"""CPU checks of the fixtures and references of tests/test_gpu_projection_paths.py: every seeded case holds every
population it is built from, measured with the fp32 oracle (so a later edit of the generator cannot drop an edge
unnoticed), and the references agree with the host-compiled kernel math where they must."""
import numpy as np
import pytest
import torch

from oracle import gsplat_oracle as O
from tests import host_harness as hh
from tests import test_gpu_projection_paths as T


def _census(case):
    """population -> present, from the fp32 oracle's projection of the case"""
    C, N = case.C, case.N
    radii, m2, dep, con = O.fully_fused_projection(case.means, case.quats, case.scales, case.viewmats, case.Ks, T.W, T.H,
                                                   T.EPS2D, T.NEAR, T.FAR, T.CLIP)
    vis = (radii > 0).numpy()
    vm = case.viewmats.double()
    pc = (torch.einsum("cij,nj->cni", vm[:, :3, :3], case.means.double()) + vm[:, None, :3, 3]).numpy()
    z = pc[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        ax, ay = np.abs(pc[..., 0] / z) / T.TAN_X, np.abs(pc[..., 1] / z) / T.TAN_Y
    s_px = case.scales.double().numpy().max(1)[None] * T.FX / np.abs(z)
    c32 = con.numpy()
    det = c32[..., 0] * c32[..., 2] - c32[..., 1] * c32[..., 1]  # fp32, as tighten_tile_rect computes it
    needle = det <= np.float32(1e-4) * c32[..., 0] * c32[..., 2]
    op = case.opacities.numpy()[None]
    campos = torch.inverse(case.viewmats)[:, :3, 3]
    dirs = case.means[None] - campos[:, None]
    sh_neg = {}
    for deg in (0, 3):
        s = O.spherical_harmonics(deg, dirs, case.sh[None].expand(C, -1, -1, -1)) + 0.5
        sh_neg[deg] = (s < 0).any(-1).numpy()
    n_cams = vis.sum(0)
    q = case.quats.numpy()
    qn = np.linalg.norm(q, axis=1)
    return {
        "general": vis.any(),
        "near_plane": (vis & (z >= T.NEAR) & (z < 1.3 * T.NEAR)).any() and (~vis & (z > 0.7 * T.NEAR) & (z < T.NEAR)).any(),
        "behind": (~vis & (z < 0)).any(),
        "fov_clamped": (vis & (z > 0) & (np.maximum(ax, ay) > 1.35)).any(),
        "fov_inside": (vis & (z > 0) & (np.maximum(ax, ay) > 1.15) & (np.maximum(ax, ay) < 1.29)).any(),
        "off_screen": (~vis & (z > T.NEAR)).any(),
        "tiny": (vis & (s_px < 0.01)).any(),
        "huge": (vis & (radii.numpy() > max(T.W, T.H))).any(),
        "needle": (vis & needle).any(),
        "opacity_low": (vis & (op > 1 / 255.0) & (op < 1.02 / 255.0)).any(),
        "opacity_high": (vis & (op >= 0.999)).any(),
        "sh_clamped": (vis & sh_neg[0]).any() and (vis & sh_neg[3]).any(),
        "edge": ((n_cams > 0) & (n_cams < C)).any(),
        "quaternions": qn.min() < 0.3 and qn.max() > 3.0 and (q[:, 0] < 0).any(),
    }, vis


def _required(case):
    if case.N == 1:  # one Gaussian cannot hold several populations: it is simply visible
        return {"general"}
    req = set(T.POPULATIONS) | {"quaternions"}
    if case.C == 1:  # seen by some cameras only needs more than one
        req.discard("edge")
    return req


@pytest.mark.parametrize("ck", T.CASES, ids=T.case_id)
def test_every_case_holds_every_population(ck):
    case = T.make_case(*ck)
    present, vis = _census(case)
    missing = sorted(p for p in _required(case) if not present[p])
    assert not missing, f"{T.case_id(ck)}: populations missing {missing}"
    seen = vis.any(0)
    lay = case.layout
    if case.N >= 97:
        w = lambda i: seen[32 * i:32 * (i + 1)]
        assert not w(lay["empty_warp"]).any(), "a warp that sees nothing"
        assert w(lay["one_lane_warp"]).sum() == 1, "a warp with exactly one visible lane"
        last = w(lay["last_warp"])
        assert last[-1] and not last[:-1].any(), "the last warp: only its final lane visible"
    elif case.N > 32:
        assert seen[-1], "the last, partial warp's lane is visible"


def test_cases_are_reproducible():
    a, b = T.make_case(*T.CASES[4]), T.make_case(*T.CASES[4])
    for k in ("means", "quats", "scales", "opacities", "sh", "rgb", "rgb_cam", "viewmats", "Ks"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k


def _harness_forward(case, path, aa):
    """The forward outputs the kernels must produce, from the host-compiled math (what test_gpu_projection_paths
    compares the device with): the CPU stand-in for run_fwd."""
    d = dict(scales=case.scales, opacities=case.opacities, sh=case.sh[:, :path.K].contiguous())
    sc = T.harness_scene(case, d, path)
    h = hh.projection_fwd(sc, path.deg, T.EPS2D, T.NEAR, T.FAR, T.CLIP, T.TILE)
    out = {k: torch.from_numpy(v) for k, v in h.items()}
    if not aa:
        out.pop("compensations")
    return out, d


@pytest.mark.parametrize("aa", [False, True])
def test_fp64_reference_matches_the_host_math(aa):
    """ref64_bwd (fp64 autograd through the oracle) and harness_bwd must describe the same functional: the fp32 host
    math sits within 1e-4 of the fp64 reference on a case with every population."""
    ck = T.CASES[4]
    case = T.get_case(*ck)
    path = T.PATHS[3]  # K = 16, degree 3
    fwd, d = _harness_forward(case, path, aa)
    rec = T.records(case, fwd["radii"])
    extra = T.extra_grad(case)
    h = T.harness_bwd(case, d, path, aa, fwd, rec, extra)
    r64 = T.ref64_bwd(ck, path, aa, d, fwd, rec, extra, use_cache=False)
    h["v_opacities"] = T.v_opacities_ref(rec, fwd, aa)
    # needles lose their conic's determinant to fp32 cancellation (that is their point), so they are left out here
    keep = torch.tensor([lab != "needle" for lab in case.labels])
    for k in ("v_means", "v_quats", "v_scales", "v_sh", "v_opacities"):
        a, b = torch.as_tensor(np.asarray(h[k])).double()[keep], r64[k][keep]
        if k == "v_sh":
            a = a[:, :16]
        rel = ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
        assert rel <= 1e-4, (k, rel)
        assert b.abs().max() > 0, k


def test_tight_rect_reference_is_conservative_on_a_case():
    """The brute-force fp64 coverage check used on the device's rectangles, run on the host-compiled rectangles."""
    case = T.get_case(*T.CASES[4])
    path = T.PATHS[3]
    fwd, _ = _harness_forward(case, path, False)
    op = torch.where(fwd["radii"] > 0, case.opacities[None].expand(case.C, -1), torch.zeros(()))
    _, packed = hh.tight_rects(fwd["means2d"].reshape(-1, 2).numpy(), fwd["radii"].reshape(-1).numpy(),
                               fwd["conics"].reshape(-1, 3).numpy(), op.reshape(-1).numpy(), T.TW, T.TH, T.TILE)
    fwd["tight_rects"] = torch.from_numpy(packed).reshape(case.C, case.N, 2)
    T.check_tight_rects(None, fwd, op, "host", True)
    # and it does fail when a rectangle drops a reachable tile
    i = int(np.nonzero((fwd["radii"].reshape(-1) > 0).numpy() & (packed[:, 1] != 0))[0][0])
    shrunk = packed.copy()
    shrunk[i, 1] = 0
    fwd["tight_rects"] = torch.from_numpy(shrunk).reshape(case.C, case.N, 2)
    with pytest.raises(AssertionError):
        T.check_tight_rects(None, fwd, op, "host", True)


def test_v_opacities_reference_sums_in_camera_order():
    rec = torch.zeros(3, 2, 12)
    rec[:, 0, 5] = torch.tensor([1e8, 1.0, -1e8])
    out = T.v_opacities_ref(rec, None, False)
    assert out[0] == np.float32(0.0)  # (1e8 + 1) rounds to 1e8 in fp32 before the -1e8
    assert T.ulp_diff(np.float32([1.0]), np.float32([np.nextafter(np.float32(1), np.float32(2))]))[0] == 1
