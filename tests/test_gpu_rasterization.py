"""-m gpu: the whole boundary call `rasterization()` against the CPU oracle, plus API contract checks
(/root/reference/model/gaussian.py:353-374 call contract, :188-197 consumer semantics)."""
import pytest
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from tests.util import PARAMS, cuda_run, image_report, oracle_run, rel_err

pytestmark = pytest.mark.gpu

CASES = [
    dict(kind="blob", N=10_000, width=256, height=256, fx=274.5, seed=0, n_views=1),               # BASELINE cfg1
    dict(kind="blob", N=2_000, width=131, height=77, fx=120.0, seed=7, n_views=3),                  # C=3, ragged
    dict(kind="object", N=20_000, width=400, height=400, fx=555.0, seed=1, n_views=1, white_background=True),
    dict(kind="outdoor", N=60_000, width=489, height=273, fx=290.0, seed=2, n_views=1),             # cfg3-shaped, scaled
]


@pytest.mark.parametrize("cfg", CASES)
@pytest.mark.parametrize("sh_degree", [3, 1])
def test_end_to_end_parity(cfg, sh_degree):
    sc = make_scene(**cfg)
    ref = oracle_run(sc, sh_degree=sh_degree)
    out = cuda_run(sc, sh_degree=sh_degree)
    m, mo = out["meta"], ref["meta"]
    # bit-exact integer / index outputs
    assert torch.equal(m["radii"].cpu(), mo["radii"])
    assert torch.equal(m["tiles_per_gauss"].cpu(), mo["tiles_per_gauss"])
    assert torch.equal(m["isect_ids"].cpu(), mo["isect_ids"])
    assert torch.equal(m["flatten_ids"].cpu(), mo["flatten_ids"])
    assert torch.equal(m["isect_offsets"].cpu(), mo["isect_offsets"])
    assert torch.equal(m["means2d"].detach().cpu(), mo["means2d"].detach())
    assert torch.equal(m["depths"].cpu(), mo["depths"].detach())
    border = ref["counters"]["borderline"]
    rep_c = image_report(out["colors"], ref["colors"], border)
    rep_a = image_report(out["alphas"], ref["alphas"], border)
    print("colours", rep_c, "alphas", rep_a)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4  # north_star: 1e-4 absolute
    assert rep_c["max_border"] <= 2e-2
    errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in PARAMS}
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"])
    print("grad rel errs", errs)
    assert all(e <= 1e-3 for e in errs.values()), errs  # north_star: 1e-3 relative


def test_meta_contract_and_absgrad_tagging():
    from easy_gaussian_splatting_b200 import rasterization
    sc = make_scene("blob", 2000, 96, 64, 100.0, 3).to("cuda")
    p = {k: getattr(sc, k).clone().requires_grad_(True) for k in PARAMS}
    rc, ra, meta = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], p["colors"], sc.viewmats, sc.Ks,
                                 sc.width, sc.height, sh_degree=3, backgrounds=sc.background[None], absgrad=True, packed=False)
    N = sc.means.shape[0]
    assert rc.shape == (1, 64, 96, 3) and ra.shape == (1, 64, 96, 1)
    assert meta["radii"].shape == (1, N) and meta["radii"].dtype == torch.int32
    assert meta["means2d"].shape == (1, N, 2) and meta["means2d"].dtype == torch.float32
    assert not hasattr(meta["means2d"], "absgrad")
    batch_xys = meta["means2d"]  # the reference keeps this exact object (gaussian.py:371)
    torch.clamp(rc[0], 0.0, 1.0).mean().backward()
    assert hasattr(batch_xys, "absgrad") and batch_xys.absgrad.shape == (1, N, 2)
    assert (batch_xys.absgrad >= 0).all()
    vis = meta["radii"][0] > 0
    assert batch_xys.absgrad[0][~vis].abs().sum() == 0
    for k in PARAMS:
        assert p[k].grad is not None and torch.isfinite(p[k].grad).all()
    assert p["means"].grad[~vis].abs().sum() == 0
    # no_grad: nothing recorded, no absgrad attribute
    with torch.no_grad():
        rc2, ra2, meta2 = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], p["colors"], sc.viewmats,
                                        sc.Ks, sc.width, sc.height, sh_degree=3, backgrounds=sc.background[None],
                                        absgrad=True, packed=False)
    assert rc2.grad_fn is None and not hasattr(meta2["means2d"], "absgrad")
    assert torch.equal(rc2, rc.detach())  # forward is deterministic


@pytest.mark.parametrize("W,H", [(1, 1), (17, 1), (1, 33), (16, 16), (250, 3)])
def test_viewer_edge_sizes(W, H):
    """viewer can request any W,H >= 1 (viewer_runtime.py:225,232)"""
    sc = make_scene("blob", 500, W, H, 50.0, 11)
    ref = oracle_run(sc, backward=True)
    out = cuda_run(sc, backward=True)
    assert torch.equal(out["meta"]["radii"].cpu(), ref["meta"]["radii"])
    assert torch.equal(out["meta"]["flatten_ids"].cpu(), ref["meta"]["flatten_ids"])
    border = ref["counters"]["borderline"]
    assert image_report(out["colors"], ref["colors"], border)["max_clean"] <= 1e-4
    for k in PARAMS:
        assert rel_err(out["grads"][k], ref["grads"][k]) <= 1e-3 or ref["grads"][k].abs().max() < 1e-12


def test_degenerate_cameras_and_empty():
    """fx = inf / ~0 (viewer fov 0 / 180 deg, viewer/utils.py:10-11), everything behind the camera, N = 0."""
    from easy_gaussian_splatting_b200 import rasterization
    sc = make_scene("blob", 300, 64, 48, 60.0, 5).to("cuda")
    args = lambda K: (sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, sc.viewmats, K, sc.width, sc.height)
    for fx in (float("inf"), 1e-30, float("nan")):
        K = sc.Ks.clone()
        K[:, 0, 0] = fx
        K[:, 1, 1] = fx
        rc, ra, meta = rasterization(*args(K), sh_degree=3, packed=False, backgrounds=sc.background[None])
        torch.cuda.synchronize()
        assert torch.isfinite(rc).all()
    V = sc.viewmats.clone()
    V[:, 2, 3] -= 100.0  # push everything behind the near plane
    rc, ra, meta = rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, V, sc.Ks, sc.width, sc.height,
                                 sh_degree=3, packed=False, backgrounds=torch.ones(1, 3, device="cuda"))
    assert int(meta["radii"].sum()) == 0 and meta["flatten_ids"].numel() == 0
    assert torch.equal(rc, torch.ones_like(rc)) and float(ra.abs().sum()) == 0
    e = lambda *s: torch.zeros(*s, device="cuda")
    rc, ra, meta = rasterization(e(0, 3), e(0, 4), e(0, 3), e(0), e(0, 16, 3), sc.viewmats, sc.Ks, 32, 32, sh_degree=3, packed=False)
    assert rc.shape == (1, 32, 32, 3) and float(rc.abs().sum()) == 0


def test_direct_colors_and_unsupported_modes():
    from easy_gaussian_splatting_b200 import rasterization
    sc = make_scene("blob", 1500, 80, 60, 90.0, 9)
    from oracle import gsplat_oracle as O
    cols = torch.rand(1500, 3, generator=torch.Generator().manual_seed(1))
    rc_o, ra_o, _ = O.rasterization(sc.means, sc.quats, sc.scales, sc.opacities, cols, sc.viewmats, sc.Ks, 80, 60, sh_degree=None, packed=False)
    d = sc.to("cuda")
    rc, ra, _ = rasterization(d.means, d.quats, d.scales, d.opacities, cols.cuda(), d.viewmats, d.Ks, 80, 60, sh_degree=None, packed=False)
    assert (rc.cpu() - rc_o).abs().max() <= 1e-4 + 1e-2 * 0  # tiny scene: no borderline pixels expected
    for kw in (dict(render_mode="RGB+D"), dict(sparse_grad=True), dict(tile_size=8)):
        base = dict(sh_degree=3, packed=False)
        base.update(kw)
        with pytest.raises(NotImplementedError):
            rasterization(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, 80, 60, **base)
    with pytest.raises(RuntimeError):
        rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, sc.viewmats, sc.Ks, 80, 60, sh_degree=3, packed=False)


@pytest.mark.parametrize("cfg", [CASES[0], CASES[1], CASES[3]])
def test_antialiased_mode_parity(cfg):
    """SURVEY.md §8f-4: rasterize_mode="antialiased" (opacity * sqrt(det_orig / det_blur)) against the oracle."""
    sc = make_scene(**cfg)
    ref = oracle_run(sc, rasterize_mode="antialiased")
    out = cuda_run(sc, rasterize_mode="antialiased")
    m, mo = out["meta"], ref["meta"]
    for k in ("radii", "flatten_ids", "isect_offsets"):
        assert torch.equal(m[k].cpu(), mo[k])
    assert torch.equal(m["opacities"].cpu(), mo["opacities"].detach())  # opacity * compensation, bit-exact
    vis = mo["radii"] > 0
    assert float(mo["opacities"][vis].max()) < float(sc.opacities.max()) + 1e-6
    border = ref["counters"]["borderline"]
    rep_c = image_report(out["colors"], ref["colors"], border)
    rep_a = image_report(out["alphas"], ref["alphas"], border)
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in PARAMS}
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"])
    print("grad rel errs", errs)
    assert all(e <= 1e-3 for e in errs.values()), errs
    # and it is a different image from the classic mode (the factor is < 1 for every visible Gaussian)
    classic = cuda_run(sc, backward=False)
    assert (classic["alphas"] - out["alphas"]).abs().max() > 1e-3


@pytest.mark.parametrize("cfg", [CASES[1], CASES[3]])
@pytest.mark.parametrize("mode", ["classic", "antialiased"])
def test_packed_mode_matches_dense(cfg, mode):
    """SURVEY.md §8f-4: packed=True returns gsplat's packed layout (nnz visible (camera, Gaussian) entries in flat
    order, camera_ids / gaussian_ids, flatten_ids into the packed list); images and gradients equal the dense call."""
    sc = make_scene(**cfg)
    dense = cuda_run(sc, rasterize_mode=mode)
    pk = cuda_run(sc, rasterize_mode=mode, packed=True)
    assert torch.equal(pk["colors"], dense["colors"]) and torch.equal(pk["alphas"], dense["alphas"])
    md, mp = dense["meta"], pk["meta"]
    C, N = md["radii"].shape
    vis = md["radii"] > 0
    cam, gid = vis.nonzero(as_tuple=True)
    nnz = cam.numel()
    assert torch.equal(mp["camera_ids"], cam) and torch.equal(mp["gaussian_ids"], gid)
    assert mp["radii"].shape == (nnz,) and mp["means2d"].shape == (nnz, 2) and mp["conics"].shape == (nnz, 3)
    for k in ("radii", "depths", "tiles_per_gauss", "opacities"):
        assert torch.equal(mp[k], md[k][vis]), k
    for k in ("means2d", "conics", "colors"):
        assert torch.equal(mp[k].detach(), md[k].detach()[vis]), k
    assert torch.equal(mp["isect_ids"], md["isect_ids"]) and torch.equal(mp["isect_offsets"], md["isect_offsets"])
    flat = cam * N + gid
    assert torch.equal(flat[mp["flatten_ids"].long()].int(), md["flatten_ids"])
    assert pk["absgrad"].shape == (nnz, 2) and rel_err(pk["absgrad"], dense["absgrad"][vis.cpu()]) <= 1e-5
    for k in PARAMS:  # same kernels, same inputs: only the atomic order differs
        assert rel_err(pk["grads"][k], dense["grads"][k]) <= 1e-5, k


@pytest.mark.parametrize("cfg", [CASES[1], CASES[2], CASES[3]])
@pytest.mark.parametrize("segment", [64, 192, 1024])
def test_segmented_backward_matches_unsegmented(cfg, segment, monkeypatch):
    """Long tile lists are replayed by one warp per `segment` entries, starting from forward checkpoints
    (include/egs_raster.h, egs_rasterize_bwd_segmented).  Same images bit for bit, same gradients up to fp32
    summation order, for segment lengths from one batch (every list is segmented) to the default."""
    sc = make_scene(**cfg)
    monkeypatch.setenv("EGS_BWD_SEGMENT", "0")
    base = cuda_run(sc)
    monkeypatch.setenv("EGS_BWD_SEGMENT", str(segment))
    seg = cuda_run(sc)
    assert torch.equal(seg["colors"], base["colors"]) and torch.equal(seg["alphas"], base["alphas"])
    n_long = int(((base["meta"]["isect_offsets"].flatten()[1:] - base["meta"]["isect_offsets"].flatten()[:-1]) > segment).sum())
    print("tiles longer than", segment, ":", n_long)
    if segment == 64:
        assert n_long > 0  # the test must exercise the segment launch
    for k in PARAMS:
        assert rel_err(seg["grads"][k], base["grads"][k]) <= 2e-5, k
    assert rel_err(seg["absgrad"], base["absgrad"]) <= 2e-5
    ref = oracle_run(sc)
    for k in PARAMS:
        assert rel_err(seg["grads"][k], ref["grads"][k]) <= 1e-3, k


GOLDEN = sorted(__import__("pathlib").Path(__file__).parent.glob("golden/*.npz"))


@pytest.mark.parametrize("path", GOLDEN, ids=[p.stem for p in GOLDEN])
def test_cuda_matches_committed_golden_vectors(path):
    """CUDA path against the frozen fixtures (tests/golden/make_golden.py) — no oracle execution involved."""
    import numpy as np
    from easy_gaussian_splatting_b200 import rasterization
    g = np.load(path)
    t = lambda k: torch.from_numpy(g[k]).cuda()
    p = {k: t(f"in_{k}").clone().requires_grad_(True) for k in PARAMS}
    W, H, deg = int(g["in_width"]), int(g["in_height"]), int(g["in_sh_degree"])
    rc, ra, meta = rasterization(p["means"], p["quats"], p["scales"], p["opacities"], p["colors"], t("in_viewmats"),
                                 t("in_Ks"), W, H, sh_degree=deg, packed=False, absgrad=True, backgrounds=t("in_background"),
                                 rasterize_mode="antialiased" if "in_antialiased" in g else "classic")
    ((rc * t("in_Wc")).sum() + (ra * t("in_Wa")).sum()).backward()
    if "in_antialiased" in g:
        assert torch.equal(meta["opacities"].cpu(), torch.from_numpy(g["opacities"]))
    for k in ("radii", "tiles_per_gauss", "isect_ids", "flatten_ids", "isect_offsets"):
        assert torch.equal(meta[k].cpu(), torch.from_numpy(g[k])), k
    assert torch.equal(meta["means2d"].detach().cpu(), torch.from_numpy(g["means2d"]))
    assert torch.equal(meta["depths"].cpu(), torch.from_numpy(g["depths"]))
    assert torch.equal(meta["conics"].cpu(), torch.from_numpy(g["conics"]))
    border = torch.from_numpy(g["borderline"])
    assert image_report(rc.detach().cpu(), torch.from_numpy(g["render_colors"]), border)["max_clean"] <= 1e-4
    assert image_report(ra.detach().cpu(), torch.from_numpy(g["render_alphas"]), border)["max_clean"] <= 1e-4
    for k in PARAMS:
        assert rel_err(p[k].grad.cpu(), torch.from_numpy(g[f"grad_{k}"])) <= 1e-3, k
    assert rel_err(meta["means2d"].absgrad.cpu(), torch.from_numpy(g["absgrad"])) <= 1e-3


def _pile_scene(n=6000, seed=5):
    """Thousands of faint Gaussians stacked in one or two tiles: exercises the long-tile (8 warps per tile) launch."""
    sc = make_scene("blob", n, 160, 96, 200.0, seed)
    g = torch.Generator().manual_seed(seed)
    sc.means = (torch.randn(n, 3, generator=g) * torch.tensor([0.03, 0.03, 0.3])).contiguous()
    sc.scales = torch.exp(torch.log(torch.tensor(0.01)) + 0.3 * torch.randn(n, 3, generator=g)).contiguous()
    sc.opacities = (0.004 + 0.05 * torch.rand(n, generator=g)).contiguous()
    return sc


def test_long_tile_parity():
    """A pile of faint Gaussians behind one another: tiles with thousands of entries of which almost every one is
    blended (no early termination) — the long-list case of the blend kernels, default settings."""
    sc = _pile_scene()
    ref = oracle_run(sc)
    offs = ref["meta"]["isect_offsets"].reshape(-1).long()
    n = ref["meta"]["flatten_ids"].numel()
    lens = torch.diff(torch.cat([offs, torch.tensor([n])]))
    assert int(lens.max()) > 2048, "scene must contain long tile lists"
    out = cuda_run(sc)
    assert torch.equal(out["meta"]["flatten_ids"].cpu(), ref["meta"]["flatten_ids"])
    border = ref["counters"]["borderline"]
    rep_c = image_report(out["colors"], ref["colors"], border)
    rep_a = image_report(out["alphas"], ref["alphas"], border)
    print(rep_c, rep_a, "max tile", int(lens.max()))
    assert rep_c["max_clean"] <= 1e-4 and rep_a["max_clean"] <= 1e-4
    errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in PARAMS}
    errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"])
    assert all(e <= 1e-3 for e in errs.values()), errs


def test_view_pipeline_matches_sequential_accumulation():
    """training.ViewPipeline (two alternating streams) must accumulate the same gradients and statistics as a
    plain sequential loop over the views."""
    from easy_gaussian_splatting_b200.distributed import DensifyStats, FlatGradBucket
    from easy_gaussian_splatting_b200.training import ViewPipeline
    sc = make_scene("outdoor", 40_000, 320, 200, 200.0, 3, n_views=5).to("cuda")
    W, H = sc.width, sc.height
    g = torch.Generator().manual_seed(0)
    Wc, Wa = torch.rand(1, H, W, 3, generator=g).cuda(), torch.rand(1, H, W, 1, generator=g).cuda()
    results = []
    for enabled in (False, True):
        params = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
        bucket = FlatGradBucket(params)
        stats = DensifyStats(sc.means.shape[0], "cuda")
        pipe = ViewPipeline("cuda", enabled=enabled)
        for rep in range(2):  # two steps: stream reuse across steps
            bucket.zero_()
            pipe.fork()
            for v in range(sc.viewmats.shape[0]):
                pipe.render_backward(v, params, sc.viewmats[v:v + 1], sc.Ks[v:v + 1], W, H,
                                     lambda rc, ra: (rc * Wc).sum() + (ra * Wa).sum(), sh_degree=3,
                                     backgrounds=sc.background[None],
                                     after_backward=lambda meta: stats.update_local(meta["radii"], meta["means2d"].absgrad, W, H))
            pipe.join()
        torch.cuda.synchronize()
        results.append((bucket.flat.clone(), stats.buf.clone()))
    (g0, s0), (g1, s1) = results
    assert rel_err(g1.cpu(), g0.cpu()) <= 1e-5
    assert torch.equal(s0[1], s1[1]) and torch.equal(s0[2], s1[2])  # counts and max radii are exact
    assert rel_err(s1[0].cpu(), s0[0].cpu()) <= 1e-5


@pytest.mark.parametrize("sh_degree", [0, 2, 3])
def test_folded_activations_match_unfolded(sh_degree):
    """§8f-2: rasterization_from_parameters(raw params) == rasterization(exp, sigmoid, cat of them), forward and
    gradients w.r.t. the raw parameters (autograd through torch's exp / sigmoid / cat on the unfolded side)."""
    from easy_gaussian_splatting_b200 import rasterization, rasterization_from_parameters
    sc = make_scene("outdoor", 30_000, 320, 200, 200.0, 11, n_views=2).to("cuda")
    W, H = sc.width, sc.height
    raw = dict(means=sc.means, quats=sc.quats, log_scales=torch.log(sc.scales), logit_opacities=torch.logit(sc.opacities),
               sh_0=sc.colors[:, :1].contiguous(), sh_rest=sc.colors[:, 1:].contiguous())
    g = torch.Generator().manual_seed(2)
    Wc, Wa = torch.rand(2, H, W, 3, generator=g).cuda(), torch.rand(2, H, W, 1, generator=g).cuda()
    bg = sc.background[None].expand(2, 3).contiguous()

    a = {k: v.clone().requires_grad_(True) for k, v in raw.items()}
    rc_a, ra_a, meta_a = rasterization(a["means"], a["quats"], torch.exp(a["log_scales"]), torch.sigmoid(a["logit_opacities"]),
                                       torch.cat([a["sh_0"], a["sh_rest"]], 1), sc.viewmats, sc.Ks, W, H,
                                       sh_degree=sh_degree, packed=False, absgrad=True, backgrounds=bg)
    ((rc_a * Wc).sum() + (ra_a * Wa).sum()).backward()

    b = {k: v.clone().requires_grad_(True) for k, v in raw.items()}
    rc_b, ra_b, meta_b = rasterization_from_parameters(b["means"], b["quats"], b["log_scales"], b["logit_opacities"],
                                                       b["sh_0"], b["sh_rest"], sc.viewmats, sc.Ks, W, H, sh_degree,
                                                       backgrounds=bg, absgrad=True)
    ((rc_b * Wc).sum() + (ra_b * Wa).sum()).backward()

    assert torch.equal(meta_a["radii"], meta_b["radii"]) and torch.equal(meta_a["flatten_ids"], meta_b["flatten_ids"])
    assert torch.equal(meta_a["means2d"], meta_b["means2d"])
    assert float((rc_a - rc_b).abs().max()) <= 1e-6 and float((ra_a - ra_b).abs().max()) <= 1e-6
    for k in raw:
        assert rel_err(b[k].grad.cpu(), a[k].grad.cpu()) <= 1e-5, k
    assert rel_err(meta_b["means2d"].absgrad.cpu(), meta_a["means2d"].absgrad.cpu()) <= 1e-5
    nb = (sh_degree + 1) ** 2
    if nb < 16:
        assert float(b["sh_rest"].grad[:, nb - 1:].abs().sum()) == 0.0  # inactive bands get exactly zero


def test_direct_gradient_bucket():
    """FlatGradBucket.begin_direct(): the fused backward writes the gradients straight into the caller's flat bucket
    (param.grad becomes a view of it, no zero fill / accumulate pass) — same numbers as the ordinary route."""
    from easy_gaussian_splatting_b200 import rasterization
    from easy_gaussian_splatting_b200.distributed import FlatGradBucket
    from easy_gaussian_splatting_b200.synthetic import loss_weights
    sc = make_scene(**CASES[1]).to("cuda")
    C = sc.viewmats.shape[0]
    Wc, Wa = (t.cuda() for t in loss_weights(sc.seed, C, sc.height, sc.width))

    def run(params):
        rc, ra, _ = rasterization(*params, sc.viewmats, sc.Ks, sc.width, sc.height, sh_degree=3, packed=False,
                                  absgrad=True, backgrounds=sc.background[None].expand(C, 3).contiguous())
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()

    ref = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
    run(ref)
    params = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
    bucket = FlatGradBucket(params)
    bucket.flat.fill_(float("nan"))  # direct mode must overwrite every element without a zero fill
    bucket.begin_direct()
    run(params)
    direct_ptrs = [p.grad.data_ptr() for p in params]
    bucket.end_direct()
    assert direct_ptrs == [v.data_ptr() for v in bucket.views], "autograd did not adopt the bucket views"
    assert torch.isfinite(bucket.flat).all()
    for p, r, k in zip(params, ref, PARAMS):
        assert p.grad.data_ptr() == bucket.views[PARAMS.index(k)].data_ptr()
        assert rel_err(p.grad.cpu(), r.grad.cpu()) <= 1e-5, k
    # a second, ordinary backward accumulates on top (the registry is cleared)
    run(params)
    for p, r, k in zip(params, ref, PARAMS):
        assert rel_err(p.grad.cpu(), 2 * r.grad.cpu()) <= 1e-5, k


def test_non_contiguous_inputs_give_the_same_gradients():
    """ADVICE r1 (high): `viewmats = torch.linalg.inv(camtoworlds)` has strides (16, 1, 4), and a transposed `means`
    is column-major; forward AND backward must see dense copies, and gradients come back in the input's shape."""
    from easy_gaussian_splatting_b200 import rasterization
    from easy_gaussian_splatting_b200.synthetic import loss_weights
    sc = make_scene(**CASES[1]).to("cuda")
    C = sc.viewmats.shape[0]
    Wc, Wa = (t.cuda() for t in loss_weights(sc.seed, C, sc.height, sc.width))
    bg = sc.background[None].expand(C, 3)  # stride-0 expand, not made contiguous on purpose

    def run(params, viewmats, Ks):
        rc, ra, meta = rasterization(*params, viewmats, Ks, sc.width, sc.height, sh_degree=3, packed=False, absgrad=True,
                                     backgrounds=bg)
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()
        return rc.detach(), meta

    ref = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
    rc_ref, meta_ref = run(ref, sc.viewmats, sc.Ks)
    c2w = torch.linalg.inv(sc.viewmats)
    viewmats = torch.linalg.inv(c2w)  # the gsplat idiom; batch-of-column-major on CUDA
    odd = []
    for k in PARAMS:
        t = getattr(sc, k)
        if t.dim() >= 2:
            perm = list(range(t.dim()))[::-1]
            t2 = t.permute(*perm).contiguous().permute(*perm)  # same values, reversed strides
            assert not t2.is_contiguous()
        else:
            t2 = torch.stack([t, t], 1)[:, 0]  # stride 2
        odd.append(t2.detach().requires_grad_(True))
    Ks = torch.stack([sc.Ks, sc.Ks], 1)[:, 0]
    rc, meta = run(odd, viewmats, Ks)
    assert (viewmats - sc.viewmats).abs().max() < 1e-5
    assert torch.equal(meta["radii"], meta_ref["radii"]) or (meta["radii"] != meta_ref["radii"]).float().mean() < 1e-3
    for p, r, k in zip(odd, ref, PARAMS):
        assert p.grad.shape == r.grad.shape
        assert rel_err(p.grad.cpu(), r.grad.cpu()) <= 2e-3, k  # inv(inv(V)) differs from V in the last bits
    # exactly the same camera, strided: bit-identical forward, gradients to reduction-order noise
    vm_strided = torch.stack([sc.viewmats, sc.viewmats], 1)[:, 0]
    odd2 = [t.detach().clone(memory_format=torch.preserve_format).requires_grad_(True) for t in odd]
    rc2, _ = run(odd2, vm_strided, Ks)
    assert torch.equal(rc2, rc_ref)
    for p, r, k in zip(odd2, ref, PARAMS):
        assert rel_err(p.grad.cpu(), r.grad.cpu()) <= 1e-5, k


@pytest.mark.parametrize("n", [4001, 4002, 4003])
def test_direct_gradient_bucket_any_n(n):
    """ADVICE r1 (medium): N % 4 != 0 (any N after densify / prune) must not misalign the float4 gradient stores of the
    direct-to-bucket backward, on the activated-tensor path and on the raw-parameter path."""
    from easy_gaussian_splatting_b200 import rasterization, rasterization_from_parameters
    from easy_gaussian_splatting_b200.distributed import FlatGradBucket
    from easy_gaussian_splatting_b200.synthetic import loss_weights
    sc = make_scene("blob", n, 96, 80, 100.0, 21, n_views=2).to("cuda")
    C = sc.viewmats.shape[0]
    Wc, Wa = (t.cuda() for t in loss_weights(sc.seed, C, sc.height, sc.width))
    bg = sc.background[None].expand(C, 3).contiguous()

    def loss(rc, ra):
        return (rc * Wc).sum() + (ra * Wa).sum()

    ref = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
    rc, ra, _ = rasterization(*ref, sc.viewmats, sc.Ks, sc.width, sc.height, sh_degree=3, packed=False, absgrad=True, backgrounds=bg)
    loss(rc, ra).backward()
    params = [getattr(sc, k).clone().requires_grad_(True) for k in PARAMS]
    bucket = FlatGradBucket(params)
    bucket.flat.fill_(float("nan"))
    with bucket.direct():
        rc, ra, _ = rasterization(*params, sc.viewmats, sc.Ks, sc.width, sc.height, sh_degree=3, packed=False, absgrad=True, backgrounds=bg)
        loss(rc, ra).backward()
        adopted = [p.grad.data_ptr() for p in params]
    torch.cuda.synchronize()
    assert adopted == [v.data_ptr() for v in bucket.views]
    for p, r, k in zip(params, ref, PARAMS):
        assert torch.isfinite(p.grad).all() and rel_err(p.grad.cpu(), r.grad.cpu()) <= 1e-5, k
    # raw-parameter entry point: six tensors, sh_0 [N,1,3] and sh_rest [N,15,3] slices
    raw_src = [sc.means, sc.quats, torch.log(sc.scales), torch.logit(sc.opacities), sc.colors[:, :1].contiguous(), sc.colors[:, 1:].contiguous()]
    raw = [t.clone().requires_grad_(True) for t in raw_src]
    rbucket = FlatGradBucket(raw)
    rbucket.flat.fill_(float("nan"))
    with rbucket.direct():
        rc, ra, _ = rasterization_from_parameters(*raw, sc.viewmats, sc.Ks, sc.width, sc.height, 3, backgrounds=bg, absgrad=True)
        loss(rc, ra).backward()
        adopted = [p.grad.data_ptr() for p in raw]
    torch.cuda.synchronize()
    assert adopted == [v.data_ptr() for v in rbucket.views]
    assert rel_err(raw[0].grad.cpu(), ref[0].grad.cpu()) <= 1e-4 and rel_err(raw[1].grad.cpu(), ref[1].grad.cpu()) <= 1e-4
    assert rel_err(torch.cat([raw[4].grad, raw[5].grad], 1).cpu(), ref[4].grad.cpu()) <= 1e-4


def test_automatic_segmentation_from_the_previous_call(monkeypatch):
    """No environment knob: the second call of a shape knows (from the first) that the scene has outlier-long tile
    lists and replays them in segments; images, lists and gradients must not change."""
    from easy_gaussian_splatting_b200 import rendering, stages
    monkeypatch.delenv("EGS_BWD_SEGMENT", raising=False)
    sc = _pile_scene()
    ref = oracle_run(sc)
    stages.reset_binning_hints()
    used = []
    real = stages.segment_policy
    monkeypatch.setattr(stages, "segment_policy", lambda hint, n: used.append(real(hint, n)) or used[-1])
    first = cuda_run(sc)
    torch.cuda.synchronize()
    second = cuda_run(sc)
    assert used[0] == (0, 0), "first call of a shape: nothing known yet"
    assert used[1][0] == stages.SEGMENT_ENTRIES and used[1][1] >= stages.SEGMENT_MIN_ENTRIES, used
    border = ref["counters"]["borderline"]
    for out in (first, second):
        assert torch.equal(out["meta"]["flatten_ids"].cpu(), ref["meta"]["flatten_ids"])
        assert image_report(out["colors"], ref["colors"], border)["max_clean"] <= 1e-4
        errs = {k: rel_err(out["grads"][k], ref["grads"][k]) for k in PARAMS}
        errs["absgrad"] = rel_err(out["absgrad"], ref["absgrad"])
        assert all(e <= 1e-3 for e in errs.values()), errs
    assert torch.equal(first["colors"], second["colors"])
    # an ordinary scene of another shape keeps the plain path on its second call
    sc2 = make_scene(**CASES[3])
    cuda_run(sc2)
    torch.cuda.synchronize()
    cuda_run(sc2)
    assert used[-1] == (0, 0), used
