"""CPU tests of the D-channel oracle (tests/features_oracle.py): a D-channel render is D one-channel renders side by
side, three channels reproduce oracle/gsplat_oracle.py's RGB render, D > 32 is blended in 32-channel chunks (geometry
gradients and absgrad summed over the chunks), and the blend's gradients w.r.t. colours and backgrounds pass an fp64
gradcheck."""
import torch

from easy_gaussian_splatting_b200.synthetic import make_scene
from oracle import gsplat_oracle as O
from tests import features_oracle as FO


def _scene(N=60, width=40, height=24, n_views=2, seed=3):
    return make_scene("blob", N, width, height, 40.0, seed, n_views=n_views)


def _render(sc, colors, bg=None, absgrad=False, grad=True, dtype=torch.float64, mode="classic"):
    leaves = [t.detach().to(dtype).requires_grad_(grad) for t in (sc.means, sc.quats, sc.scales, sc.opacities)]
    cols = colors.detach().to(dtype).requires_grad_(grad)
    bgs = None if bg is None else bg.detach().to(dtype).requires_grad_(grad)
    rc, ra, meta = FO.rasterization_features(*leaves, cols, sc.viewmats.to(dtype), sc.Ks.to(dtype), sc.width, sc.height,
                                   sh_degree=None, packed=False, absgrad=absgrad, backgrounds=bgs, rasterize_mode=mode)
    return rc, ra, meta, leaves, cols, bgs


def test_d_channels_equal_per_channel_renders():
    sc = _scene()
    C, N, D = 2, sc.means.shape[0], 5
    g = torch.Generator().manual_seed(0)
    feats = torch.rand(C, N, D, generator=g)
    bg = torch.rand(C, D, generator=g)
    rc, ra, _, _, _, _ = _render(sc, feats, bg, grad=False)
    assert rc.shape == (C, sc.height, sc.width, D) and ra.shape == (C, sc.height, sc.width, 1)
    for k in range(D):
        rk, ak, _, _, _, _ = _render(sc, feats[..., k:k + 1], bg[:, k:k + 1], grad=False)
        assert torch.equal(ak, ra)
        torch.testing.assert_close(rk, rc[..., k:k + 1], rtol=1e-12, atol=1e-12)
    # three channels through the D-channel code are the RGB render
    r3, a3, _, _, _, _ = _render(sc, feats[..., :3], bg[:, :3], grad=False)
    torch.testing.assert_close(r3, rc[..., :3], rtol=1e-12, atol=1e-12)


def test_forty_channels_are_a_32_and_an_8_channel_chunk():
    sc = _scene()
    C, N, D = 2, sc.means.shape[0], 40
    g = torch.Generator().manual_seed(1)
    feats = torch.rand(N, D, generator=g)
    bg = torch.rand(C, D, generator=g)
    Wc = torch.rand(C, sc.height, sc.width, D, generator=g, dtype=torch.float64)
    Wa = torch.rand(C, sc.height, sc.width, 1, generator=g, dtype=torch.float64)

    rc, ra, meta, leaves, cols, bgs = _render(sc, feats, bg, absgrad=True)
    ((rc * Wc).sum() + (ra * Wa).sum()).backward()

    parts = []
    for lo, hi, with_alpha in ((0, 32, True), (32, 40, False)):
        r, a, m, lv, cl, b = _render(sc, feats[:, lo:hi], bg[:, lo:hi], absgrad=True)
        loss = (r * Wc[..., lo:hi]).sum() + ((a * Wa).sum() if with_alpha else 0.0)
        loss.backward()
        parts.append((r, a, m, lv, cl, b))
    torch.testing.assert_close(rc, torch.cat([parts[0][0], parts[1][0]], -1), rtol=0, atol=0)
    assert torch.equal(ra, parts[0][1]) and torch.equal(ra, parts[1][1])
    for i in range(4):  # means, quats, scales, opacities: summed over the chunks
        torch.testing.assert_close(leaves[i].grad, parts[0][3][i].grad + parts[1][3][i].grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(cols.grad, torch.cat([parts[0][4].grad, parts[1][4].grad], -1), rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(bgs.grad, torch.cat([parts[0][5].grad, parts[1][5].grad], -1), rtol=1e-12, atol=1e-14)
    absgrad = meta["means2d"].absgrad
    assert absgrad.abs().sum() > 0
    torch.testing.assert_close(absgrad, parts[0][2]["means2d"].absgrad + parts[1][2]["means2d"].absgrad,
                               rtol=1e-12, atol=1e-14)


def test_single_chunk_absgrad_is_per_pixel_abs_over_all_channels():
    """D <= 32: one chunk, so absgrad sums |d loss / d means2d| per pixel over all channels together (gsplat's)."""
    sc = _scene(n_views=1)
    N = sc.means.shape[0]
    feats = torch.rand(N, 7, generator=torch.Generator().manual_seed(2))
    rc, ra, meta, leaves, _, _ = _render(sc, feats, absgrad=True)
    W = torch.rand(rc.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64) - 0.5
    meta["means2d"].retain_grad()
    (rc * W).sum().backward()
    ag = meta["means2d"].absgrad
    assert ag.shape == (1, N, 2) and ag.abs().sum() > 0
    # a sum of per-pixel absolute values bounds the absolute value of the plain gradient
    assert torch.all(ag + 1e-12 >= meta["means2d"].grad.abs())


def test_gradcheck_features_and_backgrounds():
    sc = _scene(N=8, width=16, height=16, n_views=2, seed=5)
    C, N, D = 2, 8, 3 + 2
    g = torch.Generator().manual_seed(4)
    feats = torch.rand(C, N, D, generator=g, dtype=torch.float64).requires_grad_(True)
    bg = torch.rand(C, D, generator=g, dtype=torch.float64).requires_grad_(True)
    fixed = [t.double() for t in (sc.means, sc.quats, sc.scales, sc.opacities)]

    def f(cols, bgs):
        rc, ra, _ = FO.rasterization_features(*fixed, cols, sc.viewmats.double(), sc.Ks.double(), sc.width, sc.height,
                                    sh_degree=None, packed=False, backgrounds=bgs)
        return rc

    assert f(feats, bg).shape == (C, 16, 16, D)
    assert torch.autograd.gradcheck(f, (feats, bg), eps=1e-6, atol=1e-7)


def test_three_channels_reproduce_the_rgb_oracle():
    """D = 3 through the D-channel tile loop equals oracle/gsplat_oracle.py's RGB blend: images, alphas, last_ids,
    gradients and absgrad."""
    sc = _scene()
    C, N = 2, sc.means.shape[0]
    g = torch.Generator().manual_seed(6)
    feats = torch.rand(C, N, 3, generator=g, dtype=torch.float64)
    bg = torch.rand(C, 3, generator=g, dtype=torch.float64)
    W = torch.rand(C, sc.height, sc.width, 3, generator=g, dtype=torch.float64)
    outs = []
    for fn in (O.rasterization, FO.rasterization_features):
        leaves = [t.detach().double().requires_grad_(True) for t in (sc.means, sc.quats, sc.scales, sc.opacities)]
        cols, bgs = feats.clone().requires_grad_(True), bg.clone().requires_grad_(True)
        rc, ra, meta = fn(*leaves, cols, sc.viewmats.double(), sc.Ks.double(), sc.width, sc.height, sh_degree=None,
                          packed=False, backgrounds=bgs, absgrad=True)
        ((rc * W).sum() + ra.sum()).backward()
        outs.append([rc, ra, meta["last_ids"], meta["means2d"].absgrad, cols.grad, bgs.grad] + [t.grad for t in leaves])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
