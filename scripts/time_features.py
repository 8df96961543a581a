"""What colours with D channels cost: forward + backward of one rasterization() call on the benchmark's metric scene
(1 M Gaussians, 1920 x 1080, 4 views per call, the functional sum(colors * Wc) + sum(alphas * Wa)) for D = 3 (the RGB
path, SH degree 0 colours given directly) and D = 1, 4, 8, 16, 32, 64 (the feature kernels), alternated in one run and
timed with CUDA events.  Also times the blend kernels alone on the same records and lists: the RGB kernels against
D = 3 through the feature entries (CH = 4), which prices the generic path.

``python scripts/time_features.py [--iters 20] [--warmup 3] [--views 4] [--out DIR]``

Prints the GPU name and power limit next to the times."""
import argparse
import json
import os
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from easy_gaussian_splatting_b200 import rasterization, stages  # noqa: E402
from easy_gaussian_splatting_b200.synthetic import make_config_scene  # noqa: E402
from scripts.time_viewmat_grad import gpu_info  # noqa: E402

GEOM = ("means", "quats", "scales", "opacities")
WIDTHS = (3, 1, 4, 8, 16, 32, 64)


def _timed(fn):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--views", type=int, default=4)
    ap.add_argument("--out", default=None, help="directory for a JSON copy of the result")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script times the GPU")
    sc = make_config_scene("metric", n_views=a.views).to("cuda")
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    g = torch.Generator(device="cuda").manual_seed(0)
    params = {k: getattr(sc, k).clone().requires_grad_(True) for k in GEOM}
    cols = {D: (torch.rand(N, D, device="cuda", generator=g)).requires_grad_(True) for D in WIDTHS}
    Wc = {D: torch.rand(C, sc.height, sc.width, D, device="cuda", generator=g) for D in WIDTHS}
    Wa = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)

    def step(D):
        for p in list(params.values()) + [cols[D]]:
            p.grad = None
        rc, ra, _ = rasterization(params["means"], params["quats"], params["scales"], params["opacities"], cols[D],
                                  sc.viewmats, sc.Ks, sc.width, sc.height, packed=False, absgrad=True)
        ((rc * Wc[D]).sum() + (ra * Wa).sum()).backward()

    for _ in range(a.warmup):
        for D in WIDTHS:
            step(D)
    times = {D: [] for D in WIDTHS}
    for i in range(a.iters):
        for D in (WIDTHS if i % 2 == 0 else WIDTHS[::-1]):
            times[D].append(_timed(lambda: step(D)))

    # blend kernels alone: RGB kernels vs D = 3 through the feature entries, on the same records and lists
    d = sc
    rgb = cols[3].detach()
    with torch.no_grad():
        proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, rgb, d.viewmats, d.Ks, sc.width, sc.height, None)
        tw, th = stages.tile_grid(sc.width, sc.height)
        _, flat, offs = stages.isect_sorted(proj["means2d"], proj["radii"], proj["depths"], proj["tiles_per_gauss"], 16,
                                            tw, th)
        sp = proj["splats"]
        v_c = torch.rand(C, sc.height, sc.width, 3, device="cuda", generator=g)
        v_a = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)

        def blend_rgb():
            _, ra, last = stages.rasterize_fwd(sp, offs, flat, None, sc.width, sc.height)
            stages.rasterize_bwd(sp, offs, flat, None, sc.width, sc.height, ra, last, v_c, v_a)

        def blend_feat():
            _, ra, last = stages.rasterize_fwd_features(sp, offs, flat, rgb, None, sc.width, sc.height)
            stages.rasterize_bwd_features(sp, offs, flat, rgb, None, sc.width, sc.height, ra, last, v_c, v_a)

        for _ in range(a.warmup):
            blend_rgb(), blend_feat()
        blend = {"rgb_kernels": [], "feature_kernels_d3": []}
        for i in range(a.iters):
            order = (("rgb_kernels", blend_rgb), ("feature_kernels_d3", blend_feat))
            for name, fn in (order if i % 2 == 0 else order[::-1]):
                blend[name].append(_timed(fn))

    res = dict(gpu_info(), scene="metric", n_gaussians=N, width=sc.width, height=sc.height, views_per_call=C,
               iters=a.iters,
               fwd_bwd_ms_median={("D=3 (RGB path)" if D == 3 else f"D={D}"): statistics.median(times[D]) for D in WIDTHS},
               fwd_bwd_ms_min={("D=3 (RGB path)" if D == 3 else f"D={D}"): min(times[D]) for D in WIDTHS},
               blend_fwd_bwd_ms_median={k: statistics.median(v) for k, v in blend.items()})
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_features.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
