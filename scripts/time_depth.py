"""What the expected-depth render modes cost: forward + backward of one rasterization() call on the benchmark's metric
scene (1 M Gaussians, 1920 x 1080, 4 views per call, SH degree 3, a random linear functional of the images and the
alphas) in render_mode "RGB", "RGB+ED" and "ED", alternated in one run and timed with CUDA events.  Also times the blend
forward and backward stages alone on the same lists, with and without the depth channel (stages.rasterize_fwd / _bwd
against rasterize_fwd_depth / _bwd_depth).

The depth channel costs, per accepted (pixel, Gaussian) pair, one more FFMA2 forward and two more packed ops backward,
plus one more reduced value and one more RED per Gaussian per warp.

``python scripts/time_depth.py [--iters 20] [--warmup 3] [--views 4] [--out DIR]``

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
MODES = ("RGB", "RGB+ED", "ED")
STAGES = ("blend fwd", "blend fwd DEPTH", "blend bwd", "blend bwd DEPTH")


def _timed(fn):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1)


def _alternated(fn, variants, iters, warmup):
    for _ in range(warmup):
        for v in variants:
            fn(v)
    times = {v: [] for v in variants}
    for i in range(iters):
        order = variants if i % 2 == 0 else variants[::-1]
        for v in order:
            times[v].append(_timed(lambda: fn(v)))
    return times


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
    params = {k: getattr(sc, k).clone().requires_grad_(True) for k in (*GEOM, "colors")}
    weights = {m: torch.rand(C, sc.height, sc.width, {"RGB": 3, "RGB+ED": 4, "ED": 1}[m], device="cuda", generator=g)
               for m in MODES}
    Wa = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)

    def step(m):
        for p in params.values():
            p.grad = None
        rc, ra, _ = rasterization(*[params[k] for k in (*GEOM, "colors")], sc.viewmats, sc.Ks, sc.width, sc.height,
                                  sh_degree=3, packed=False, absgrad=True, render_mode=m)
        ((rc * weights[m]).sum() + (ra * Wa).sum()).backward()

    times = _alternated(step, MODES, a.iters, a.warmup)

    d = sc  # the blend stages alone, on one binning result
    with torch.no_grad():
        proj = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, d.colors, d.viewmats, d.Ks, sc.width,
                                     sc.height, 3)
        tw, th = stages.tile_grid(sc.width, sc.height)
        _, flat, offs = stages.isect_sorted(proj["means2d"], proj["radii"], proj["depths"], proj["tiles_per_gauss"], 16,
                                            tw, th)
        splats, bg = proj["splats"], None
        rc, ra, last = stages.rasterize_fwd(splats, offs, flat, bg, sc.width, sc.height)
        v_c3 = torch.rand(C, sc.height, sc.width, 3, device="cuda", generator=g)
        v_c4 = torch.rand(C, sc.height, sc.width, 4, device="cuda", generator=g)

        def stage(v):
            if v == "blend fwd":
                stages.rasterize_fwd(splats, offs, flat, bg, sc.width, sc.height)
            elif v == "blend fwd DEPTH":
                stages.rasterize_fwd_depth(splats, offs, flat, bg, sc.width, sc.height)
            elif v == "blend bwd":
                stages.rasterize_bwd(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_c3, Wa)
            else:
                stages.rasterize_bwd_depth(splats, offs, flat, bg, sc.width, sc.height, ra, last, v_c4, Wa)

        stage_times = _alternated(stage, STAGES, a.iters, a.warmup)

    res = dict(gpu_info(), scene="metric", n_gaussians=N, width=sc.width, height=sc.height, views_per_call=C,
               n_isects=int(flat.numel()), iters=a.iters,
               fwd_bwd_ms_median={m: statistics.median(times[m]) for m in MODES},
               fwd_bwd_ms_min={m: min(times[m]) for m in MODES},
               blend_stage_ms_median={v: statistics.median(stage_times[v]) for v in STAGES},
               blend_stage_ms_min={v: min(stage_times[v]) for v in STAGES})
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_depth.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
