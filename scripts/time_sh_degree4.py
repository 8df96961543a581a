"""What SH degree 4 costs: forward + backward of one rasterization() call on the benchmark's metric scene (1 M
Gaussians, 1920 x 1080, 4 views per call, the functional sum(colors * Wc) + sum(alphas * Wa)) at degree 3 with
[N,16,3] coefficients against degree 4 with [N,25,3] and per-camera [C,N,25,3] coefficients, alternated in one run and
timed with CUDA events.  Also times the projection forward + backward stages alone on the same records.

Degree 4 reads 300 B instead of 192 B of coefficients per visible pair forward and moves 2 x 300 B instead of 2 x 192 B
of coefficient and gradient rows per Gaussian backward.

``python scripts/time_sh_degree4.py [--iters 20] [--warmup 3] [--views 4] [--out DIR]``

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
VARIANTS = ("degree 3 [N,16,3]", "degree 4 [N,25,3]", "degree 4 per-camera [C,N,25,3]")
DEGREE = dict(zip(VARIANTS, (3, 4, 4)))


def _timed(fn):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1)


def _alternated(fn, iters, warmup):
    for _ in range(warmup):
        for v in VARIANTS:
            fn(v)
    times = {v: [] for v in VARIANTS}
    for i in range(iters):
        order = VARIANTS if i % 2 == 0 else VARIANTS[::-1]
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
    params = {k: getattr(sc, k).clone().requires_grad_(True) for k in GEOM}
    sh25 = torch.cat([sc.colors, 0.05 * torch.randn(N, 9, 3, device="cuda", generator=g)], 1)
    sh25_pc = sh25[None] + 0.05 * torch.randn(C, N, 25, 3, device="cuda", generator=g)
    cols = {v: t.contiguous().requires_grad_(True) for v, t in zip(VARIANTS, (sc.colors.clone(), sh25, sh25_pc))}
    Wc = torch.rand(C, sc.height, sc.width, 3, device="cuda", generator=g)
    Wa = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)

    def step(v):
        for p in list(params.values()) + [cols[v]]:
            p.grad = None
        rc, ra, _ = rasterization(params["means"], params["quats"], params["scales"], params["opacities"], cols[v],
                                  sc.viewmats, sc.Ks, sc.width, sc.height, sh_degree=DEGREE[v], packed=False,
                                  absgrad=True)
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()

    times = _alternated(step, a.iters, a.warmup)

    d = sc  # projection stages alone, on the same gradient records
    with torch.no_grad():
        radii = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols[VARIANTS[0]].detach(), d.viewmats,
                                      d.Ks, sc.width, sc.height, 3)["radii"]
        v_splats = torch.randn(C, N, stages.SPLAT_FLOATS, device="cuda", generator=g) * (radii > 0)[..., None]
        pairs = int((radii > 0).sum())

        def stage(v):
            c = cols[v].detach()
            p = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, c, d.viewmats, d.Ks, sc.width, sc.height,
                                      DEGREE[v])
            stages.projection_bwd(d.means, d.quats, d.scales, c, d.viewmats, d.Ks, sc.width, sc.height, DEGREE[v], 0.3,
                                  p["radii"], p["colors"], v_splats, want_absgrad=True)

        stage_times = _alternated(stage, a.iters, a.warmup)

    res = dict(gpu_info(), scene="metric", n_gaussians=N, width=sc.width, height=sc.height, views_per_call=C,
               visible_pairs=pairs, iters=a.iters,
               fwd_bwd_ms_median={v: statistics.median(times[v]) for v in VARIANTS},
               fwd_bwd_ms_min={v: min(times[v]) for v in VARIANTS},
               projection_stages_ms_median={v: statistics.median(stage_times[v]) for v in VARIANTS})
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_sh_degree4.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
