"""What per-camera SH coefficients cost: forward + backward of one rasterization() call on the benchmark's metric scene
(1 M Gaussians, 1920 x 1080, 4 views per call, SH degree 3, the functional sum(colors * Wc) + sum(alphas * Wa)) with
shared coefficients [N,16,3] against per-camera coefficients [4,N,16,3], alternated in one run and timed with CUDA
events.  Also times the projection forward + backward stages alone on the same records.

Per camera, the coefficient reads of visible pairs and the gradient writes grow from N * 192 B to C * N * 192 B.

``python scripts/time_per_camera_sh.py [--iters 20] [--warmup 3] [--views 4] [--out DIR]``

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
VARIANTS = ("shared [N,16,3]", "per-camera [C,N,16,3]")


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
    shared = sc.colors.clone().requires_grad_(True)
    percam = (sc.colors[None] + 0.05 * torch.randn(C, *sc.colors.shape, device="cuda", generator=g)).requires_grad_(True)
    cols = dict(zip(VARIANTS, (shared, percam)))
    Wc = torch.rand(C, sc.height, sc.width, 3, device="cuda", generator=g)
    Wa = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)

    def step(v):
        for p in list(params.values()) + [cols[v]]:
            p.grad = None
        rc, ra, _ = rasterization(params["means"], params["quats"], params["scales"], params["opacities"], cols[v],
                                  sc.viewmats, sc.Ks, sc.width, sc.height, sh_degree=3, packed=False, absgrad=True)
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()

    for _ in range(a.warmup):
        for v in VARIANTS:
            step(v)
    times = {v: [] for v in VARIANTS}
    for i in range(a.iters):
        for v in (VARIANTS if i % 2 == 0 else VARIANTS[::-1]):
            times[v].append(_timed(lambda: step(v)))

    # projection stages alone, on the same gradient records
    d = sc
    with torch.no_grad():
        proj = {v: stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols[v].detach(), d.viewmats, d.Ks,
                                         sc.width, sc.height, 3) for v in VARIANTS}
        v_splats = torch.randn(C, N, stages.SPLAT_FLOATS, device="cuda", generator=g) * (proj[VARIANTS[0]]["radii"] > 0)[..., None]
        pairs = int((proj[VARIANTS[0]]["radii"] > 0).sum())

        def stage(v):
            p = stages.projection_fwd(d.means, d.quats, d.scales, d.opacities, cols[v].detach(), d.viewmats, d.Ks, sc.width,
                                      sc.height, 3)
            stages.projection_bwd(d.means, d.quats, d.scales, cols[v].detach(), d.viewmats, d.Ks, sc.width, sc.height, 3,
                                  0.3, p["radii"], p["colors"], v_splats, want_absgrad=True)

        for _ in range(a.warmup):
            for v in VARIANTS:
                stage(v)
        stage_times = {v: [] for v in VARIANTS}
        for i in range(a.iters):
            for v in (VARIANTS if i % 2 == 0 else VARIANTS[::-1]):
                stage_times[v].append(_timed(lambda: stage(v)))

    res = dict(gpu_info(), scene="metric", n_gaussians=N, width=sc.width, height=sc.height, views_per_call=C,
               visible_pairs=pairs, iters=a.iters,
               fwd_bwd_ms_median={v: statistics.median(times[v]) for v in VARIANTS},
               fwd_bwd_ms_min={v: min(times[v]) for v in VARIANTS},
               projection_stages_ms_median={v: statistics.median(stage_times[v]) for v in VARIANTS})
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_per_camera_sh.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
