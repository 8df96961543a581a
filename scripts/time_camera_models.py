"""What the camera models cost: forward and backward of one rasterization_camera_model() call on the benchmark's metric
scene (1 M Gaussians, 1920 x 1080, 4 views per call, SH degree 3, a random linear functional of the images and the
alphas; with --camera-grads viewmats and Ks get gradients too) for camera_model "pinhole", "ortho" and "fisheye",
alternated in one run and timed with CUDA events (forward: the call; backward: .backward()).  The fisheye camera gets
the pinhole's field of view across the width (fx = (W / 2) / atan((W / 2) / fx_pinhole), about 1834 for the metric scene's +-30 degrees), the
orthographic one fx = fx_pinhole / (median depth of camera 0), so that all three see about the same Gaussians.  Prints
the visible (camera, Gaussian) pairs and intersections of each model, and the GPU name and power limit.

``python scripts/time_camera_models.py [--iters 20] [--warmup 3] [--views 4] [--camera-grads] [--out DIR]``"""
import argparse
import json
import math
import os
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from easy_gaussian_splatting_b200 import rasterization_camera_model  # noqa: E402
from easy_gaussian_splatting_b200.synthetic import make_config_scene  # noqa: E402
from scripts.time_viewmat_grad import gpu_info  # noqa: E402

GEOM = ("means", "quats", "scales", "opacities")
MODELS = ("pinhole", "ortho", "fisheye")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--views", type=int, default=4)
    ap.add_argument("--camera-grads", action="store_true", help="viewmats and Ks require grad")
    ap.add_argument("--out", default=None, help="directory for a JSON copy of the result")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script times the GPU")
    sc = make_config_scene("metric", n_views=a.views).to("cuda")
    C, N = sc.viewmats.shape[0], sc.means.shape[0]
    fx = sc.Ks[0, 0, 0].item()
    z = (sc.means @ sc.viewmats[0, :3, :3].T + sc.viewmats[0, :3, 3])[:, 2]
    Ks = {"pinhole": sc.Ks, "ortho": sc.Ks.clone(), "fisheye": sc.Ks.clone()}
    Ks["ortho"][:, 0, 0] *= 1.0 / z[z > 0].median().item()
    Ks["ortho"][:, 1, 1] *= 1.0 / z[z > 0].median().item()
    f_fish = (0.5 * sc.width) / math.atan((0.5 * sc.width) / fx)
    Ks["fisheye"][:, 0, 0] *= f_fish / fx
    Ks["fisheye"][:, 1, 1] *= f_fish / fx
    viewmats = sc.viewmats.clone().requires_grad_(a.camera_grads)
    Ks = {m: K.clone().requires_grad_(a.camera_grads) for m, K in Ks.items()}
    g = torch.Generator(device="cuda").manual_seed(0)
    params = {k: getattr(sc, k).clone().requires_grad_(True) for k in (*GEOM, "colors")}
    Wc = torch.rand(C, sc.height, sc.width, 3, device="cuda", generator=g)
    Wa = torch.rand(C, sc.height, sc.width, 1, device="cuda", generator=g)
    counts = {}

    def step(m, count=False):
        for p in (*params.values(), viewmats, Ks[m]):
            p.grad = None
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        rc, ra, meta = rasterization_camera_model(*[params[k] for k in (*GEOM, "colors")], viewmats, Ks[m], sc.width,
                                                  sc.height, sh_degree=3, packed=False, absgrad=True, camera_model=m)
        e[1].record()
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()
        e[2].record()
        e[2].synchronize()
        if count:
            counts[m] = dict(n_visible=int((meta["radii"] > 0).sum()), n_isects=int(meta["flatten_ids"].numel()))
        return e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])

    for _ in range(a.warmup):
        for m in MODELS:
            step(m, count=True)
    fwd, bwd = {m: [] for m in MODELS}, {m: [] for m in MODELS}
    for i in range(a.iters):
        for m in (MODELS if i % 2 == 0 else MODELS[::-1]):
            f, b = step(m)
            fwd[m].append(f)
            bwd[m].append(b)
    res = dict(gpu_info(), scene="metric", n_gaussians=N, width=sc.width, height=sc.height, views_per_call=C,
               iters=a.iters, camera_grads=a.camera_grads, library=os.environ.get("EGS_RASTER_LIB", "in-tree"),
               fx={m: Ks[m][0, 0, 0].item() for m in MODELS}, counts=counts,
               fwd_ms_median={m: statistics.median(fwd[m]) for m in MODELS},
               bwd_ms_median={m: statistics.median(bwd[m]) for m in MODELS},
               fwd_ms_min={m: min(fwd[m]) for m in MODELS}, bwd_ms_min={m: min(bwd[m]) for m in MODELS})
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        name = "time_camera_models" + ("_camera_grads" if a.camera_grads else "") + ".json"
        Path(a.out, name).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
