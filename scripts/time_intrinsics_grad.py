"""What asking for camera gradients costs: forward + backward of one rasterization() call on the benchmark's metric
scene (1 M Gaussians, 1920 x 1080, 4 views per call, SH degree 3, the bench functional sum(colors * Wc) + sum(alphas *
Wa)) with no camera gradient, with ``viewmats.requires_grad``, with ``Ks.requires_grad`` and with both, alternated in one
run (the order rotates every iteration) and timed with CUDA events.

``python scripts/time_intrinsics_grad.py [--iters 30] [--warmup 5] [--views 4] [--out DIR]``

Prints the GPU name and power limit next to the medians, and the largest relative difference between the parameter
gradients of the plain and the Ks + viewmats variants on the timed inputs."""
import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from easy_gaussian_splatting_b200 import rasterization  # noqa: E402
from easy_gaussian_splatting_b200.synthetic import loss_weights, make_config_scene  # noqa: E402

PARAMS = ("means", "quats", "scales", "opacities", "colors")


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--views", type=int, default=4)
    ap.add_argument("--out", default=None, help="directory for a JSON copy of the result")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script times the GPU")
    sc = make_config_scene("metric", n_views=a.views).to("cuda")
    C = sc.viewmats.shape[0]
    Wc, Wa = (w.cuda() for w in loss_weights(sc.seed, C, sc.height, sc.width))
    params = {k: getattr(sc, k).clone().requires_grad_(True) for k in PARAMS}
    bg = sc.background[None].expand(C, 3).contiguous()

    variants = {"plain": (False, False), "viewmats_grad": (True, False), "Ks_grad": (False, True),
                "viewmats_and_Ks_grad": (True, True)}

    def step(name):
        vg, kg = variants[name]
        for p in params.values():
            p.grad = None
        vm = sc.viewmats.clone().requires_grad_(vg)
        Ks = sc.Ks.clone().requires_grad_(kg)
        rc, ra, _ = rasterization(params["means"], params["quats"], params["scales"], params["opacities"],
                                  params["colors"], vm, Ks, sc.width, sc.height, sh_degree=3, packed=False,
                                  backgrounds=bg, absgrad=True)
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()
        return vm, Ks

    names = list(variants)
    for _ in range(a.warmup):
        for name in names:
            step(name)
    times = {name: [] for name in names}
    for i in range(a.iters):
        for name in names[i % len(names):] + names[:i % len(names)]:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            step(name)
            t1.record()
            t1.synchronize()
            times[name].append(t0.elapsed_time(t1))
    step("plain")
    g_plain = {k: p.grad.clone() for k, p in params.items()}
    vm, Ks = step("viewmats_and_Ks_grad")
    # the projection backward's parameter gradients do not depend on the camera gradients (bit for bit,
    # tests/test_gpu_intrinsics_grad.py); two separate calls differ by the order of the blend backward's atomic adds
    diff = max(((g_plain[k] - params[k].grad).double().norm() / g_plain[k].double().norm().clamp_min(1e-30)).item()
               for k in PARAMS)
    med = {name: statistics.median(t) for name, t in times.items()}
    res = dict(gpu_info(), scene="metric", n_gaussians=int(sc.means.shape[0]), width=sc.width, height=sc.height,
               views_per_call=C, iters=a.iters, fwd_bwd_ms_median=med,
               fwd_bwd_ms_min={name: min(t) for name, t in times.items()},
               added_ms_median={name: med[name] - med["plain"] for name in names[1:]},
               param_grads_max_rel_diff=diff, v_viewmats_finite=bool(torch.isfinite(vm.grad).all()),
               v_Ks_finite=bool(torch.isfinite(Ks.grad).all()))
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_intrinsics_grad.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
