"""What asking for viewmat gradients costs: forward + backward of one rasterization() call on the benchmark's metric
scene (1 M Gaussians, 1920 x 1080, 4 views per call, SH degree 3, the bench functional sum(colors * Wc) + sum(alphas *
Wa)), with and without ``viewmats.requires_grad``, alternated in one run and timed with CUDA events.

``python scripts/time_viewmat_grad.py [--iters 30] [--warmup 5] [--views 4] [--out DIR]``

Prints the GPU name and power limit next to the times, and the largest relative difference between the parameter
gradients of the two variants on the timed inputs."""
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

    def step(vg):
        for p in params.values():
            p.grad = None
        vm = sc.viewmats.clone().requires_grad_(vg)
        rc, ra, _ = rasterization(params["means"], params["quats"], params["scales"], params["opacities"],
                                  params["colors"], vm, sc.Ks, sc.width, sc.height, sh_degree=3, packed=False,
                                  backgrounds=bg, absgrad=True)
        ((rc * Wc).sum() + (ra * Wa).sum()).backward()
        return vm

    for _ in range(a.warmup):
        step(False)
        step(True)
    times = {False: [], True: []}
    for i in range(a.iters):
        for vg in ((False, True) if i % 2 == 0 else (True, False)):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            step(vg)
            t1.record()
            t1.synchronize()
            times[vg].append(t0.elapsed_time(t1))
    step(False)
    g_plain = {k: p.grad.clone() for k, p in params.items()}
    vm = step(True)
    # the projection backward's parameter gradients do not depend on the flag (bit for bit, tests/test_gpu_viewmat_grad.py);
    # two separate calls differ by the order of the blend backward's atomic adds, so this reports the relative difference
    diff = max(((g_plain[k] - params[k].grad).double().norm() / g_plain[k].double().norm().clamp_min(1e-30)).item()
               for k in PARAMS)
    res = dict(gpu_info(), scene="metric", n_gaussians=int(sc.means.shape[0]), width=sc.width, height=sc.height,
               views_per_call=C, iters=a.iters,
               fwd_bwd_ms_median={"plain": statistics.median(times[False]), "viewmats_grad": statistics.median(times[True])},
               fwd_bwd_ms_min={"plain": min(times[False]), "viewmats_grad": min(times[True])},
               param_grads_max_rel_diff=diff, v_viewmats_finite=bool(torch.isfinite(vm.grad).all()))
    res["added_ms_median"] = res["fwd_bwd_ms_median"]["viewmats_grad"] - res["fwd_bwd_ms_median"]["plain"]
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "time_viewmat_grad.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
