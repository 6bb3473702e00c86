"""Times one refine iteration's four render_point calls (800^2, 400^2, 200^2 with 19 channels and the 800^2 3-channel coverage
mask; K = 8, NDC radius 2 px at 800^2, fov 20) forward and backward on a seeded ~1.3 M point cloud, the size load_views produces.
CUDA events, median over the timed iterations after warm-up; per-kernel times from a separate torch.profiler run.  Beside it the
oracle's torch splat formulation (oracle/points_ref.py: footprint splat + sort + composite, autograd backward) on the same GPU and
inputs: the "what you write without pytorch3d" baseline (pytorch3d itself is not available to time).  It imports the oracle, so it
lives under tests/.  MEASUREMENT TOOL, not product.
    python tests/measure_point_render.py --out profiles/r3_point_render.json        (GPU box)"""
import argparse
import importlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import points_ref as opr      # noqa: E402
import points_cases as pc                 # noqa: E402

SIZES = (800, 400, 200)


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q


def med_ms(fn, n, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--oracle-iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    ru = importlib.import_module("make-it-3d_b200.nerf.refine_utils")
    xyz, feats = pc.refine_cloud()
    xyz, feats = torch.from_numpy(xyz).cuda(), torch.from_numpy(feats).cuda().requires_grad_()
    ones = torch.ones(len(xyz), 3, device="cuda")
    w2c = torch.from_numpy(pc.look_at_world2cam()).cuda()
    Ks = {S: torch.from_numpy(pc.intrinsics(S)).cuda() for S in SIZES}
    r, ppp = pc.REFINE_RADIUS, 8
    g_outs = {S: torch.randn(1, 19, S, S, device="cuda") for S in SIZES}

    def fwd():
        outs = [ru.render_point(xyz, feats, S, S, Ks[S], w2c, (S, S), r, ppp) for S in SIZES]
        outs.append(ru.render_point(xyz, ones, 800, 800, Ks[800], w2c, (800, 800), r, ppp))
        return outs

    def step():
        outs = fwd()
        torch.autograd.backward(outs[:3], [g_outs[S] for S in SIZES])
        feats.grad = None

    with torch.no_grad():
        t_fwd = med_ms(fwd, args.iters, args.warmup)
    t_step = med_ms(step, args.iters, args.warmup)
    with torch.no_grad():
        covered = {S: float((ru.point_render(opr.project(xyz, S, S, Ks[S], w2c), ones, S, r, ppp)[1][..., 0] >= 0).float().mean())
                   for S in SIZES}

    # per-kernel device time, separate run
    from torch.profiler import ProfilerActivity, profile
    n_prof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            step()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        m = re.search(r"k_pr_\w+(<\d+>)?", ev.key)
        if t and m:
            name = m.group(0)
            k = kern.setdefault(name, {"us_per_iter": 0.0, "launches_per_iter": 0})
            k["us_per_iter"] += t / n_prof
            k["launches_per_iter"] += ev.count // n_prof

    # oracle torch splat formulation, same inputs
    f_or = feats.detach().clone().requires_grad_()

    def oracle_step():
        outs = []
        for S in SIZES:
            pts = opr.project(xyz, S, S, Ks[S], w2c)
            i, d = opr.raster_splat(pts, S, ppp, r)
            outs.append(opr.composite(i, d, f_or, r))
        pts = opr.project(xyz, 800, 800, Ks[800], w2c)
        i, d = opr.raster_splat(pts, 800, ppp, r)
        opr.composite(i, d, ones, r)
        torch.autograd.backward(outs, [g_outs[S] for S in SIZES])
        f_or.grad = None

    t_oracle = med_ms(oracle_step, args.oracle_iters, 1)
    res = {
        "what": "one refine iteration's render_point calls: 800^2, 400^2, 200^2 x 19 channels + 800^2 x 3 mask; K=8, radius 2 px at "
                "800^2; forward and backward of the three 19-channel renders",
        "device": card(),
        "points": int(len(xyz)),
        "covered_pixel_fraction": covered,
        "forward_4_calls_ms": {"median": t_fwd[0], "min": t_fwd[1], "max": t_fwd[2]},
        "forward_plus_backward_ms": {"median": t_step[0], "min": t_step[1], "max": t_step[2]},
        "iters": args.iters, "warmup": args.warmup,
        "kernels_from_profiler": kern,
        "oracle_torch_splat_forward_plus_backward_ms": {"median": t_oracle[0], "min": t_oracle[1], "max": t_oracle[2],
                                                        "iters": args.oracle_iters,
                                                        "note": "baseline: the oracle's torch formulation, not pytorch3d"},
        "working_set_note": "points + features ~ 114 MB, about the size of L2 (126 MB): repeated iterations read partly from L2",
    }
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
