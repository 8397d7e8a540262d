"""Time and judge adaptive sampling of a view sweep (b2pt_render_views_adaptive) on cuda:0.
  overhead  tau = 0 (every pixel gets every round, so the same paths) against b2pt_render_views_checkpoints(rounds)
            with sums of squares (which also copies K images and K moment slices to pageable host memory) and against
            b2pt_render_views(rounds[-1]) (one image): wall time of one call (host clock around calls that end in a
            stream synchronise), alternating the three, and paths/s.  Workloads: the reference's 225-view
            hemisphere at 128^2 and one 1024^2 view, depth 50, rounds 2, 4, ..., 64.  Cornell box.
  quality   rel-MSE against a 4096-spp target (as DESIGN.md 8e measures it, depth 5) of 8 tilted views at 128^2 for
            adaptive renders at several tau (rounds 4, 8, ..., 256) and for uniform renders of the same total paths,
            with the mean samples per pixel.
The GPU name and power limit are read in the same run.  One JSON line per workload goes to stdout (and
OUT/time_adaptive.jsonl with --out).

  python scripts/time_adaptive.py [--out DIR] [--reps 3] [--skip-overhead] [--skip-quality]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import raytracingtherestofyourlife_b200 as B  # noqa: E402
from time_direct_views import gpu_info, hemisphere, row  # noqa: E402


def params(tau, eps=0.01, radius=1):
    prm = B.AdaptiveParams()
    prm.threshold, prm.epsilon, prm.radius = tau, eps, radius
    return prm


def overhead(ctx, name, views, w, reps):
    rounds = (2, 4, 8, 16, 32, 64)
    depth = 50
    calls = {
        "checkpoints": lambda: ctx.render_views_checkpoints(views, w, w, rounds, depth, 0, moments=True),
        "adaptive_tau0": lambda: ctx.render_views_adaptive(views, w, w, rounds, depth, params(0.0)),
        "uniform": lambda: ctx.render_views(views, w, w, rounds[-1], depth),
    }
    for f in calls.values():  # warm-up: modules, buffers, tail decisions
        f()
    times = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    paths = len(views) * w * w * rounds[-1]
    res = dict(workload=name, rounds=rounds, depth=depth, paths=paths)
    for k, ts in times.items():
        med = statistics.median(ts)
        res[k] = dict(ms_median=round(med, 2), ms_range=[round(min(ts), 2), round(max(ts), 2)],
                      gpaths_per_s=round(paths / med / 1e6, 3))
    return res


def quality(ctx):
    c = 278 / 555.0
    tilted = []
    for v in range(8):
        ang = 0.35 * (v - 3.5) / 8
        tilted.append(row([c + 1.95 * np.sin(ang), c + 0.1 * (v % 3), c - 1.95 * np.cos(ang)]))
    views = np.stack(tilted)
    w = 128
    depth = 5
    rounds = (4, 8, 16, 32, 64, 128, 256)
    target = np.nan_to_num(ctx.render_views(views, w, w, 4096, depth)[..., :3].astype(np.float64) / 4096)

    def rel(x):
        return round(float(((x - target) ** 2 / (target ** 2 + 1e-2)).mean()), 6)
    rows = []
    for tau in (0.01, 0.02, 0.03, 0.05, 0.1):
        for eps, radius in ((0.01, 1), (0.01, 0), (0.1, 1)):
            img, _, counts, active = ctx.render_views_adaptive(views, w, w, rounds, depth, params(tau, eps, radius))
            mean_spp = float(counts.mean())
            adaptive = rel(np.nan_to_num(img[..., :3].astype(np.float64)) / counts[..., None])
            spp = max(1, int(round(mean_spp)))
            uniform = rel(np.nan_to_num(ctx.render_views(views, w, w, spp, depth)[..., :3].astype(np.float64)) / spp)
            rows.append(dict(tau=tau, eps=eps, radius=radius, mean_spp=round(mean_spp, 2), active=active.tolist(),
                             relmse_adaptive=adaptive, uniform_spp=spp, relmse_uniform=uniform))
    return dict(workload="quality_8x128", rounds=rounds, depth=depth, rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-overhead", action="store_true")
    ap.add_argument("--skip-quality", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    info = gpu_info()
    lines = []
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        if not a.skip_overhead:
            lines.append(overhead(ctx, "hemisphere_225x128", np.stack(hemisphere(15, 15)), 128, a.reps))
            lines.append(overhead(ctx, "single_1024", hemisphere(15, 15)[0][None], 1024, a.reps))
        if not a.skip_quality:
            lines.append(quality(ctx))
    for line in lines:
        line.update(info)
        print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_adaptive.jsonl"), "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
