"""Time and judge an adaptive sweep denoised on the device (b2pt_render_views_adaptive_denoised) on cuda:0.
  cost      default adaptive and filter parameters, rounds 2, 4, ..., 64, depth 50; wall time of one call (host clock
            around calls that end in a stream synchronise), median of --reps alternating calls, of
              adaptive_denoised  the new call (image, counts and denoised image to the host)
              adaptive           b2pt_render_views_adaptive alone (image, sums of squares, counts)
              uniform_pipeline   what the driver's -denoise runs at rounds[-1]: render_views_checkpoints with sums of
                                 squares, render_views_features, denoise_views (inputs through pageable host memory)
            Workloads: the reference's 225-view hemisphere at 128^2 and one 1024^2 view.  Cornell box.  A separate
            torch.profiler pass over one adaptive_denoised call splits its GPU time into kernels (by name) and copies.
  quality   rel-MSE against a 4096-spp target (depth 5) of 8 tilted views at 128^2, rounds 4, 8, ..., 256: adaptive
            plus the filter against a uniform render of the adaptive mean spp plus the filter, for tau 0.02 and 0.1
            (epsilon 0.01, radius 1), also over the pixels whose first round had exactly zero variance (V0 = 0).
The GPU name and power limit are read in the same run.  One JSON line per workload goes to stdout (and
OUT/time_adaptive_denoise.jsonl with --out).

  python scripts/time_adaptive_denoise.py [--out DIR] [--reps 5] [--skip-cost] [--skip-profile] [--skip-quality]
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
from time_adaptive import params  # noqa: E402
from time_direct_views import gpu_info, hemisphere, row  # noqa: E402

ROUNDS = (2, 4, 8, 16, 32, 64)
DEPTH = 50


def calls(ctx, views, w):
    c = ROUNDS[-1]

    def uniform_pipeline():
        color, m2 = ctx.render_views_checkpoints(views, w, w, (c,), DEPTH, 0, moments=True)
        alb, nd = ctx.render_views_features(views, w, w, (c,))
        return ctx.denoise_views(color, m2, alb, nd, w, w, (c,))
    return {
        "adaptive_denoised": lambda: ctx.render_views_adaptive_denoised(views, w, w, ROUNDS, DEPTH),
        "adaptive": lambda: ctx.render_views_adaptive(views, w, w, ROUNDS, DEPTH),
        "uniform_pipeline": uniform_pipeline,
    }


def cost(ctx, name, views, w, reps):
    fs = calls(ctx, views, w)
    for f in fs.values():  # warm-up: modules, buffers, tail decisions
        f()
    times = {k: [] for k in fs}
    for _ in range(reps):
        for k, f in fs.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    _, counts, _ = fs["adaptive_denoised"]()
    res = dict(workload=name, rounds=ROUNDS, depth=DEPTH, views=len(views), size=w, reps=reps,
               mean_spp=round(float(counts.mean()), 3))
    for k, ts in times.items():
        res[k] = dict(ms_median=round(statistics.median(ts), 2), ms_range=[round(min(ts), 2), round(max(ts), 2)])
    return res


def profile(ctx, name, views, w, out):
    """GPU time of one adaptive_denoised call by kernel name and copy kind (torch.profiler, as time_denoise.py)."""
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    f = calls(ctx, views, w)["adaptive_denoised"]
    f()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    if out:
        prof.export_chrome_trace(os.path.join(out, "adaptive_denoise_%s.json" % name))
    groups = {}
    for ev in prof.key_averages():
        dev = getattr(ev, "device_time_total", None)
        if dev is None:
            dev = getattr(ev, "cuda_time_total", 0)
        if not dev or not ("b2pt::" in ev.key or "Memcpy" in ev.key or "Memset" in ev.key or "cub" in ev.key):
            continue
        key = ev.key
        for stem in ("k_view_features_counts", "k_denoise_prep_counts", "k_atrous", "k_pnm16", "k_trace", "k_shade",
                     "k_tail_loop", "k_accumulate", "k_adaptive", "k_list_pad", "k_primary", "k_bvh_hits"):
            if stem in key:
                key = stem
                break
        groups[key] = groups.get(key, 0.0) + dev / 1e3
    top = sorted(groups.items(), key=lambda kv: -kv[1])
    copies = sum(v for k, v in groups.items() if "Memcpy" in k)
    denoise = sum(groups.get(k, 0.0) for k in ("k_view_features_counts", "k_denoise_prep_counts", "k_atrous",
                                               "k_pnm16"))
    return dict(workload=name + "_profile", gpu_ms_listed=round(sum(groups.values()), 3), copies_ms=round(copies, 3),
                denoise_kernels_ms=round(denoise, 3), by_name={k[:80]: round(v, 3) for k, v in top[:24]})


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

    def rel(x, mask=None):
        e = (np.asarray(x, np.float64) - target) ** 2 / (target ** 2 + 1e-2)
        return round(float((e if mask is None else e[mask]).mean()), 6)
    rows = []
    for tau in (0.02, 0.1):
        img, counts, den = ctx.render_views_adaptive_denoised(views, w, w, rounds, depth, params(tau, 0.01, 1))
        p0 = B.DenoiseParams.defaults()
        p0.levels = 0
        v0 = ctx.render_views_adaptive_denoised(views, w, w, rounds, depth, params(tau, 0.01, 1), p0)[2][..., 3]
        flat = (v0 == 0) & (counts == rounds[0])  # first round had exactly zero variance
        mean_spp = float(counts.mean())
        spp = max(2, int(round(mean_spp)))
        color, m2 = ctx.render_views_checkpoints(views, w, w, (spp,), depth, 0, moments=True)
        alb, nd = ctx.render_views_features(views, w, w, (spp,))
        uden = ctx.denoise_views(color, m2, alb, nd, w, w, (spp,))[0]
        noisy_a = np.nan_to_num(img[..., :3].astype(np.float64)) / counts[..., None]
        noisy_u = np.nan_to_num(color[0, ..., :3].astype(np.float64)) / spp
        rows.append(dict(tau=tau, eps=0.01, radius=1, mean_spp=round(mean_spp, 2), uniform_spp=spp,
                         relmse_adaptive=rel(noisy_a), relmse_adaptive_denoised=rel(den[..., :3]),
                         relmse_uniform=rel(noisy_u), relmse_uniform_denoised=rel(uden[..., :3]),
                         zero_var_fraction=round(float(flat.mean()), 4),
                         zero_var_relmse_adaptive_denoised=rel(den[..., :3], flat) if flat.any() else None,
                         zero_var_relmse_uniform_denoised=rel(uden[..., :3], flat) if flat.any() else None,
                         zero_var_relmse_adaptive=rel(noisy_a, flat) if flat.any() else None))
    return dict(workload="quality_8x128", rounds=rounds, depth=depth, target_spp=4096, rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-cost", action="store_true")
    ap.add_argument("--skip-profile", action="store_true")
    ap.add_argument("--skip-quality", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    lines = []
    workloads = [("hemisphere_225x128", np.stack(hemisphere(15, 15)), 128),
                 ("single_1024", hemisphere(15, 15)[0][None], 1024)]
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        if not a.skip_cost:
            for name, views, w in workloads:
                lines.append(cost(ctx, name, views, w, a.reps))
                print(json.dumps(lines[-1]), flush=True)
        if not a.skip_profile:
            for name, views, w in workloads:
                lines.append(profile(ctx, name, views, w, a.out))
                print(json.dumps(lines[-1]), flush=True)
        if not a.skip_quality:
            lines.append(quality(ctx))
            print(json.dumps(lines[-1]), flush=True)
    for line in lines:
        line.update(info)
    print(json.dumps(info), flush=True)
    if a.out:
        with open(os.path.join(a.out, "time_adaptive_denoise.jsonl"), "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
