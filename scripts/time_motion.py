"""Cost of the motion vectors (b2pt_render_views_motion) against the features (b2pt_render_views_features) on cuda:0,
Cornell box, the reference's 225-view 128^2 hemisphere with checkpoints 1, 2, 4, ..., 64; each view compared with the
one before it in sweep order (the first with itself):
  whole call   host clock around calls that end in a stream synchronise, median of --reps alternating calls;
  kernels      in a separate torch.profiler pass over one call of each: the GPU time of k_view_motion and of
               k_view_features, and of every kernel of the call together.
Motion traces a primary ray and, for every hit seen on the previous camera's canvas, a visibility ray; the features
trace the primary ray only.  The GPU name and power limit are read in the same run.  One JSON line per measurement goes
to stdout (and OUT/time_motion.jsonl with --out).

  python scripts/time_motion.py [--out DIR] [--reps 7] [--skip-profile]
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
from time_direct_views import gpu_info, hemisphere  # noqa: E402

W = H = 128
CKPTS = (1, 2, 4, 8, 16, 32, 64)


def calls(ctx):
    views = hemisphere(15, 15)
    prev = np.concatenate([views[:1], views[:-1]])
    return {"motion": lambda: ctx.render_views_motion(views, prev, W, H, CKPTS),
            "features": lambda: ctx.render_views_features(views, W, H, CKPTS)}


def timed(fs, reps):
    for f in fs.values():  # warm-up: modules, trace structures, staging buffers
        f()
    times = {k: [] for k in fs}
    for _ in range(reps):
        for k, f in fs.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    res = dict(workload="hemisphere_225x128sq_ckpt1-64", reps=reps)
    for k, ts in times.items():
        res[k] = dict(ms_median=round(statistics.median(ts), 2), ms_range=[round(min(ts), 2), round(max(ts), 2)])
    res["motion_over_features"] = round(res["motion"]["ms_median"] / res["features"]["ms_median"], 4)
    return res


def profile(fs, out):
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    res = dict(workload="hemisphere_225x128sq_ckpt1-64_profile")
    for k, f in fs.items():
        f()
        with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        if out:
            prof.export_chrome_trace(os.path.join(out, "motion_%s.json" % k))
        kernel = total = 0.0
        for ev in prof.key_averages():
            dev = getattr(ev, "device_time_total", None)
            if dev is None:
                dev = getattr(ev, "cuda_time_total", 0)
            if not dev:
                continue
            total += dev / 1e3
            if ("k_view_motion" if k == "motion" else "k_view_features") in ev.key:
                kernel += dev / 1e3
        res[k] = dict(kernel_ms=round(kernel, 3), gpu_ms=round(total, 3))
    res["kernel_motion_over_features"] = round(res["motion"]["kernel_ms"] / res["features"]["kernel_ms"], 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--skip-profile", action="store_true")
    a = ap.parse_args()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    rows = []
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        ctx.build_bvh()
        fs = calls(ctx)
        rows.append(dict(timed(fs, a.reps), **info))
        print(json.dumps(rows[-1]), flush=True)
        if not a.skip_profile:
            rows.append(dict(profile(fs, a.out), **info))
            print(json.dumps(rows[-1]), flush=True)
        m = fs["motion"]()
        last = m[-1]
        rows.append(dict(workload="hemisphere_motion_stats", valid_share=round(float((last[..., 3] > 0).mean()), 4),
                         visible_over_valid=round(float(last[..., 2].sum() / max(last[..., 3].sum(), 1)), 4)))
        print(json.dumps(rows[-1]), flush=True)
    if a.out:
        with open(os.path.join(a.out, "time_motion.jsonl"), "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
