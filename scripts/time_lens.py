"""Cost of the thin lens (b2pt_set_lens) on cuda:0, Cornell box, depth 50, pinhole against aperture 0.05 (focus at each
camera's look-at point):
  whole call   host clock around calls that end in a stream synchronise, median of --reps alternating calls, of
                 render     one 1024^2 view at 1024 spp (b2pt_render + read_color)
                 sweep      the reference's 225-view 128^2 hemisphere at 64 spp (b2pt_render_views)
  primary      in a separate torch.profiler pass over one call of each: the GPU time of the primary-ray trace launches
               (k_trace<true, ...> for the pinhole, k_trace_lens for the lens) and of every kernel together.
The lens traces primary rays without the Cornell per-tile candidate masks, which assume one ray origin per view, so the
primary launch is where the cost shows.  The GPU name and power limit are read in the same run.  One JSON line per
workload goes to stdout (and OUT/time_lens.jsonl with --out).

  python scripts/time_lens.py [--out DIR] [--reps 5] [--skip-profile]
"""
import argparse
import json
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import raytracingtherestofyourlife_b200 as B  # noqa: E402
from time_direct_views import gpu_info, hemisphere  # noqa: E402

DEPTH = 50
APERTURE = 0.05


def workloads(ctx):
    views = hemisphere(15, 15)

    def render():
        ctx.set_camera(B.Camera(1024, 1024))
        ctx.render(1024, DEPTH)
        return ctx.read_color()
    return {"render_1024sq_1024spp": render,
            "sweep_225x128sq_64spp": lambda: ctx.render_views(views, 128, 128, 64, DEPTH)}


def timed(ctx, name, f, reps):
    lenses = {"pinhole": 0.0, "lens": APERTURE}
    for a in lenses.values():  # warm-up: modules, buffers, tail decisions
        ctx.set_lens(a, 0)
        f()
    times = {k: [] for k in lenses}
    for _ in range(reps):
        for k, a in lenses.items():
            ctx.set_lens(a, 0)
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    res = dict(workload=name, depth=DEPTH, aperture=APERTURE, reps=reps)
    for k, ts in times.items():
        res[k] = dict(ms_median=round(statistics.median(ts), 2), ms_range=[round(min(ts), 2), round(max(ts), 2)])
    res["lens_over_pinhole"] = round(res["lens"]["ms_median"] / res["pinhole"]["ms_median"], 4)
    return res


def profile(ctx, name, f, out):
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    res = dict(workload=name + "_profile", aperture=APERTURE)
    for k, a in (("pinhole", 0.0), ("lens", APERTURE)):
        ctx.set_lens(a, 0)
        f()
        with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        if out:
            prof.export_chrome_trace(os.path.join(out, "lens_%s_%s.json" % (name, k)))
        primary = total = 0.0
        for ev in prof.key_averages():
            dev = getattr(ev, "device_time_total", None)
            if dev is None:
                dev = getattr(ev, "cuda_time_total", 0)
            if not dev or "b2pt::" not in ev.key:
                continue
            total += dev / 1e3
            if "k_trace_lens" in ev.key or "k_trace<true" in ev.key:
                primary += dev / 1e3
        res[k] = dict(primary_trace_ms=round(primary, 3), kernels_ms=round(total, 3))
    res["primary_lens_over_pinhole"] = round(res["lens"]["primary_trace_ms"] / res["pinhole"]["primary_trace_ms"], 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-profile", action="store_true")
    a = ap.parse_args()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    rows = []
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        ctx.build_bvh()
        fs = workloads(ctx)
        for name, f in fs.items():
            rows.append(dict(timed(ctx, name, f, a.reps), **info))
            print(json.dumps(rows[-1]), flush=True)
        if not a.skip_profile:
            for name, f in fs.items():
                rows.append(dict(profile(ctx, name, f, a.out), **info))
                print(json.dumps(rows[-1]), flush=True)
    if a.out:
        with open(os.path.join(a.out, "time_lens.jsonl"), "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
