"""Cost and quality of the temporal accumulation of a sweep (b2pt_denoise_views_temporal) on cuda:0, Cornell box.

Timing, on the reference's 225-view 128^2 hemisphere with checkpoints 1, 2, 4, ..., 256 (K = 9, the workload of
DESIGN.md 8e's table), each view chained to the one before it in sweep order:
  whole call   host clock around calls that end in a stream synchronise, median of --reps alternating calls of
               denoise_views_temporal and denoise_views (same inputs, default parameters);
  kernels      in a separate torch.profiler pass over one call: the GPU time of all k_temporal launches together (one per
               view), of k_denoise_prep, of k_atrous and of the copies.
--sweep: the quality sweep of DESIGN.md 8j instead: one ring of 15 views of the 15 x 15 hemisphere at 128^2, depth 8,
checkpoints (4, 16), against render_views at 4096 spp; rel-MSE of DESIGN.md 8e on the lambertian pixels of views >= 5
for the temporal result at levels 0 and with the default filter, one temporal parameter at a time off its default; the
same under a lens; and the calibration of V_bar (squared error over predicted variance) by motion length.
The GPU name and power limit are read in the same run.  One JSON line per measurement goes to stdout (and
OUT/time_temporal.jsonl with --out).

  python scripts/time_temporal.py [--out DIR] [--reps 7] [--skip-profile] [--sweep]
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
CKPTS = (1, 2, 4, 8, 16, 32, 64, 128, 256)
LUM = np.array([0.2126, 0.7152, 0.0722])


def chain(views):
    return np.concatenate([views[:1], views[:-1]])


def inputs(ctx, views, w, h, ck, depth):
    color, m2 = ctx.render_views_checkpoints(views, w, h, ck, depth, 0, moments=True)
    alb, nd = ctx.render_views_features(views, w, h, ck)
    mot = ctx.render_views_motion(views, chain(views), w, h, ck)
    return dict(color=color, m2=m2, alb=alb, nd=nd, mot=mot, views=views)


def calls(ctx, s):
    return {"temporal": lambda: ctx.denoise_views_temporal(s["color"], s["m2"], s["alb"], s["nd"], s["mot"],
                                                           s["views"], W, H, CKPTS),
            "spatial": lambda: ctx.denoise_views(s["color"], s["m2"], s["alb"], s["nd"], W, H, CKPTS)}


def timed(fs, reps):
    for f in fs.values():  # warm-up: modules and staging buffers
        f()
    times = {k: [] for k in fs}
    for _ in range(reps):
        for k, f in fs.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    res = dict(workload="hemisphere_225x128sq_ckpt1-256", reps=reps)
    for k, ts in times.items():
        res[k] = dict(ms_median=round(statistics.median(ts), 2), ms_range=[round(min(ts), 2), round(max(ts), 2)])
    res["temporal_over_spatial"] = round(res["temporal"]["ms_median"] / res["spatial"]["ms_median"], 4)
    return res


def profile(f, out):
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    f()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    if out:
        prof.export_chrome_trace(os.path.join(out, "temporal.json"))
    res = dict(workload="hemisphere_225x128sq_ckpt1-256_profile", k_temporal_ms=0.0, k_temporal_launches=0,
               k_denoise_prep_ms=0.0, k_atrous_ms=0.0, memcpy_ms=0.0, gpu_ms=0.0)
    for ev in prof.key_averages():
        dev = getattr(ev, "device_time_total", None)
        if dev is None:
            dev = getattr(ev, "cuda_time_total", 0)
        if not dev:
            continue
        ms = dev / 1e3
        res["gpu_ms"] += ms
        for name in ("k_temporal", "k_denoise_prep", "k_atrous"):
            if name in ev.key:
                res[name + "_ms"] += ms
                if name == "k_temporal":
                    res["k_temporal_launches"] += ev.count
        if "memcpy" in ev.key.lower():
            res["memcpy_ms"] += ms
    return {k: (round(v, 3) if isinstance(v, float) else v) for k, v in res.items()}


def rel_mse(x, t):
    return float(((x - t) ** 2 / (t ** 2 + 1e-2)).mean())


def quality(ctx, aperture):
    """rel-MSE rows of the ring for the default and one-at-a-time parameters."""
    w = h = 128
    ck, depth = (4, 16), 8
    pos = hemisphere(15, 15)[3 * 15:4 * 15]
    ctx.set_lens(aperture, 0)
    s = inputs(ctx, pos, w, h, ck, depth)
    target = np.nan_to_num(ctx.render_views(pos, w, h, 4096, depth)[..., :3].astype(np.float64) / 4096)
    ctx.set_lens(0, 0)
    albm = s["alb"][-1][..., :3] / ck[-1]
    nrm = np.linalg.norm(s["nd"][-1][..., :3] / ck[-1], axis=-1)
    lamb = (albm.max(-1) <= 0.7301) & (nrm > 0.999)
    lamb[:5] = False
    glass = (albm.min(-1) >= 0.999) & (albm.max(-1) <= 1.001) & (s["alb"][-1][..., 3] == ck[-1]) & \
        (target.max(-1) < 5)  # albedo 1 and not the light (emitters have albedo 1 too)
    glass[:5] = False
    sp = ctx.denoise_views(s["color"], s["m2"], s["alb"], s["nd"], w, h, ck)
    p0 = B.DenoiseParams.defaults()
    p0.levels = 0
    rows = []
    variants = [("defaults", {})]
    if aperture == 0:
        for name, vals in (("alpha", (0.05, 0.1, 0.3, 0.5)), ("minVisible", (0.0, 0.25, 0.75, 1.0)),
                           ("normalTol", (0.1, 1.0, float("inf"))), ("albedoTol", (0.03, 0.3, float("inf"))),
                           ("depthTol", (0.02, 0.1, 0.2, float("inf")))):
            variants += [("%s=%g" % (name, v), {name: v}) for v in vals]
    for label, kw in variants:
        tp = B.TemporalParams.defaults()
        for k, v in kw.items():
            setattr(tp, k, v)
        t0, n = ctx.denoise_views_temporal(s["color"], s["m2"], s["alb"], s["nd"], s["mot"], pos, w, h, ck, tp, p0,
                                           history=True)
        tf = ctx.denoise_views_temporal(s["color"], s["m2"], s["alb"], s["nd"], s["mot"], pos, w, h, ck, tp)
        row = dict(workload="temporal_quality_ring3_15x128sq_depth8", aperture=aperture, variant=label)
        for k, c in enumerate(ck):
            noisy = np.nan_to_num(s["color"][k, ..., :3].astype(np.float64)) / c
            row["%dspp" % c] = dict(
                noisy=rel_mse(noisy[lamb], target[lamb]), temporal=rel_mse(t0[k][lamb][:, :3], target[lamb]),
                spatial=rel_mse(sp[k][lamb][:, :3], target[lamb]), temporal_spatial=rel_mse(tf[k][lamb][:, :3],
                                                                                             target[lamb]),
                glass_noisy=rel_mse(noisy[glass], target[glass]), glass_temporal=rel_mse(t0[k][glass][:, :3],
                                                                                         target[glass]),
                glass_spatial=rel_mse(sp[k][glass][:, :3], target[glass]),
                glass_temporal_spatial=rel_mse(tf[k][glass][:, :3], target[glass]),
                mean_n=float(n[k][lamb].mean()), share_n1=float((n[k][lamb] == 1).mean()), glass_pixels=int(glass.sum()),
                glass_mean_n=float(n[k][glass].mean()) if glass.any() else None)
            if label == "defaults":
                m = s["mot"][k]
                speed = np.hypot(m[..., 0], m[..., 1]) / np.maximum(m[..., 3], 1)
                err2 = ((t0[k][..., :3].astype(np.float64) - target) @ LUM) ** 2
                for nm, mk in (("lt1px", speed < 1), ("ge1px", speed >= 1)):
                    sel = lamb & (n[k] >= 3) & mk
                    row["%dspp" % c]["err2_over_Vbar_" + nm] = \
                        [int(sel.sum()), float(err2[sel].mean() / max(t0[k][..., 3][sel].mean(), 1e-30))] \
                        if sel.sum() else [0, None]
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--skip-profile", action="store_true")
    ap.add_argument("--sweep", action="store_true")
    a = ap.parse_args()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    rows = []
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        ctx.build_bvh()
        if a.sweep:
            for aperture in (0.0, 0.05, 0.1):
                rows += [dict(r, **info) for r in quality(ctx, aperture)]
        else:
            s = inputs(ctx, hemisphere(15, 15), W, H, CKPTS, 5)
            fs = calls(ctx, s)
            rows.append(dict(timed(fs, a.reps), **info))
            print(json.dumps(rows[-1]), flush=True)
            if not a.skip_profile:
                rows.append(dict(profile(fs["temporal"], a.out), **info))
                print(json.dumps(rows[-1]), flush=True)
    if a.out:
        with open(os.path.join(a.out, "time_temporal%s.jsonl" % ("_sweep" if a.sweep else "")), "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
