"""Cost of a temporally denoised view sweep in one call (b2pt_render_views_temporal_denoised) against the four-call chain
it is defined as, on cuda:0, Cornell box: the reference's 225-view 128^2 hemisphere, checkpoints 1, 2, 4, ..., 256
(K = 9), depth 5, default parameters (DESIGN.md 8j's workload).

  whole call   host clock around calls that end in a stream synchronise, median of --reps alternating rounds of
               chain       render_views_checkpoints (moments) + render_views_features + render_views_motion (towards the
                           previous view) + denoise_views_temporal, host arrays between the calls;
               one_out     the one call with only the denoised result requested;
               one_all     the one call with every output requested (noisy sums, squares, guides, motion, history).
               The first round checks that one_all returns the chain's bits.
  kernels      in a separate torch.profiler pass over one chain and one one_all call: the GPU time of every kernel
               family and of the copies by direction, and the fused guide/motion kernel (k_view_guides_motion) against
               k_view_features + k_view_motion, which the chain launches on the same chunks of views.
The GPU name and power limit are read in the same run.  One JSON line per measurement goes to stdout (and
OUT/time_temporal_denoised.jsonl with --out).

  python scripts/time_temporal_denoised.py [--out DIR] [--reps 7] [--skip-profile]
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
DEPTH = 5
WORKLOAD = "hemisphere_225x128sq_ckpt1-256_depth5"


def chain_views(views):
    return np.concatenate([views[:1], views[:-1]])


def calls(ctx, views):
    def chain():
        color, m2 = ctx.render_views_checkpoints(views, W, H, CKPTS, DEPTH, 0, moments=True)
        alb, nd = ctx.render_views_features(views, W, H, CKPTS)
        mot = ctx.render_views_motion(views, chain_views(views), W, H, CKPTS)
        out, n = ctx.denoise_views_temporal(color, m2, alb, nd, mot, views, W, H, CKPTS, history=True)
        return out, n, (color, m2, alb, nd, mot)

    return {"chain": chain,
            "one_out": lambda: ctx.render_views_temporal_denoised(views, W, H, CKPTS, DEPTH),
            "one_all": lambda: ctx.render_views_temporal_denoised(views, W, H, CKPTS, DEPTH, history=True,
                                                                  inputs=True)}


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint32),
                                                 np.ascontiguousarray(b).view(np.uint32))


def timed(fs, reps):
    want = fs["chain"]()  # warm-up: modules, trees and staging buffers
    got = fs["one_all"]()
    fs["one_out"]()
    identical = same_bits(got[0], want[0]) and same_bits(got[1], want[1]) and \
        all(same_bits(a, b) for a, b in zip(got[2], want[2]))
    del want, got
    times = {k: [] for k in fs}
    for _ in range(reps):
        for k, f in fs.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    res = dict(workload=WORKLOAD, reps=reps, one_all_is_chain_bits=bool(identical))
    for k, ts in times.items():
        res[k] = dict(ms_median=round(statistics.median(ts), 2), ms_range=[round(min(ts), 2), round(max(ts), 2)])
    for k in ("one_out", "one_all"):
        res["chain_over_" + k] = round(res["chain"]["ms_median"] / res[k]["ms_median"], 3)
    return res


FAMILIES = ("k_view_guides_motion", "k_view_features", "k_view_motion", "k_denoise_prep", "k_temporal", "k_atrous",
            "k_pnm16")


def profile(name, f, out):
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    if out:
        prof.export_chrome_trace(os.path.join(out, "temporal_denoised_%s.json" % name))
    res = dict(workload=WORKLOAD + "_profile", call=name, gpu_ms=0.0, render_kernels_ms=0.0, memcpy_HtoD_ms=0.0,
               memcpy_DtoH_ms=0.0, memcpy_DtoD_ms=0.0, memset_ms=0.0)
    for fam in FAMILIES:
        res[fam + "_ms"] = 0.0
    for ev in prof.key_averages():
        dev = getattr(ev, "device_time_total", None)
        if dev is None:
            dev = getattr(ev, "cuda_time_total", 0)
        if not dev or ev.key.startswith("cuda") or ev.key.startswith("aten"):
            continue
        ms = dev / 1e3
        res["gpu_ms"] += ms
        key = ev.key.lower()
        if "memcpy" in key:
            d = "HtoD" if "htod" in key else "DtoH" if "dtoh" in key else "DtoD"
            res["memcpy_%s_ms" % d] += ms
        elif "memset" in key:
            res["memset_ms"] += ms
        else:
            fam = next((f for f in FAMILIES if "::%s<" % f in ev.key or "::%s(" % f in ev.key), None)
            if fam is None:
                res["render_kernels_ms"] += ms
            else:
                res[fam + "_ms"] += ms
    return {k: (round(v, 3) if isinstance(v, float) else v) for k, v in res.items()}


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
    views = hemisphere(15, 15)
    with B.Context(0) as ctx:
        ctx.set_scene(B.Scene.cornell())
        ctx.build_bvh()
        fs = calls(ctx, views)
        rows.append(dict(timed(fs, a.reps), **info))
        print(json.dumps(rows[-1]), flush=True)
        if not a.skip_profile:
            prof = {}
            for name in ("chain", "one_all"):
                prof[name] = profile(name, fs[name], a.out)
                rows.append(dict(prof[name], **info))
                print(json.dumps(rows[-1]), flush=True)
            sep = prof["chain"]["k_view_features_ms"] + prof["chain"]["k_view_motion_ms"]
            fused = prof["one_all"]["k_view_guides_motion_ms"]
            rows.append(dict(workload=WORKLOAD + "_guides_motion", separate_ms=round(sep, 3),
                             fused_ms=round(fused, 3), separate_over_fused=round(sep / fused, 3) if fused else None,
                             **info))
            print(json.dumps(rows[-1]), flush=True)
    if a.out:
        with open(os.path.join(a.out, "time_temporal_denoised.jsonl"), "w") as fo:
            for r in rows:
                fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
