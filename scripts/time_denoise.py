"""Time the spatial denoiser of one view sweep (b2pt_denoise_views) on cuda:0, next to the render that produced its input:
  call      wall time of one b2pt_denoise_views call (float output, default parameters), host clock around a call that
            ends in a stream synchronise; pageable host arrays, as a Python user passes them
  kernels   the k_denoise_prep / k_atrous / k_pnm16 time of the same call from torch.profiler (a separate run), and
            the copies it lists
  render    one b2pt_render_views_checkpoints call with sums of squares (depth 5) of the same views and checkpoints
Workloads: the reference's 225-view hemisphere (generateHemisphere, 15 x 15) at 128^2, checkpoints 1, 2, 4, ..., 256
(K = 9); one 1024^2 view, checkpoints 1, 2, 4, ..., 1024 (K = 11).  Cornell box.  H2D / D2H bytes are computed from
the shapes (4 float4 inputs in, one float4 out per pixel and slice).

--quality also prints the rel-MSE against a 4096-spp target of 8 views at 128^2, checkpoints (4, 16, 64), for the
default parameters and a few variations of each sigma (the measurements behind the defaults, DESIGN.md 8e).

The GPU name and power limit are read in the same run.  One JSON line per workload goes to stdout (and
OUT/time_denoise.jsonl with --out).

  python scripts/time_denoise.py [--out DIR] [--reps 5] [--quality]
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
from time_direct_views import gpu_info, hemisphere, p, row  # noqa: E402


def kernel_profile(ctx, args, out_dir):
    """torch.profiler over one call: per-kernel device time and the listed copies (ms)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ctx.denoise_views(*args)
        torch.cuda.synchronize()
    res = {}
    for ev in prof.key_averages():
        dev = getattr(ev, "device_time_total", None)
        if dev is None:
            dev = getattr(ev, "cuda_time_total", 0)
        if dev and ("k_atrous" in ev.key or "k_denoise_prep" in ev.key or "k_pnm16" in ev.key or "Memcpy" in ev.key):
            res[ev.key[:60]] = round(dev / 1e3, 3)
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, "time_denoise_trace.json"))
    return res


def quality(ctx):
    tilted = []
    c = 278 / 555.0
    for v in range(8):
        ang = 0.35 * (v - 3.5) / 8
        pos = [c + 1.95 * np.sin(ang), c + 0.1 * (v % 3), c - 1.95 * np.cos(ang)]
        tilted.append(row(pos))
    views = np.stack(tilted)
    w = h = 128
    ck = (4, 16, 64)
    color, m2 = ctx.render_views_checkpoints(views, w, h, ck, 5, 0, moments=True)
    alb, nd = ctx.render_views_features(views, w, h, ck)
    target = np.nan_to_num(ctx.render_views(views, w, h, 4096, 5)[..., :3].astype(np.float64) / 4096)

    def rel(x):
        return [round(float(((x[k] - target) ** 2 / (target ** 2 + 1e-2)).mean()), 6) for k in range(len(ck))]
    noisy = np.nan_to_num(color[..., :3].astype(np.float64)) / np.array(ck, np.float64)[:, None, None, None]
    rows = [dict(setting="noisy", relmse=rel(noisy))]
    d = B.DenoiseParams.defaults()
    grid = [("defaults", {})]
    for name, vals in (("levels", (3, 4, 6)), ("sigmaLum", (1.0, 2.0, 8.0, float("inf"))),
                       ("sigmaAlbedo", (0.05, 0.2, 0.5)), ("sigmaNormal", (0.1, 0.6, 1.0)),
                       ("sigmaDepth", (0.5, 1.0, 4.0, 8.0))):
        grid += [("%s=%g" % (name, v), {name: v}) for v in vals]
    for label, change in grid:
        prm = B.DenoiseParams.defaults()
        for k, v in change.items():
            setattr(prm, k, v)
        out = ctx.denoise_views(color, m2, alb, nd, w, h, ck, prm)
        rows.append(dict(setting=label, relmse=rel(out[..., :3].astype(np.float64))))
    return dict(workload="quality_8x128", checkpoints=ck, defaults=[d.levels, d.sigmaLum, d.sigmaAlbedo,
                                                                     d.sigmaNormal, d.sigmaDepth], rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quality", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    L = B.lib()
    info = gpu_info()
    ctx = B.Context(0)
    ctx.set_scene(B.Scene.cornell())
    ctx.build_bvh()
    h = ctx._h
    lines = []
    default_view = row([278 / 555.0, 278 / 555.0, -800 / 555.0])[None]  # main.cc:616-622
    for name, views, W, H, top in [("hemisphere_225_128", hemisphere(15, 15), 128, 128, 256),
                                   ("one_view_1024", default_view, 1024, 1024, 1024)]:
        ck = np.array([1 << i for i in range(top.bit_length())], np.int32)
        K, V, N = len(ck), views.shape[0], W * H
        color = np.empty((K, V, N, 4), np.float32)
        m2 = np.empty_like(color)
        B._check(L.b2pt_render_views_checkpoints(h, V, p(views), W, H, K, p(ck), 5, 0, p(color), p(m2)))
        alb, nd = ctx.render_views_features(views, W, H, ck)
        out = np.empty_like(color)
        prm = B.DenoiseParams.defaults()
        args = (color, m2, alb, nd, W, H, ck, prm)
        ctx.denoise_views(*args)  # warm-up (staging allocation)
        t_call, t_render = [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            B._check(L.b2pt_denoise_views(h, V, W, H, K, p(ck), p(color), p(m2), p(alb), p(nd), None, 0, p(out)))
            t_call.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            B._check(L.b2pt_render_views_checkpoints(h, V, p(views), W, H, K, p(ck), 5, 0, p(color), p(m2)))
            t_render.append((time.perf_counter() - t0) * 1e3)
        kern = kernel_profile(ctx, args, a.out)
        h2d, d2h = 4 * K * V * N * 16, K * V * N * 16
        kernel_ms = sum(v for k, v in kern.items() if "Memcpy" not in k)
        call_ms = statistics.median(t_call)
        res = dict(workload=name, views=V, W=W, H=H, checkpoints=K, levels=prm.levels,
                   call_ms=round(call_ms, 3), call_ms_range=[round(min(t_call), 3), round(max(t_call), 3)],
                   kernel_ms=round(kernel_ms, 3), kernel_share=round(kernel_ms / call_ms, 4), profile=kern,
                   h2d_bytes=h2d, d2h_bytes=d2h, render_ms=round(statistics.median(t_render), 3),
                   render_ms_range=[round(min(t_render), 3), round(max(t_render), 3)], **info)
        lines.append(res)
        print(json.dumps(res), flush=True)
        del color, m2, alb, nd, out
    if a.quality:
        q = quality(ctx)
        q.update(info)
        lines.append(q)
        print(json.dumps(q), flush=True)
    ctx.close()
    if a.out:
        with open(os.path.join(a.out, "time_denoise.jsonl"), "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()
