"""Time the denoiser guide buffers of one view sweep on cuda:0, next to the radiance images they describe:
  features  one b2pt_render_views_features call (albedo and normal/depth sums at every checkpoint, both outputs)
  ckpt      one b2pt_render_views_checkpoints call of the same views and checkpoints, depth 50 (the noisy inputs and
            target the guides go with)
Workloads: the reference's 225-view hemisphere (generateHemisphere, 15 x 15) at 128^2, checkpoints 1, 2, 4, ..., 256;
one 1024^2 view, checkpoints 1, 2, 4, ..., 1024.  Cornell box.

Both ways are called through the C-ABI with preallocated, pre-touched host arrays after one warm-up call each; then the
repetitions alternate the two ways, each timed by the host wall clock around a call that ends in a stream synchronise,
and the median is reported.  The GPU name and power limit are read in the same run.  One JSON line per workload goes to
stdout (and OUT/time_features.jsonl with --out), then a markdown table.

  python scripts/time_features.py [--out DIR] [--reps 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import raytracingtherestofyourlife_b200 as B  # noqa: E402
from time_direct_views import gpu_info, hemisphere, p, row  # noqa: E402

WAYS = ("features", "ckpt")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    L = B.lib()
    info = gpu_info()
    info["torch_device"] = torch.cuda.get_device_name(0)
    ctx = B.Context(0)
    ctx.set_scene(B.Scene.cornell())
    ctx.build_bvh()
    h = ctx._h
    depth = 50
    lines, rows = [], []
    default_view = row([278 / 555.0, 278 / 555.0, -800 / 555.0])[None]  # main.cc:616-622
    for name, views, W, H, top in [("hemisphere_225_128", hemisphere(15, 15), 128, 128, 256),
                                   ("one_view_1024", default_view, 1024, 1024, 1024)]:
        ck = np.array([1 << i for i in range(top.bit_length())], np.int32)
        K, V, N = len(ck), views.shape[0], W * H
        alb = np.ones((K, V, N, 4), np.float32)
        nd = np.ones((K, V, N, 4), np.float32)
        img = np.ones((K, V, N, 4), np.float32)

        def run(way):
            if way == "features":
                B._check(L.b2pt_render_views_features(h, V, p(views), W, H, K, p(ck), 0, p(alb), p(nd)))
            else:
                B._check(L.b2pt_render_views_checkpoints(h, V, p(views), W, H, K, p(ck), depth, 0, p(img), None))

        for w in WAYS:  # warm-up: module load, staging buffers
            run(w)
        first = (alb.copy(), nd.copy())
        t = {w: [] for w in WAYS}
        for _ in range(a.reps):
            for w in WAYS:
                t0 = time.perf_counter()
                run(w)
                t[w].append(time.perf_counter() - t0)
        repeatable = all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(first, (alb, nd)))
        med = {w: float(np.median(v)) for w, v in t.items()}
        rays = int(ck[-1]) * V * N  # primary rays the feature pass traces
        host_bytes = 2 * K * V * N * 16  # both outputs, copied to the host
        rec = dict(info, workload=name, views=V, canvas=[W, H], depth=depth, checkpoints=ck.tolist(), reps=a.reps,
                   seconds=t, median_seconds=med, feature_rays=rays, feature_host_bytes=host_bytes,
                   feature_rays_per_s=rays / med["features"], features_over_ckpt=med["features"] / med["ckpt"],
                   repeatable=bool(repeatable), hit_fraction=float(alb[-1][..., 3].sum() / (ck[-1] * V * N)))
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        rows.append("| %s | %d x %d^2, ck %d..%d | %.1f | %.1f | %.3f | %.2f G |" % (
            name, V, W, ck[0], ck[-1], 1e3 * med["features"], 1e3 * med["ckpt"], rec["features_over_ckpt"],
            rec["feature_rays_per_s"] * 1e-9))
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_features.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")
    print("\n%s, power limit %s (median of %d)\n" % (info.get("gpu"), info.get("power_limit"), a.reps))
    print("| workload | views | features ms | render_views_checkpoints ms | features / ckpt | feature rays/s |")
    print("|---|---|---|---|---|---|")
    print("\n".join(rows))


if __name__ == "__main__":
    main()
