"""Time the images of one view sweep at several sample counts on cuda:0, host outputs in every way:
  ckpt     one b2pt_render_views_checkpoints call (float4 sums of every checkpoint)
  ckpt_m2  the same call with the per-pixel sums of squares as well
  loop     one b2pt_render_views call per checkpoint (what a caller without checkpoints does)
  last     one b2pt_render_views call at the last checkpoint only: ckpt / last is the cost of the snapshots and of the
           larger copy to the host
Workloads: the reference's 225-view hemisphere (generateHemisphere, 15 x 15) at 128^2, depth 50, checkpoints 1, 2, 4,
..., 256 (views share batches: the flat view-batched path); one 1024^2 view, depth 50, checkpoints 1, 2, 4, ..., 1024
(the per-view fallback: several sample batches per view).

Every way is called through the C-ABI with preallocated, pre-touched host arrays after one warm-up call each; then the
repetitions alternate the four ways, each timed by the host wall clock around a call that ends in a stream synchronise,
and the median is reported.  The checkpointed slices are checked bit for bit against the loop's images.  The GPU name
and power limit are read in the same run.  One JSON line per workload goes to stdout (and OUT/time_checkpoints.jsonl
with --out), then a markdown table.

  python scripts/time_checkpoints.py [--out DIR] [--reps 5]
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

WAYS = ("ckpt", "ckpt_m2", "loop", "last")


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
        img = {w: np.ones((K, V, N, 4), np.float32) for w in ("ckpt", "ckpt_m2", "loop")}
        m2 = np.ones((K, V, N, 4), np.float32)
        last = np.ones((V, N, 4), np.float32)
        paths = {}

        def run(way):
            if way in ("ckpt", "ckpt_m2"):
                B._check(L.b2pt_render_views_checkpoints(h, V, p(views), W, H, K, p(ck), depth, 0, p(img[way]),
                                                         p(m2) if way == "ckpt_m2" else None))
            elif way == "loop":
                for k, c in enumerate(ck):
                    B._check(L.b2pt_render_views(h, V, p(views), W, H, int(c), depth, 0, p(img["loop"][k])))
            else:
                B._check(L.b2pt_render_views(h, V, p(views), W, H, int(ck[-1]), depth, 0, p(last)))

        for w in WAYS:  # warm-up: module load, batch buffers, tail-mode depths
            run(w)
            paths[w] = ctx.stats().paths
        t = {w: [] for w in WAYS}
        for _ in range(a.reps):
            for w in WAYS:
                t0 = time.perf_counter()
                run(w)
                t[w].append(time.perf_counter() - t0)
        same = all(np.array_equal(img[w].view(np.uint32), img["loop"].view(np.uint32)) for w in ("ckpt", "ckpt_m2"))
        same = same and np.array_equal(last.view(np.uint32), img["ckpt"][-1].view(np.uint32))
        med = {w: float(np.median(v)) for w, v in t.items()}
        traced = {"ckpt": int(ck[-1]), "ckpt_m2": int(ck[-1]), "loop": int(ck.sum()), "last": int(ck[-1])}
        rec = dict(info, workload=name, views=V, canvas=[W, H], depth=depth, checkpoints=ck.tolist(), reps=a.reps,
                   seconds=t, median_seconds=med, spp_traced=traced, paths_last_call=paths,
                   loop_over_ckpt=med["loop"] / med["ckpt"], ckpt_over_last=med["ckpt"] / med["last"],
                   ckpt_m2_over_ckpt=med["ckpt_m2"] / med["ckpt"], bit_identical=bool(same))
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        rows.append("| %s | %d x %d^2, ck %d..%d | %.1f | %.1f | %.1f | %.1f | %.2f | %.3f |" % (
            name, V, W, ck[0], ck[-1], 1e3 * med["ckpt"], 1e3 * med["ckpt_m2"], 1e3 * med["loop"], 1e3 * med["last"],
            rec["loop_over_ckpt"], rec["ckpt_over_last"]))
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_checkpoints.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")
    print("\n%s, power limit %s (median of %d)\n" % (info.get("gpu"), info.get("power_limit"), a.reps))
    print("| workload | views | checkpointed ms | + moments ms | loop ms | render_views(c_K) ms | loop / ckpt | "
          "ckpt / c_K |")
    print("|---|---|---|---|---|---|---|---|")
    print("\n".join(rows))


if __name__ == "__main__":
    main()
