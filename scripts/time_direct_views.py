"""Time the -direct G-buffers of the camera sweeps (main.cc:386-561 with -direct) two ways on cuda:0, host outputs in
both:
  loop     one b2pt_set_camera + b2pt_render_direct per view (what a port of the reference's generate() loop does)
  batched  one b2pt_render_direct_views call for the whole view list
Workloads: the reference's 225-view hemisphere at 128^2 (15 x 15, generateHemisphere), the 5000 views of the lower half
of the default 10000-point Fibonacci lattice at 128^2 (fibonacciHemisphere), and the 64 views of a 128-point lattice at 512^2.

Both ways are called through the C-ABI with preallocated, pre-touched host arrays (no page faults, no numpy allocation in
the timed window), after one warm-up call each; then at least three repetitions alternate loop and batched, each timed by
the host wall clock around calls that end in a stream synchronise.  Reported: views/s, the bytes per second of the
device-to-host copy the outputs need (40 B per pixel: normals and albedo float4, depth float, primitive id int32), and,
as the yardstick for that copy, a plain pageable device-to-host copy of the same bytes (torch, one chunk of 2^22 pixels
at a time).  The GPU name and power limit are read in the same run.  One JSON line per workload goes to
OUT/time_direct_views.jsonl and to stdout.

  python scripts/time_direct_views.py --out DIR [--reps 3]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import raytracingtherestofyourlife_b200 as B  # noqa: E402

CTR = 278 / 555.0
BYTES_PER_PIXEL = 40


def row(pos):
    return np.array(list(pos) + [CTR] * 3 + [0, 1, 0, 40.0], np.float32)


def hemisphere(n_phi, n_theta):
    """generateHemisphere's view points (host/main.cc, float32 arithmetic)."""
    f = np.float32
    theta_end = f(2 * math.pi)
    r_theta, r_phi, r = f(theta_end / f(n_theta)), f(f(1) / f(n_phi)), f(-1078 / 555.0)
    out, phi = [], f(0)
    while float(phi) < 1.0 - 0.5 * float(r_phi):
        theta = f(0)
        while theta < theta_end:
            x = f(f(r * f(math.cos(theta))) * f(math.sin(phi)))
            y = f(f(r * f(math.sin(theta))) * f(math.sin(phi)))
            z = f(r * f(math.cos(phi)))
            out.append(row([float(x) + CTR, float(y) + CTR, float(z) + CTR]))
            theta = f(theta + r_theta)
        phi = f(phi + r_phi)
    return np.stack(out)


def fibonacci(n=10000, rnd=0):
    """fibonacciHemisphere's view points (host/main.cc): the lattice points with z < 0."""
    offset, inc = np.float32(2.0 / n), math.pi * (3.0 - math.sqrt(5.0))
    out = []
    for i in range(n):
        z = np.float32(np.float32(np.float32(i * offset) - np.float32(1)) + np.float32(offset / np.float32(2)))
        r = np.float32(math.sqrt(1 - float(z) ** 2))
        phi = ((i + rnd) % n) * inc
        if z < 0:
            out.append(row([float(np.float32(math.cos(phi) * float(r))) + CTR,
                            float(np.float32(math.sin(phi) * float(r))) + CTR, float(z) + CTR]))
    return np.stack(out)


def gpu_info():
    info = {}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in q[0].split(",")]
        info.update(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers stay usable; the missing card description is reported
        info["gpu_query_error"] = repr(e)
    return info


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
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
    lines = []
    for name, views, W, H in [("hemisphere_225_128", hemisphere(15, 15), 128, 128),
                              ("fibonacci_5000_128", fibonacci(), 128, 128),
                              ("fibonacci_64_512", fibonacci(128), 512, 512)]:
        V, N = views.shape[0], W * H
        outs = {m: [np.ones((V, N, 4), np.float32), np.ones((V, N, 4), np.float32), np.ones((V, N), np.float32),
                    np.ones((V, N), np.int32)] for m in ("loop", "batched")}

        def loop():
            nrm, alb, dep, prim = outs["loop"]
            for k, v in enumerate(views):
                B._check(L.b2pt_set_camera(h, p(v[0:3]), p(v[3:6]), p(v[6:9]), float(v[9]), W, H))
                B._check(L.b2pt_render_direct(h, p(nrm[k]), p(alb[k]), p(dep[k]), p(prim[k])))

        def batched():
            nrm, alb, dep, prim = outs["batched"]
            B._check(L.b2pt_render_direct_views(h, V, p(views), W, H, p(nrm), p(alb), p(dep), p(prim)))

        loop()  # warm-up: module load, staging buffers
        batched()
        t = {"loop": [], "batched": []}
        for _ in range(a.reps):
            for m, fn in (("loop", loop), ("batched", batched)):
                t0 = time.perf_counter()
                fn()
                t[m].append(time.perf_counter() - t0)
        same = all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(outs["loop"], outs["batched"]))
        # yardstick: the same bytes through plain pageable device-to-host copies, one 2^22-pixel chunk at a time
        nbytes = V * N * BYTES_PER_PIXEL
        chunk = min(nbytes, (1 << 22) * BYTES_PER_PIXEL)
        dev = torch.empty(chunk, dtype=torch.uint8, device="cuda")
        host = torch.from_numpy(np.ones(chunk, np.uint8))
        host.copy_(dev)
        torch.cuda.synchronize()
        tc = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            done = 0
            while done < nbytes:
                host.copy_(dev)
                done += chunk
            torch.cuda.synchronize()
            tc.append(time.perf_counter() - t0)
        del dev, host, outs
        best = {m: min(v) for m, v in t.items()}
        med = {m: float(np.median(v)) for m, v in t.items()}
        rec = dict(info, workload=name, views=V, canvas=[W, H], pixels=V * N, d2h_bytes=nbytes, reps=a.reps,
                   seconds=t, copy_seconds=tc,
                   loop_views_per_s=V / med["loop"], batched_views_per_s=V / med["batched"],
                   speedup=med["loop"] / med["batched"],
                   loop_d2h_bytes_per_s=nbytes / med["loop"], batched_d2h_bytes_per_s=nbytes / med["batched"],
                   plain_copy_bytes_per_s=nbytes / float(np.median(tc)),
                   batched_over_plain_copy_time=med["batched"] / float(np.median(tc)),
                   best_loop_views_per_s=V / best["loop"], best_batched_views_per_s=V / best["batched"],
                   bit_identical=bool(same))
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    ctx.close()
    with open(os.path.join(a.out, "time_direct_views.jsonl"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
