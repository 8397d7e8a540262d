#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native path tracer (contract: see the task statement / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--spp S] [--size W] [--dump-outputs DIR]

One "step" = one full render of the workload through the hot path:
  workload (N=1)  BASELINE.json configs[1]: Cornell box 1024x1024, 1024 spp, max depth 50
  N>1 (torchrun)  weak scaling: every rank renders its own 1024 samples of every pixel (global sample
                  indices [rank*1024, (rank+1)*1024)), then ONE NCCL all-reduce (sum) of the W*H float4
                  radiance sums -- the only exchange step of the path (SURVEY.md 8e).
value  = path samples/s over all ranks, device-timed (CUDA events on the launching stream, max over ranks),
         scene/BVH/camera already resident in HBM.
e2e    = same metric through the C-ABI with HOST buffers inside the timed region: b2pt_set_scene (H2D of the
         scene arrays) + b2pt_build_bvh + b2pt_set_camera + b2pt_render + b2pt_read_color (D2H of the W*H*16 B
         radiance sum into pinned host memory).
--impl reference  times the reference's own CPU code on the box's host cores: its header-only worklets compiled
         from the reference sources (oracle/_ref, built by oracle/Makefile against a minimal VTK-m stand-in) and
         launched in the reference's order, one OpenMP parallel-for per worklet launch (kind "reference").  When
         that library is absent the C restatement (oracle PASSES mode) is timed instead (kind "port").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cornell_1024_path_samples_per_s"
UNIT = "path samples/s"


def metric_name(size):
    return METRIC if size == 1024 else "cornell_%d_path_samples_per_s" % size


def workload_label(size, total_spp, depth, world):
    """One string for both arms (this arm and --impl reference): the workload of the whole job."""
    if size == 1024 and total_spp == 1024 and depth == 50:
        tag = "BASELINE.json configs[1]"
    elif size == 1024 and total_spp == 4096 and depth == 50:
        tag = "north_star target: 1024^2 x 4096 spp"
    elif size == 4096 and total_spp == 4096 and depth == 50:
        tag = "BASELINE.json configs[2]"
    else:
        tag = "a variation of BASELINE.json configs[1]"
    return "Cornell box %dx%d, %d spp, max depth %d (%s)" % (size, size, total_spp, depth, tag)


def job_spp(args, world):
    """Samples per pixel of the whole job.  N=1: BASELINE.json configs[1] (1024 spp).  N>1: a FIXED job -- the
    north_star target, 1024^2 x 4096 spp -- whose samples are partitioned over the ranks (strong scaling); --weak keeps
    the per-GPU work fixed instead (args.spp samples per rank)."""
    if world == 1:
        return args.spp
    if args.weak:
        return args.spp * world
    return args.total_spp


ALGO_BYTES_PER_SEGMENT = 88  # SURVEY.md 8d: 44 B ray record read + 44 B written per live segment


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2pt", choices=["b2pt", "reference"])
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--depth", type=int, default=50)
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-image-check", action="store_true")
    ap.add_argument("--ref-spp", type=int, default=1, help="samples per step of the CPU reference arm")
    ap.add_argument("--total-spp", type=int, default=4096, help="N>1: samples per pixel of the whole (fixed) job")
    ap.add_argument("--weak", action="store_true", help="N>1: weak scaling, --spp samples per rank")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the radiance sum of the last timed step to DIR/radiance_sum.npy (float32 [W*H, 4], "
                         "NaN-poisoned channels as 0) and where they were to DIR/radiance_sum_nonfinite.npy; above %d "
                         "MB in all a fixed, seeded sample of pixel rows" % (DUMP_LIMIT_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 4096  # upper bound of one .npy header (numpy writes 128 bytes for these shapes)


def dump_outputs(out_dir, **arrays):
    """Saves each array as out_dir/<name>.npy with finite values only: a non-finite entry (a NaN-poisoned pixel sum) is
    stored as 0, as the reference's NormalizeFunctor de-NaNs it, and out_dir/<name>_nonfinite.npy holds 1 where that
    happened (the mask does not tell NaN from inf).  The inputs of a run are fixed by its arguments (scene, camera, sample
    range, seed offset 0), so two builds can be compared file for file.  When the files, headers included, would exceed
    DUMP_LIMIT_BYTES in all, every file keeps the same sorted sample of rows drawn with a fixed seed: the same rows for
    the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        bad = ~np.isfinite(a)
        out[name] = np.where(bad, 0, a).astype(a.dtype)
        out[name + "_nonfinite"] = bad.astype(a.dtype)
    rows = {a.shape[0] for a in out.values()}.pop()  # every output has one row per pixel
    payload = DUMP_LIMIT_BYTES - NPY_HEADER_BYTES * len(out)
    total = sum(a.nbytes for a in out.values())
    if total > payload:
        keep = np.sort(np.random.default_rng(0).choice(rows, payload // (total // rows), replace=False))
        out = {name: a[keep] for name, a in out.items()}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): through NVML
    (nvidia_ml_py, ~1 ms per sample) when it loads, else through the nvidia-smi command line of the recipe."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(index))
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        nv, h = self.nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bit = lambda name: "Active" if (r & getattr(nv, name, 0)) else "Not Active"
        return [str(sm), str(mx), "0", bit("nvmlClocksThrottleReasonHwSlowdown"),
                bit("nvmlClocksThrottleReasonHwThermalSlowdown"), bit("nvmlClocksThrottleReasonSwThermalSlowdown"),
                bit("nvmlClocksThrottleReasonSwPowerCap")]

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                         timeout=5).stdout
                    parts = [p.strip() for p in out.strip().split(",")]
                    if len(parts) >= 7:
                        self.rows.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.05 if self.nvml else 0.2)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "via": "nvml" if self.nvml else "nvidia-smi"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, or None."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def cpu_reference_arm():
    """(kind, description, step) of the CPU arm: the reference's own worklets when oracle/_ref is available, else
    the C restatement.  step(W, spp, depth, threads) -> (paths_per_s, seconds, paths)."""
    from oracle import oracle as O
    O.build()
    try:
        from oracle import refharness as R
        have_ref = R.available()
    except Exception:
        have_ref = False
    if have_ref:
        build = ["?"]

        def step(W, spp, depth, threads):
            os.environ["OMP_NUM_THREADS"] = str(threads)
            try:
                import ctypes
                ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(threads))  # libgomp may be loaded already
            except Exception:
                pass
            t0 = time.perf_counter()
            _, _, build[0] = R.render_timed(O.cornell_scene(), O.Camera(W, W), spp, depth)
            dt = time.perf_counter() - t0
            return W * W * spp / dt, dt, W * W * spp
        desc = ("the reference's own worklets (Surface.h, BVHTraverser.h, EmitWorklet.h, PdfWorklet.h, ScatterWorklet.h ...) "
                "compiled from its sources against a minimal VTK-m stand-in, launched in the order of "
                "MapperPathTracer.cxx:276-351, one OpenMP parallel-for per worklet launch (VTK-m itself is not installable "
                "here)")
        return "reference", desc, step, build

    def step(W, spp, depth, threads):
        t0 = time.perf_counter()
        img, st = O.render(O.cornell_scene(), O.Camera(W, W), spp, depth, mode=O.MODE_PASSES, threads=threads)
        dt = time.perf_counter() - t0
        return st.paths / dt, dt, st.paths
    return "port", ("CPU restatement (VTK-m-structured): oracle PASSES mode, OpenMP, all host cores; the reference "
                    "itself needs VTK-m, which is not installable here"), step, ["-O2 -ffp-contract=off"]


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(args.gpus, int(os.environ.get("WORLD_SIZE", "1")))
    total_spp = job_spp(args, world)
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)  # torchrun presets 1; must be set before libgomp is loaded
    kind, desc, step, build = cpu_reference_arm()
    for _ in range(args.warmup):
        step(args.size, args.ref_spp, args.depth, cores)
    t0 = time.perf_counter()
    paths = 0
    for _ in range(args.steps):
        paths += step(args.size, args.ref_spp, args.depth, cores)[2]
    dt = time.perf_counter() - t0
    val = paths / dt
    one = step(args.size, 1, args.depth, 1)  # VTK-m Serial stand-in: the same code on one thread
    sample = "%dx%d, depth %d, %d spp per step (cost is exactly linear in spp; the job is %d spp); built %s" % (
        args.size, args.size, args.depth, args.ref_spp, total_spp, build[0])
    line = {
        "impl": "reference", "metric": metric_name(args.size), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(args.size, total_spp, args.depth, world), "reference_arm": desc},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "one_thread_value": one[0]},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


RMSE_TOLERANCE = 0.02  # stated tolerance of the image check: relative RMSE over 8x8-pixel blocks of the 256^2 image
MEAN_TOLERANCE = 0.01  # ... and per-channel mean radiance


def image_check(img_sum, total_spp, size, depth):
    """RMSE vs the reference image (BASELINE.json metric, second half): the GPU image box-filtered to 256^2 against the
    committed reference-stream render of the CPU oracle (256^2, 4096 spp, depth 50: tests/golden/
    cornell256_refstream_4096spp.npz, made by tests/golden/make_reference_image.py; the oracle's reference-stream mode
    is pinned bit for bit to the reference's own worklets).  NaN-poisoned pixels (reference semantics: a NaN sample
    poisons its pixel's sum, main.cc:261-268 zeroes it at the end) are MASKED on both sides, not counted as black."""
    import numpy as np
    fix = os.path.join(ROOT, "tests", "golden", "cornell256_refstream_4096spp.npz")
    if size % 256 != 0 or depth != 50 or not os.path.exists(fix):
        return None
    z = np.load(fix)
    parts = z["parts"].astype(np.float64)  # [2, 256*256, 3]: two independent halves of 2048 spp each
    f = size // 256
    ref = parts.mean(0).reshape(256, 256, 3)  # NaN wherever a part is NaN
    g_full = (img_sum[:, :3].astype(np.float64) / total_spp).reshape(256, f, 256, f, 3)
    with np.errstate(invalid="ignore"):
        g = np.nanmean(g_full, axis=(1, 3)) if np.isnan(g_full).any() else g_full.mean((1, 3))
    ok = ~(np.isnan(ref).any(-1) | np.isnan(g).any(-1))  # [256,256]

    def blocks(x):
        w = ok[..., None].astype(np.float64)
        num = (np.where(ok[..., None], x, 0.0)).reshape(32, 8, 32, 8, 3).sum((1, 3))
        den = np.maximum(w.reshape(32, 8, 32, 8, 1).sum((1, 3)), 1.0)
        return num / den

    bg, bo = blocks(g), blocks(ref)
    rel_rmse = float(np.sqrt(((bg - bo) ** 2).mean()) / bo.mean())
    mo, mg = ref[ok].mean(0), g[ok].mean(0)
    mean_err = (np.abs(mg - mo) / mo).tolist()
    # the fixture's own Monte-Carlo noise at the same block size: half the RMSE between its two halves
    h0, h1 = blocks(parts[0].reshape(256, 256, 3)), blocks(parts[1].reshape(256, 256, 3))
    noise = float(0.5 * np.sqrt(((h0 - h1) ** 2).mean()) / bo.mean())
    return {"rel_rmse_8x8_blocks_vs_reference_stream_256x256_4096spp": rel_rmse, "per_channel_mean_rel_err": mean_err,
            "tolerance": {"rel_rmse": RMSE_TOLERANCE, "per_channel_mean": MEAN_TOLERANCE},
            "pass": bool(rel_rmse <= RMSE_TOLERANCE and max(mean_err) <= MEAN_TOLERANCE),
            "reference_image_own_noise_rel_rmse": noise,
            "nan_poisoned_pixels": int(np.isnan(img_sum[:, :3]).any(1).sum()),
            "nan_poisoned_pixels_reference_256x256": int(np.isnan(ref).any(-1).sum()),
            "masked": "NaN-poisoned pixels excluded on both sides"}


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (the NCCL version banner, torchrun's notices) write to file
    descriptor 1 as well, so everything but the result line is sent to stderr: fd 1 is pointed at fd 2 for the
    lifetime of the process and the result is written to a saved duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import raytracingtherestofyourlife_b200 as B
    from raytracingtherestofyourlife_b200.sharding import shard_samples

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = H = args.size
    N = W * H
    total_spp = job_spp(args, world)
    strong = world > 1 and not args.weak
    begin, count = shard_samples(total_spp, rank, world)

    scene, cam = B.Scene.cornell(), B.Camera(W, H)
    ctx = B.Context(local)
    # A dedicated (non-default) torch stream carries everything: the library's kernels (b2pt_set_stream), the NCCL
    # all-reduce and the timing events.  torch's default stream has handle 0, which b2pt_set_stream treats as "use
    # the context's own non-blocking stream" -- events recorded on stream 0 would then not see the kernels.
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    color = torch.zeros((N, 4), dtype=torch.float32, device="cuda")
    ctx.set_scene(scene)
    ctx.build_bvh()
    ctx.set_camera(cam)
    ctx.set_color_tensor(color)

    def step():
        ctx.clear_color()
        ctx.render_range(begin, count, args.depth, args.flags)
        if world > 1:
            dist.all_reduce(color, op=dist.ReduceOp.SUM)

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    fence()
    st = ctx.stats()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    fence()
    sampler.stop_flag.set()
    sampler.join()
    ms = ev0.elapsed_time(ev1)
    st = ctx.stats()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    seg = torch.tensor([float(st.segments)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(seg, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    segments_per_step = float(seg.item())
    paths_per_step = float(N) * total_spp
    value = paths_per_step * args.steps / (ms * 1e-3)
    img_sum = color.cpu().numpy()  # the last timed step's radiance sum (every step clears the canvas first)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, radiance_sum=img_sum)
    # Per-launch durations for the roofline: the timed steps keep 4 sample batches in flight on 4 streams, so their
    # launches overlap and a launch's own duration cannot be read off them.  One extra render of a single batch with
    # B2PT_FLAG_NO_OVERLAP (outside the timed region, same stream, CUDA events around every launch) times the
    # dominant launches alone.
    ctx.render_range(begin, min(count, st.samplesPerBatch), args.depth, args.flags | B.FLAG_NO_OVERLAP)
    ctx_profile = ctx.stage_profile(16)  # (trace ms, shade ms, rays in) per bounce of that batch

    # ---- e2e through the C-ABI with host buffers (scene upload + render + D2H inside the timed region)
    host = torch.empty((N, 4), dtype=torch.float32).pin_memory()
    ctx.set_color_tensor(None)

    def e2e_step():
        ctx.set_scene(scene)   # H2D: scene arrays -> device tables / BVH
        ctx.build_bvh()
        ctx.set_camera(cam)
        if world > 1:          # the exchange runs on torch-owned memory
            ctx.set_color_tensor(color)
        ctx.clear_color()
        ctx.render_range(begin, count, args.depth, args.flags)
        if world > 1:
            dist.all_reduce(color, op=dist.ReduceOp.SUM)
            host.copy_(color)  # D2H into pinned memory
        else:
            ctx.read_color(host.data_ptr())  # D2H into pinned memory (synchronises)

    e2e_step()
    fence()
    t0 = time.perf_counter()
    e_steps = max(1, min(args.steps, 3))
    for _ in range(e_steps):
        e2e_step()
    fence()
    e_dt = time.perf_counter() - t0
    et = torch.tensor([e_dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_value = paths_per_step * e_steps / float(et.item())

    if rank == 0:
        peak, peak_src = measured_peak()
        # Dominant launches = the bounce with the longest duration (bounce 1 of a sample batch): its k_trace and
        # k_shade launch, timed separately by CUDA events on the launching stream inside the timed steps
        # (b2pt_get_stage_profile).  Algorithmic bytes = 88 B per live segment of that bounce (SURVEY.md 8d:
        # 44 B ray record read + 44 B written per bounce), charged against BOTH launches' time.
        prof = ctx_profile
        # bounce 0 generates its rays in registers (no queue read), so the 88 B figure applies from bounce 1 on
        cand = range(1, len(prof)) if len(prof) > 1 else range(len(prof))
        top = max(cand, key=lambda k: prof[k][0] + prof[k][1]) if prof else None
        top_rays = 0
        if top is not None and prof[top][0] + prof[top][1] > 0:
            tr_ms, sh_ms, top_rays = prof[top]
            achieved = top_rays * ALGO_BYTES_PER_SEGMENT / ((tr_ms + sh_ms) * 1e-3) / 1e9
            top_desc = ("bounce %d of a %d-sample batch = k_trace<%s> launch (%.3f ms) + k_shade launch (%.3f ms), "
                        "%d rays in (CUDA events on the launching stream, launches timed alone)" % (
                            top, st.samplesPerBatch, "primary" if top == 0 else "queue", tr_ms, sh_ms, top_rays))
        else:
            achieved = segments_per_step * args.steps * ALGO_BYTES_PER_SEGMENT / (ms * 1e-3) / 1e9 / world
            top_desc = "all bounce launches of a step (aggregate)"
        step_gbs = segments_per_step * args.steps * ALGO_BYTES_PER_SEGMENT / (ms * 1e-3) / 1e9 / world
        traffic = ncu_traffic()
        line = {
            "metric": metric_name(args.size), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak" if (world > 1 and args.weak) else "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_label(W, total_spp, args.depth, world),
                       "parallelism": ("one GPU, no exchange" if world == 1 else
                                       "samples sharded across %d GPUs (%d spp each), one NCCL all-reduce of %d B" % (
                                           world, count, N * 16)),
                       "scaling_note": ("N=1 runs BASELINE.json configs[1] (1024 spp); N>1 runs ONE fixed job, the "
                                        "north_star target 1024^2 x 4096 spp, its samples partitioned over the ranks "
                                        "(strong scaling).  What limits it: every rank still pays the per-render fixed "
                                        "part (the thinly occupied deep bounces of its last batches, launch latency) on "
                                        "a shrinking share of samples, plus one 16 MiB all-reduce; per-sample work is "
                                        "unchanged and there is no other exchange."),
                       "l2": "working set of the batches in flight (ray queue + hit bins + radiance, 272 B per path, "
                             "%.1f GB per batch) exceeds the 126 MB L2" % (st.samplesPerBatch * N * 272 / 1e9),
                       "flags": args.flags, "segments_per_path": segments_per_step / paths_per_step,
                       "batches_per_step": st.batches, "samples_per_batch": st.samplesPerBatch},
            "segments_per_s": segments_per_step * args.steps / (ms * 1e-3),
            "render_ms_library_events_last_step": st.renderMs,  # cross-check of ms_per_step (same stream, own events)
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ((traffic or {}).get("dram_bytes_per_input_ray") or 0) * top_rays or None,
                         "traffic_source": (traffic or {}).get("kernel"), "peak_source": peak_src,
                         "kernel": top_desc, "algorithmic_bytes_per_segment": ALGO_BYTES_PER_SEGMENT,
                         "whole_step_achieved": step_gbs, "stage_profile_trace_ms_shade_ms_rays": prof[:8],
                         "note": "per GPU; FP32-issue bound in practice, see DESIGN.md and profiles/"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(scene.nbytes()),
                    "d2h_bytes_per_step": int(N * 16)},
            "gpu_launches": int(st.launches) * args.steps,
            "clocks": sampler.summary(),
        }
        if not args.no_image_check:
            try:
                line["image_check"] = image_check(img_sum, total_spp, W, args.depth)
            except Exception as e:  # the check must never hide the measurement
                line["image_check"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            kind, desc, cstep, build = cpu_reference_arm()
            val, dt, _ = cstep(W, 2, args.depth, cores)
            one, dt1, _ = cstep(W, 1, args.depth, 1)  # VTK-m Serial stand-in: the same code on one thread
            line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                                    "one_thread_value": one,
                                    "sample": "%dx%d, depth %d, 2 of %d spp in %.1f s on %d threads and 1 spp in %.1f s "
                                              "on one thread; built %s; %s" % (W, H, args.depth, args.spp, dt, cores,
                                                                                dt1, build[0], desc)}
        emit(line)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it
    main()
