"""bench.py contract checks: the reference arm prints one JSON line with the agreed keys, the product arm refuses to run
(loudly, no CPU fallback) when no B200 is present, and on a B200 --dump-outputs writes what the last timed step
computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--size", "64", "--depth", "8"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "path samples/s" and d["higher_is_better"] is True
    assert d["metric"] == "cornell_64_path_samples_per_s" and d["value"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--size", "64"], capture_output=True, text=True, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_refuses_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_product_arm_dumps_the_last_step(b2pt, tmp_path):
    """--dump-outputs: the radiance sum of the last timed step, bit for bit the same in two runs with the same arguments
    and the same as one render of that workload through the binding; its NaN-poisoned channels (about 15 pixels at this
    size) are stored as 0 and marked in the second file, so both files hold finite values only."""
    import numpy as np
    W, spp, depth, steps = 256, 256, 50, 2
    dumps = []
    for run in range(2):
        out = tmp_path / ("run%d" % run)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                            "--size", str(W), "--spp", str(spp), "--depth", str(depth), "--no-cpu-baseline",
                            "--no-image-check", "--dump-outputs", str(out)], capture_output=True, text=True, cwd=ROOT)
        assert r.returncode == 0, r.stderr
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
        assert sorted(os.listdir(out)) == ["radiance_sum.npy", "radiance_sum_nonfinite.npy"]
        dumps.append(np.stack([np.load(out / "radiance_sum.npy"), np.load(out / "radiance_sum_nonfinite.npy")]))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (2, W * W, 4) and np.isfinite(dumps[0]).all()
    assert np.array_equal(dumps[0].view(np.uint32), dumps[1].view(np.uint32))
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(b2pt.Camera(W, W))
        ctx.render(spp, depth, 0)
        want = ctx.read_color()
    bad = ~np.isfinite(want)
    assert bad.any()
    assert np.array_equal(dumps[0][1], bad.astype(np.float32))
    assert np.array_equal(dumps[0][0].view(np.uint32), np.where(bad, 0, want).astype(np.float32).view(np.uint32))


def test_dump_outputs_samples_large_arrays(tmp_path, monkeypatch):
    """Non-finite entries are stored as 0 and marked in <name>_nonfinite.npy; above the size limit (both files together)
    the same seeded, sorted sample of rows is kept in both files and in every run, and the files stay within the limit,
    headers included."""
    import numpy as np
    import bench

    def size(d):
        return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))

    big = np.zeros((2048 * 2048, 4), np.float32)  # 64 MiB of radiance sums + 64 MiB of mask before sampling
    bench.dump_outputs(str(tmp_path / "big"), radiance_sum=big)
    assert bench.DUMP_LIMIT_BYTES - 2 * bench.NPY_HEADER_BYTES - 32 < size(tmp_path / "big") <= bench.DUMP_LIMIT_BYTES
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1000 * 32 + 2 * bench.NPY_HEADER_BYTES)
    a = np.arange(4000 * 4, dtype=np.float32).reshape(4000, 4)
    a[::7, 1] = np.nan
    a[5, 2] = np.inf
    got = []
    for run in range(2):
        d = tmp_path / str(run)
        bench.dump_outputs(str(d), radiance_sum=a)
        got.append((np.load(d / "radiance_sum.npy"), np.load(d / "radiance_sum_nonfinite.npy")))
    (v, m), (v1, m1) = got
    assert v.shape == m.shape == (1000, 4) and np.array_equal(v, v1) and np.array_equal(m, m1)
    assert size(tmp_path / "0") <= bench.DUMP_LIMIT_BYTES
    assert np.isfinite(v).all() and m.dtype == np.float32 and m.any()
    rows = v[:, 0].astype(np.int64) // 4
    assert (np.diff(rows) > 0).all()
    assert np.array_equal(m, (~np.isfinite(a[rows])).astype(np.float32))
    assert np.array_equal(v, np.where(np.isfinite(a[rows]), a[rows], 0))


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       cwd=ROOT)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr
