"""Images of one view sweep at several sample counts (b2pt_render_views_checkpoints, k_accumulate_checkpoints).

Bar: slice k is BIT-IDENTICAL to b2pt_render_views(spp = checkpoints[k]) with the same flags, whatever the split of
the render into view batches or sample batches, on small and BVH scenes; the sums of squared samples are bit-identical
to a float32 sum of r*r in sample order over the per-sample images; and a checkpoint equals the oracle's production
stream at its sample count.
"""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
W, H, DEPTH = 64, 48, 7
N = W * H
CKPTS = (1, 2, 5, 7)
# per-view fallback: sample batches of 4 ([0,4), [4,7)); 4 ends the first batch, 5 starts the second
CKPTS_SPLIT = (1, 2, 4, 5, 7)


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


def hemisphere_views(n_phi, n_theta, fov=40.0):
    """n_phi x n_theta view points in front of the box opening, tilted up vectors and varying fields of view."""
    c = np.array([278 / 555.0] * 3, np.float32)
    out = []
    for a in range(n_phi):
        for b in range(n_theta):
            ang = 0.5 * (b - (n_theta - 1) / 2.0) / max(n_theta, 1)
            elev = 0.25 * a
            d = 1078 / 555.0 + 0.2 * a
            pos = c + d * np.array([math.sin(ang) * math.cos(elev), math.sin(elev), -math.cos(ang) * math.cos(elev)])
            up = (0.1 * b, 1, 0.05 * a)
            out.append(np.concatenate([pos, c, np.array(up), [fov + 3 * a + b]]).astype(np.float32))
    return np.stack(out)


def camera(b2pt_or_oracle, v, w, h):
    return b2pt_or_oracle.Camera(w, h, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9]))


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def same_bits_nan(a, b):
    """Bit-identical where finite or inf; NaN in the same places (a NaN's payload is not compared)."""
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


def set_regime(monkeypatch, regime, spp):
    if regime == "views2":  # 2 views per batch: 3 batches on separate streams
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(2 * N * spp + 5))
    elif regime == "one_view":
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(N * spp))
    elif regime == "split_view":  # a view no longer fits a batch: per-view fallback, sample batches of 4
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(N * 4))


@pytest.mark.parametrize("regime, batches", [(None, 1), ("views2", 3), ("one_view", 6), ("split_view", 2)])
def test_slices_bit_identical_to_render_views(gpu_ctx, b2pt, regime, batches, monkeypatch):
    views = hemisphere_views(2, 3)
    ck = CKPTS_SPLIT if regime == "split_view" else CKPTS
    set_regime(monkeypatch, regime, ck[-1])
    got = gpu_ctx.render_views_checkpoints(views, W, H, ck, DEPTH)
    st = gpu_ctx.stats()
    monkeypatch.delenv("B2PT_BATCH_PATHS", raising=False)
    assert got.shape == (len(ck), 6, N, 4) and got.dtype == np.float32
    assert st.paths == N * ck[-1] * 6
    assert st.batches == batches  # (split_view: the last view's render)
    for k, c in enumerate(ck):
        assert same_bits(got[k], gpu_ctx.render_views(views, W, H, c, DEPTH)), c
    assert got[0][:, :, :3].max() > 0 and not same_bits(got[0], got[1])


@pytest.mark.parametrize("flag", ["normalize", "pnm16"])
def test_flags(gpu_ctx, b2pt, flag):
    views = hemisphere_views(2, 3)
    f = b2pt.FLAG_VIEWS_NORMALIZE if flag == "normalize" else b2pt.FLAG_VIEWS_PNM16
    got, m2 = gpu_ctx.render_views_checkpoints(views, W, H, CKPTS, DEPTH, f, moments=True)
    if flag == "pnm16":
        assert got.shape == (4, 6, N, 3) and got.dtype == np.uint16
    for k, c in enumerate(CKPTS):
        want = gpu_ctx.render_views(views, W, H, c, DEPTH, f)
        assert np.array_equal(got[k], want) if flag == "pnm16" else same_bits(got[k], want), c
    # the sums of squares are raw float4 whatever the flags
    _, m2_raw = gpu_ctx.render_views_checkpoints(views, W, H, CKPTS, DEPTH, moments=True)
    assert same_bits(m2, m2_raw)


def test_bvh_scene(gpu_ctx, b2pt):
    views = hemisphere_views(1, 3)
    f = b2pt.FLAG_FORCE_BVH
    ck = (1, 3, 4)
    got = gpu_ctx.render_views_checkpoints(views, W, H, ck, 6, f)
    assert gpu_ctx.stats().tracePath == 1
    for k, c in enumerate(ck):
        assert same_bits(got[k], gpu_ctx.render_views(views, W, H, c, 6, f)), c


def per_sample_images(ctx, b2pt, views, spp):
    """[spp, view, pixel, 4]: sample s of every pixel alone (added to a cleared canvas, 0 + r is r)."""
    out = np.empty((spp, len(views), N, 4), np.float32)
    for v, row in enumerate(views):
        ctx.set_camera(camera(b2pt, row, W, H))
        for s in range(spp):
            ctx.clear_color()
            ctx.render_range(s, 1, DEPTH)
            out[s, v] = ctx.read_color()
    return out


@pytest.mark.parametrize("regime", [None, "split_view"])
def test_moments_bit_identical_to_sequential_squares(gpu_ctx, b2pt, regime, monkeypatch):
    views = hemisphere_views(2, 3)
    ck = CKPTS_SPLIT if regime == "split_view" else CKPTS
    set_regime(monkeypatch, regime, ck[-1])
    img, m2 = gpu_ctx.render_views_checkpoints(views, W, H, ck, DEPTH, moments=True)
    monkeypatch.delenv("B2PT_BATCH_PATHS", raising=False)
    assert m2.shape == (len(ck), 6, N, 4) and m2.dtype == np.float32
    r = per_sample_images(gpu_ctx, b2pt, views, ck[-1])
    assert not r[..., 3].any()
    s1 = np.zeros((6, N, 4), np.float32)
    s2 = np.zeros((6, N, 4), np.float32)
    k = 0
    with np.errstate(invalid="ignore", over="ignore"):
        for s in range(ck[-1]):
            s1 = s1 + r[s]
            s2 = s2 + r[s] * r[s]
            if s + 1 == ck[k]:
                assert same_bits_nan(img[k], s1), s + 1
                assert same_bits_nan(m2[k], s2), s + 1
                k += 1
    assert k == len(ck)
    assert not m2[..., 3].any() and m2[-1][:, :, :3].max() > 0


def test_checkpoint_matches_oracle(gpu_ctx, b2pt, oracle):
    w, h, depth = 40, 40, 5
    view = hemisphere_views(2, 2)[1:2]
    got = gpu_ctx.render_views_checkpoints(view, w, h, (2, 4), depth)
    sc, cam = oracle.cornell_scene(), camera(oracle, view[0], w, h)
    for k, spp in enumerate((2, 4)):
        o, _ = oracle.render(sc, cam, spp, depth, mode=oracle.MODE_FORWARD_FAST)
        g3, o3 = got[k][0][:, :3].astype(np.float64), o[:, :3].astype(np.float64)
        assert np.array_equal(np.isnan(g3), np.isnan(o3))
        ok = ~np.isnan(o3)
        rel = np.abs(g3[ok] - o3[ok]) / np.maximum(np.abs(o3[ok]), 1e-3 * spp)
        assert (rel <= 1e-4).mean() > 0.999, spp


def test_contract(b2pt):
    L, p = b2pt.lib(), b2pt._p
    views = hemisphere_views(2, 3)[:4]
    w, h, depth = 32, 24, 5
    n = w * h
    ck = (1, 3, 4)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(b2pt.Camera(48, 16))
        ctx.render(2, 3)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        full, m2 = ctx.render_views_checkpoints(views, w, h, ck, depth, moments=True)
        st = ctx.stats()
        assert st.paths == n * 4 * len(views)
        ptr = L.b2pt_views_device_ptr(ctx._h)
        assert ptr

        def fails(message, *args, **kw):
            with pytest.raises(b2pt.B2ptError, match=message) as e:
                ctx.render_views_checkpoints(*args, **kw)
            assert e.value.code == b2pt.ERR_BAD_VALUE

        fails(r"nCheckpoints must be in \[1,32\]", views, w, h, (), depth)
        fails(r"nCheckpoints must be in \[1,32\]", views, w, h, range(1, 34), depth)
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (0, 2), depth)
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (2, 2), depth)
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (3, 2), depth)
        fails("REFERENCE_STREAM cannot be combined", views, w, h, ck, depth, b2pt.FLAG_REFERENCE_STREAM)
        bad = views.copy()
        bad[2, 9] = 0.0
        fails("feild of view must be greater than zero", bad, w, h, ck, depth)
        fails("width must be greater than zero", views, 0, h, ck, depth)
        vp, two = p(views), np.array([1, 2], np.int32)
        assert L.b2pt_render_views_checkpoints(ctx._h, 4, vp, w, h, 2, None, depth, 0, None, None) == b2pt.ERR_BAD_VALUE
        assert b"nCheckpoints must be in [1,32]" in L.b2pt_last_error()
        assert L.b2pt_render_views_checkpoints(ctx._h, 4, None, w, h, 2, p(two), depth, 0, None, None) == b2pt.ERR_BAD_VALUE
        assert L.b2pt_render_views_checkpoints(ctx._h, -1, vp, w, h, 2, p(two), depth, 0, None, None) == b2pt.ERR_BAD_VALUE
        # device output above 2^30 float4: four 8192^2 views (2^28 pixels) in 8 slices, (K-1) + K + 1 with sums of
        # squares, (K-1) + 1 without
        tiny = np.zeros(4, np.float32)
        four, eight = np.arange(1, 5, dtype=np.int32), np.arange(1, 9, dtype=np.int32)
        for K, c, m in ((4, four, p(tiny)), (8, eight, None)):
            assert L.b2pt_render_views_checkpoints(ctx._h, 4, vp, 8192, 8192, K, p(c), depth, 0, None,
                                                   m) == b2pt.ERR_BAD_VALUE
            assert b"more than 2^30 float4" in L.b2pt_last_error()
        # nothing was rendered: same statistics, same device image
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches) == (st.paths, st.launches, st.batches)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        # NULL outputs: any subset
        assert L.b2pt_render_views_checkpoints(ctx._h, 4, vp, w, h, 3, p(np.array(ck, np.int32)), depth, 0, None,
                                               None) == 0
        only_m2 = np.zeros_like(m2)
        assert L.b2pt_render_views_checkpoints(ctx._h, 4, vp, w, h, 3, p(np.array(ck, np.int32)), depth, 0, None,
                                               p(only_m2)) == 0
        assert same_bits(only_m2, m2)
        only_rgba = np.zeros_like(full)
        assert L.b2pt_render_views_checkpoints(ctx._h, 4, vp, w, h, 3, p(np.array(ck, np.int32)), depth, 0,
                                               p(only_rgba), None) == 0
        assert same_bits(only_rgba, full)
        assert ctx.stats().paths == n * 4 * len(views)
        # nViews == 0
        empty = ctx.render_views_checkpoints(np.zeros((0, 10), np.float32), w, h, ck, depth)
        assert empty.shape == (3, 0, n, 4)
        # the context's own camera and canvas are untouched
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])
        # the library-owned image holds the last checkpoint, as render_views(4) leaves it
        ctx.render_views_checkpoints(views, w, h, ck, depth)
        ptr = L.b2pt_views_device_ptr(ctx._h)
        ctx.set_camera(b2pt.Camera(w, h))
        for v in range(len(views)):
            assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * n * 16)) == 0
            assert same_bits(ctx.read_color(), full[-1][v]), v
        assert L.b2pt_set_color_buffer(ctx._h, None) == 0


def read_bytes(path):
    with open(path, "rb") as f:
        return f.read()


@pytest.mark.parametrize("sweep", [["-hemisphere", "-phicount", "2", "-thetacount", "3"],
                                   ["-fibonacci", "-viewcount", "12"]])
def test_driver_checkpoints(host_build, tmp_path, sweep):
    exe = os.path.join(host_build, "CornellBox_b2pt")

    def run(name, *extra):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe, "-x", "24", "-y", "16", "-raydepth", "5"] + sweep + list(extra), cwd=d,
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        assert "views rendered       = 6" in out.stdout
        return d, sorted(os.listdir(d))

    ck_dir, ck_files = run("ck", "-samplecount", "6", "-checkpoints", "2,4")
    plain_dir, plain = run("plain", "-samplecount", "6")
    assert len(plain) == 6 and all(f.startswith("output-") for f in plain)
    tails = [f[len("output-"):] for f in plain]
    assert ck_files == sorted(plain + ["output-s%d-%s" % (c, t) for c in (2, 4) for t in tails])
    for f in plain:  # the ordinary files: byte-identical to a run without -checkpoints
        assert read_bytes(ck_dir / f) == read_bytes(plain_dir / f), f
    for c in (2, 4):  # each -s<c>- file: byte-identical to the sweep at -samplecount c
        c_dir, _ = run("s%d" % c, "-samplecount", str(c))
        for t in tails:
            assert read_bytes(ck_dir / ("output-s%d-%s" % (c, t))) == read_bytes(c_dir / ("output-" + t)), (c, t)
    assert read_bytes(ck_dir / ("output-s2-" + tails[0])) != read_bytes(ck_dir / plain[0])
