"""Adaptive sampling of a view sweep (b2pt_render_views_adaptive).

Bar: every pixel's sums are the bits of b2pt_render_views at the pixel's own count and its sums of squares the slice
of b2pt_render_views_checkpoints(rounds) at that count; the counts and the per-round active totals are the numpy
selection rule (tests/adaptive_ref.py) replayed on that checkpointed render -- under default batching, sample batches
inside a listed round, the three BVH trace paths, without primary masks and on a canvas that is not whole tiles; the
per-pixel-count NORMALIZE and PNM16 conversions match render_views; the threshold edges, the radius, determinism, the
error contract and the driver's files."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import adaptive_ref as R  # noqa: E402
from test_gpu_denoise import tilted_views  # noqa: E402
from test_gpu_features import driver_view_names, generated_scene, hemisphere_positions, read_pfm, view_row  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
W, H, DEPTH = 64, 48, 7
ROUNDS = (2, 4, 8, 16, 32)
EPS = 0.01


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


@pytest.fixture(scope="module")
def ctx(b2pt):
    c = b2pt.Context(0)
    c.set_scene(b2pt.Scene.cornell())
    yield c
    c.close()


def params(b2pt, tau, eps=EPS, radius=1):
    p = b2pt.AdaptiveParams()
    p.threshold, p.epsilon, p.radius = tau, eps, radius
    return p


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def pick_tau(S, Q, rounds):
    """A threshold that stops some pixels in every round: the median relative error after rounds[2] samples of the
    pixels whose variance is not zero (misses and the light have none, and stop after round 0 at any threshold)."""
    c = rounds[2]
    m = np.nan_to_num(S[2, ..., :3].astype(np.float64)) / c
    v = np.maximum(0, np.nan_to_num(Q[2, ..., :3].astype(np.float64)) / c - m * m) / (c - 1)
    w = np.array([0.2126, 0.7152, 0.0722])
    rel = np.sqrt(v @ w) / (m @ w + EPS)
    return float(np.median(rel[rel > 0]))


def check(ctx, b2pt, views, w, h, rounds, p, flags=0):
    """One adaptive render against the checkpointed render, the replay and render_views at every count."""
    S, Q = ctx.render_views_checkpoints(views, w, h, rounds, DEPTH, flags, moments=True)
    img, m2, counts, active = ctx.render_views_adaptive(views, w, h, rounds, DEPTH, p, flags)
    want_counts, want_active = R.replay(S, Q, rounds, w, h, p.threshold, p.epsilon, p.radius)
    assert np.array_equal(counts, want_counts)
    assert np.array_equal(active, want_active)
    assert ctx.stats().paths == int(sum(active[k] * (rounds[k] - (rounds[k - 1] if k else 0))
                                        for k in range(len(rounds))))
    for k, c in enumerate(rounds):
        at = counts == c
        if not at.any():
            continue
        uni = ctx.render_views(views, w, h, c, DEPTH, flags)
        assert same_bits(img[at], uni[at]), c
        assert same_bits(m2[at], Q[k][at]), c
    return counts, active


@pytest.fixture(scope="module")
def cornell_tau(ctx, b2pt):
    views = tilted_views(6)
    S, Q = ctx.render_views_checkpoints(views, W, H, ROUNDS, DEPTH, 0, moments=True)
    return pick_tau(S, Q, ROUNDS)


@pytest.mark.parametrize("regime", ["default", "sample_batches", "no_masks", "odd_canvas"])
def test_cornell_matches_uniform_renders_and_replay(ctx, b2pt, cornell_tau, regime, monkeypatch):
    views = tilted_views(6)
    w, h = (37, 23) if regime == "odd_canvas" else (W, H)
    flags = b2pt.FLAG_NO_PRIMARY_MASKS if regime == "no_masks" else 0
    if regime == "sample_batches":  # round 0 one view at a time, every listed round in several sample batches
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(w * h * 3))
    counts, active = check(ctx, b2pt, views, w, h, ROUNDS, params(b2pt, cornell_tau), flags)
    assert all(active[k] > active[k + 1] > 0 for k in range(len(ROUNDS) - 1)), active  # every round has work
    if regime == "sample_batches":
        assert ctx.stats().batches > 1


@pytest.mark.parametrize("flags", ["FORCE_BVH", "FORCE_BVH|GPU_LBVH", "FORCE_BVH|WIDE_BVH"])
def test_bvh_scene(b2pt, flags):
    f = 0
    for name in flags.split("|"):
        f |= getattr(b2pt, "FLAG_" + name)
    g = 3.0
    views = np.stack([view_row([g, g, -6.0], [g, g, g], (0, 1, 0), 60.0),
                      view_row([-4.0, 8.0, -3.5], [g, g, g], (0.2, 1.0, 0.0), 55.0)])
    with b2pt.Context(0) as c:
        c.set_scene(generated_scene(b2pt))
        S, Q = c.render_views_checkpoints(views, 40, 30, ROUNDS, DEPTH, f, moments=True)
        tau = pick_tau(S, Q, ROUNDS)
        counts, active = check(c, b2pt, views, 40, 30, ROUNDS, params(b2pt, tau), f)
        assert c.stats().tracePath == 1
    assert active[-1] > 0 and active[1] < active[0]


@pytest.mark.parametrize("flag", ["FLAG_VIEWS_NORMALIZE", "FLAG_VIEWS_PNM16"])
def test_per_pixel_count_conversions(ctx, b2pt, cornell_tau, flag):
    views = tilted_views(6)
    f = getattr(b2pt, flag)
    p = params(b2pt, cornell_tau)
    img, m2, counts, _ = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p, f)
    raw, m2_raw, counts_raw, _ = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p, 0)
    assert np.array_equal(counts, counts_raw) and same_bits(m2, m2_raw)  # Q is raw whatever the flags
    for c in ROUNDS:
        at = counts == c
        if at.any():
            assert np.array_equal(img[at], ctx.render_views(views, W, H, c, DEPTH, f)[at]), c


def test_threshold_edges_and_radius(ctx, b2pt, cornell_tau):
    views = tilted_views(6)
    img, _, counts, active = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, params(b2pt, 0.0))
    assert (counts == ROUNDS[-1]).all() and (active == counts.size).all()
    assert same_bits(img, ctx.render_views(views, W, H, ROUNDS[-1], DEPTH))
    _, _, counts, active = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, params(b2pt, float("inf")))
    assert (counts == ROUNDS[0]).all() and list(active) == [counts.size] + [0] * (len(ROUNDS) - 1)
    c0, a0 = check(ctx, b2pt, views, W, H, ROUNDS, params(b2pt, cornell_tau, radius=0))
    c2, a2 = check(ctx, b2pt, views, W, H, ROUNDS, params(b2pt, cornell_tau, radius=2))
    assert (c2 >= c0).all() and (c2 > c0).any() and a2[1] > a0[1]


def test_determinism_and_single_round(ctx, b2pt, cornell_tau):
    views = tilted_views(6)
    p = params(b2pt, cornell_tau)
    a = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p)
    b = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    img, m2, counts, active = ctx.render_views_adaptive(views, W, H, (3,), DEPTH, p)
    assert (counts == 3).all() and list(active) == [counts.size]
    assert same_bits(img, ctx.render_views(views, W, H, 3, DEPTH))


def test_contract(b2pt):
    L = b2pt.lib()
    views = tilted_views(2)
    w, h = 32, 16
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        cam = b2pt.Camera(24, 8)
        c.set_camera(cam)
        c.render(2, 3)
        canvas = c.read_color()
        c.render_views(views, w, h, 4, 3)
        dev = c.render_views(views, w, h, 4, 3)
        st = c.stats()
        ptr = L.b2pt_views_device_ptr(c._h)

        def call(v, nv, ww, hh, rounds, p, flags, depth=3):
            r = np.ascontiguousarray(rounds, np.int32)
            return L.b2pt_render_views_adaptive(c._h, nv, None if v is None else v.ctypes.data_as(ctypes.c_void_p),
                                                ww, hh, r.size, r.ctypes.data_as(ctypes.c_void_p), depth,
                                                None if p is None else ctypes.byref(p), flags, None, None, None, None)

        def fails(msg, *args, **kw):
            assert call(*args, **kw) == b2pt.ERR_BAD_VALUE
            assert msg in L.b2pt_last_error().decode(), L.b2pt_last_error()

        ok = params(b2pt, 0.05)
        fn = "b2pt_render_views_adaptive: "
        fails(fn + "bad view list", None, 2, w, h, (2, 4), ok, 0)
        fails(fn + "bad view list", views, -1, w, h, (2, 4), ok, 0)
        fails(fn + "nCheckpoints must be in [1,32]", views, 2, w, h, (), ok, 0)
        fails(fn + "nCheckpoints must be in [1,32]", views, 2, w, h, tuple(range(2, 35)), ok, 0)
        fails(fn + "checkpoints must be >= 1 and strictly increasing", views, 2, w, h, (2, 2), ok, 0)
        fails(fn + "rounds[0] must be >= 2", views, 2, w, h, (1, 4), ok, 0)
        fails("maxDepth must be in [1,4096]", views, 2, w, h, (2, 4), ok, 0, depth=0)
        for f in (b2pt.FLAG_REFERENCE_STREAM, b2pt.FLAG_ONE_KERNEL_BOUNCE):
            fails(fn + "REFERENCE_STREAM and ONE_KERNEL_BOUNCE cannot be combined with it", views, 2, w, h, (2, 4), ok, f)
        fails(fn + "threshold must be >= 0", views, 2, w, h, (2, 4), params(b2pt, -0.1), 0)
        fails(fn + "threshold must be >= 0", views, 2, w, h, (2, 4), params(b2pt, float("nan")), 0)
        fails(fn + "epsilon must be > 0", views, 2, w, h, (2, 4), params(b2pt, 0.1, eps=0.0), 0)
        fails(fn + "epsilon must be > 0", views, 2, w, h, (2, 4), params(b2pt, 0.1, eps=float("nan")), 0)
        fails(fn + "radius must be in [0,4]", views, 2, w, h, (2, 4), params(b2pt, 0.1, radius=5), 0)
        fails(fn + "radius must be in [0,4]", views, 2, w, h, (2, 4), params(b2pt, 0.1, radius=-1), 0)
        fails("Camera width must be greater than zero.", views, 2, 0, h, (2, 4), ok, 0)
        big = np.repeat(views[:1], 17, 0)  # 17 views of 8192 x 4096 = 2^25 pixels: 2 float4 each exceed 2^30
        fails(fn + "more than 2^30 float4 of device state", big, 17, 8192, 4096, (2, 4), ok, 0)
        # nothing ran: the statistics, the view image, the canvas and the camera are the ones from before
        assert bytes(c.stats()) == bytes(st)
        assert L.b2pt_views_device_ptr(c._h) == ptr
        assert np.array_equal(c.render_views(views, w, h, 4, 3), dev)
        assert np.array_equal(c.read_color(), canvas)
        assert call(views, 0, w, h, (2, 4), ok, 0) == 0  # nViews == 0 does nothing
        # a successful call leaves the canvas alone too, and the view image is then its own
        c.render_views_adaptive(views, w, h, (2, 4), 3, ok)
        assert np.array_equal(c.read_color(), canvas)
        assert L.b2pt_views_device_ptr(c._h)
        c.render(2, 3)  # the context's own camera still renders its own canvas
        assert same_bits(c.read_color(), canvas)


def test_driver_matches_binding(b2pt, host_build, tmp_path):
    exe = os.path.join(host_build, "CornellBox_b2pt")
    w, h, tau = 24, 16, 0.15
    out = subprocess.run([exe, "-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", "16", "-hemisphere",
                          "-phicount", "2", "-thetacount", "3", "-checkpoints", "2,4,8", "-adaptive", str(tau)],
                         cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    order = driver_view_names("hemisphere", hemisphere_positions(2, 3))
    assert sorted(os.listdir(tmp_path)) == sorted(["output-adaptive-%s.pnm" % t for t in order] +
                                                  ["output-spp-%s.pfm" % t for t in order])
    views = np.stack([view_row(pos) for pos in hemisphere_positions(2, 3)])
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        pnm, _, counts, _ = c.render_views_adaptive(views, w, h, (2, 4, 8, 16), 5, params(b2pt, tau),
                                                    b2pt.FLAG_VIEWS_PNM16)
    assert len(np.unique(counts)) > 1
    for v, tail in enumerate(order):
        body = "".join("%d %d %d\n" % tuple(px) for px in pnm[v])
        assert open(tmp_path / ("output-adaptive-%s.pnm" % tail)).read() == "P3\n%d %d 255\n" % (w, h) + body
        assert np.array_equal(read_pfm(tmp_path / ("output-spp-%s.pfm" % tail), w, h, 1), counts[v].astype(np.float32))
