"""An adaptive view sweep denoised on the GPU (b2pt_render_views_adaptive_denoised).

Bar: the image and counts are b2pt_render_views_adaptive's bits under every view flag, with the same statistics; the
guides at every pixel are b2pt_render_views_features' slice at the pixel's own count, on the small scene and the three
BVH trace paths; with levels = 0 the output is the float32 prep at each pixel's own count bit for bit, and its PNM
integers are the adaptive image's; at tau = 0 and tau = +inf (one count everywhere) it is b2pt_denoise_views of the
uniform sweep bit for bit; at a general tau one level, the default levels and ten levels agree with the float64
restatement, on the sweep's canvas, a 1 x 37 and a 13 x 5 one; the result does not depend on the chunking and two
calls agree; it lowers the error of the adaptive image; bad inputs fail before anything runs; the driver's
-adaptive-denoise files are the binding's."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_ref as R  # noqa: E402
from test_gpu_adaptive import generated_scene, pick_tau, tilted_views  # noqa: E402
from test_gpu_denoise import rel_err, rel_mse  # noqa: E402
from test_gpu_features import driver_view_names, hemisphere_positions, read_pfm, view_row  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
W, H, DEPTH = 64, 48, 7
ROUNDS = (2, 4, 8, 16, 32)
EPS = 0.01
INF = float("inf")


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


def aparams(b2pt, tau, eps=EPS, radius=1):
    p = b2pt.AdaptiveParams()
    p.threshold, p.epsilon, p.radius = tau, eps, radius
    return p


def dparams(b2pt, levels=None):
    p = b2pt.DenoiseParams.defaults()
    if levels is not None:
        p.levels = levels
    return p


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def stat_tuple(st):
    return st.paths, st.segments, st.nanSamples, st.launches, st.batches


def per_pixel_prep(S, Q, A, ND, counts):
    """denoise_ref.prep with every pixel's own count: each pixel is a one-pixel slice of its own checkpoint."""
    nv, n = counts.shape
    one = lambda a: np.ascontiguousarray(a, np.float32).reshape(nv * n, 1, 1, 4)
    m, V0, ga, gn, z = R.prep(one(S), one(Q), one(A), one(ND), counts.reshape(-1))
    return m.reshape(nv, n, 3), V0.reshape(nv, n), ga.reshape(nv, n, 4), gn.reshape(nv, n, 3), z.reshape(nv, n)


@pytest.fixture(scope="module")
def cornell_tau(ctx, b2pt):
    S, Q = ctx.render_views_checkpoints(tilted_views(6), W, H, ROUNDS, DEPTH, 0, moments=True)
    return pick_tau(S, Q, ROUNDS)


@pytest.mark.parametrize("flag", ["0", "FLAG_VIEWS_NORMALIZE", "FLAG_VIEWS_PNM16"])
def test_adaptive_outputs_are_render_views_adaptive(ctx, b2pt, cornell_tau, flag):
    views = tilted_views(6)
    f = 0 if flag == "0" else getattr(b2pt, flag)
    p = aparams(b2pt, cornell_tau)
    img, _, counts, active = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p, f)
    st = stat_tuple(ctx.stats())
    assert all(active[k] > active[k + 1] > 0 for k in range(len(ROUNDS) - 1)), active  # every round has work
    img2, counts2, den = ctx.render_views_adaptive_denoised(views, W, H, ROUNDS, DEPTH, p, None, f)
    assert np.array_equal(img2.view(np.uint8), img.view(np.uint8))
    assert np.array_equal(counts2, counts)
    assert stat_tuple(ctx.stats()) == st
    assert b2pt.lib().b2pt_views_device_ptr(ctx._h)
    assert den.dtype == img.dtype and den.shape == img.shape


@pytest.mark.parametrize("scene", ["cornell", "FORCE_BVH", "FORCE_BVH|GPU_LBVH", "FORCE_BVH|WIDE_BVH"])
def test_guides_are_features_at_each_pixels_count(b2pt, scene):
    f = 0
    if scene == "cornell":
        views, w, h = tilted_views(6), W, H
    else:
        for name in scene.split("|"):
            f |= getattr(b2pt, "FLAG_" + name)
        g = 3.0
        views = np.stack([view_row([g, g, -6.0], [g, g, g], (0, 1, 0), 60.0),
                          view_row([-4.0, 8.0, -3.5], [g, g, g], (0.2, 1.0, 0.0), 55.0)])
        w, h = 40, 30
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell() if scene == "cornell" else generated_scene(b2pt))
        S, Q = c.render_views_checkpoints(views, w, h, ROUNDS, DEPTH, f, moments=True)
        p = aparams(b2pt, pick_tau(S, Q, ROUNDS))
        _, counts, _, alb, nd = c.render_views_adaptive_denoised(views, w, h, ROUNDS, DEPTH, p, None, f,
                                                                 features=True)
        if f:
            assert c.stats().tracePath == 1
        A, ND = c.render_views_features(views, w, h, ROUNDS, f)
    assert len(np.unique(counts)) > 2
    for k, n in enumerate(ROUNDS):
        at = counts == n
        assert same_bits(alb[at], A[k][at]), n
        assert same_bits(nd[at], ND[k][at]), n


def test_levels_zero_is_the_per_pixel_mean(ctx, b2pt, cornell_tau):
    views = tilted_views(6)
    p = aparams(b2pt, cornell_tau)
    S, Q, counts, _ = ctx.render_views_adaptive(views, W, H, ROUNDS, DEPTH, p)
    _, counts2, den, A, ND = ctx.render_views_adaptive_denoised(views, W, H, ROUNDS, DEPTH, p, dparams(b2pt, 0),
                                                                features=True)
    assert np.array_equal(counts2, counts)
    m, V0, *_ = per_pixel_prep(S, Q, A, ND, counts)
    assert same_bits(den[..., :3], m)
    assert same_bits(den[..., 3], V0)
    assert (V0 > 0).any()
    pnm, _, pnm_den = ctx.render_views_adaptive_denoised(views, W, H, ROUNDS, DEPTH, p, dparams(b2pt, 0),
                                                         b2pt.FLAG_VIEWS_PNM16)
    assert np.array_equal(pnm_den, pnm)


@pytest.mark.parametrize("tau, k", [(0.0, -1), (INF, 0)])
def test_one_count_everywhere_is_the_uniform_filter(ctx, b2pt, tau, k):
    views = tilted_views(6)
    c = ROUNDS[k]
    for flags in (0, b2pt.FLAG_VIEWS_PNM16):
        _, counts, den = ctx.render_views_adaptive_denoised(views, W, H, ROUNDS, DEPTH, aparams(b2pt, tau), None,
                                                            flags)
        assert (counts == c).all()
        S, Q = ctx.render_views_checkpoints(views, W, H, (c,), DEPTH, 0, moments=True)
        A, ND = ctx.render_views_features(views, W, H, (c,))
        want = ctx.denoise_views(S, Q, A, ND, W, H, (c,), flags=flags)
        assert np.array_equal(den.view(np.uint8), want[0].view(np.uint8)), flags


# the tolerances of test_gpu_denoise: one level, then the default five and all ten; on the sweep's canvas, one column
# and a canvas narrower and shorter than k_atrous' 16 x 16 tile
@pytest.mark.parametrize("levels, tol", [(1, 1e-4), (5, 1e-3), (10, 1e-3)])
def test_general_tau_against_restatement(ctx, b2pt, cornell_tau, levels, tol):
    views = tilted_views(6)
    p = aparams(b2pt, cornell_tau)
    for w, h in ((W, H), (1, 37), (13, 5)):
        S, Q, counts, _ = ctx.render_views_adaptive(views, w, h, ROUNDS, DEPTH, p)
        _, _, den, A, ND = ctx.render_views_adaptive_denoised(views, w, h, ROUNDS, DEPTH, p, dparams(b2pt, levels),
                                                              features=True)
        nv = views.shape[0]
        img = lambda a: a.astype(np.float64).reshape((nv, h, w) + a.shape[2:])
        x, V, ga, gn, z = (img(a) for a in per_pixel_prep(S, Q, A, ND, counts))
        d = R.DEFAULTS
        for lev in range(levels):
            x, V = R.atrous_level(x, V, ga, gn, z, h, w, 1 << lev, True, d["sigma_lum"], d["sigma_albedo"],
                                  d["sigma_normal"], d["sigma_depth"])
        e = rel_err(den[None, ..., :3], x.reshape(1, nv, h * w, 3))
        assert e < tol, (w, h, levels, e)


def test_chunking_and_determinism(ctx, b2pt, cornell_tau):
    # 32 x 16 views: 2^23 / 512 = 16384 views per chunk; 5 more cross into a second chunk
    w, h = 32, 16
    per = (1 << 23) // (w * h)
    V = per + 5
    views = tilted_views(6)[np.arange(V) % 6].copy()
    views[:, 9] += (np.arange(V) % 97).astype(np.float32) * 0.05  # every view its own field of view
    p = aparams(b2pt, cornell_tau)
    a = ctx.render_views_adaptive_denoised(views, w, h, ROUNDS, DEPTH, p, features=True)
    b = ctx.render_views_adaptive_denoised(views, w, h, ROUNDS, DEPTH, p, features=True)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert len(np.unique(a[1])) > 2
    for v in (0, per - 1, per, V - 1):
        one = ctx.render_views_adaptive_denoised(views[v:v + 1], w, h, ROUNDS, DEPTH, p, features=True)
        for x, y in zip(one, a):
            assert np.array_equal(x[0].view(np.uint8), y[v].view(np.uint8)), v


# DESIGN.md 8e measured denoised / noisy rel-MSE 0.22-0.28 for uniform sweeps
RATIO_BOUND = 0.5


def test_it_denoises(b2pt):
    views = tilted_views(8)
    w = h = 128
    rounds = (4, 8, 16, 32)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        img, counts, den = c.render_views_adaptive_denoised(views, w, h, rounds, 5)
        target = c.render_views(views, w, h, 1024, 5)[..., :3] / np.float32(1024)
    target = np.nan_to_num(target.astype(np.float64))
    noisy = np.nan_to_num(img[..., :3].astype(np.float64)) / counts[..., None]
    rn, rd = rel_mse(noisy, target), rel_mse(den[..., :3], target)
    assert len(np.unique(counts)) > 1
    assert rd / rn <= RATIO_BOUND, (rn, rd)


def test_contract(b2pt):
    L = b2pt.lib()
    views = tilted_views(2)
    w, h = 32, 16
    n = 2 * w * h
    with b2pt.Context(0) as c:
        r = np.array([2, 4], np.int32)
        vp = views.ctypes.data_as(ctypes.c_void_p)
        assert L.b2pt_render_views_adaptive_denoised(c._h, 2, vp, w, h, 2, r.ctypes.data_as(ctypes.c_void_p), 3,
                                                     None, None, 0, None, None, None, None, None) == b2pt.ERR_STATE
        c.set_scene(b2pt.Scene.cornell())
        cam = b2pt.Camera(24, 8)
        c.set_camera(cam)
        c.render(2, 3)
        canvas = c.read_color()
        dev = c.render_views(views, w, h, 4, 3)
        st = c.stats()
        ptr = L.b2pt_views_device_ptr(c._h)
        outs = [np.zeros((n, 4), np.float32), np.zeros(n, np.int32), np.zeros((n, 4), np.float32),
                np.zeros((n, 4), np.float32), np.zeros((n, 4), np.float32)]

        def call(v, nv, ww, hh, rounds, ap, dp, flags, depth=3):
            rr = np.ascontiguousarray(rounds, np.int32)
            return L.b2pt_render_views_adaptive_denoised(
                c._h, nv, None if v is None else v.ctypes.data_as(ctypes.c_void_p), ww, hh, rr.size,
                rr.ctypes.data_as(ctypes.c_void_p), depth, None if ap is None else ctypes.byref(ap),
                None if dp is None else ctypes.byref(dp), flags, *(o.ctypes.data_as(ctypes.c_void_p) for o in outs))

        def fails(msg, *args, **kw):
            assert call(*args, **kw) == b2pt.ERR_BAD_VALUE
            assert msg in L.b2pt_last_error().decode(), L.b2pt_last_error()

        ok = aparams(b2pt, 0.05)
        fn = "b2pt_render_views_adaptive_denoised: "
        fails(fn + "bad view list", None, 2, w, h, (2, 4), ok, None, 0)
        fails(fn + "bad view list", views, -1, w, h, (2, 4), ok, None, 0)
        fails(fn + "nCheckpoints must be in [1,32]", views, 2, w, h, (), ok, None, 0)
        fails(fn + "checkpoints must be >= 1 and strictly increasing", views, 2, w, h, (2, 2), ok, None, 0)
        fails(fn + "rounds[0] must be >= 2", views, 2, w, h, (1, 4), ok, None, 0)
        fails("maxDepth must be in [1,4096]", views, 2, w, h, (2, 4), ok, None, 0, depth=0)
        for f in (b2pt.FLAG_REFERENCE_STREAM, b2pt.FLAG_ONE_KERNEL_BOUNCE):
            fails(fn + "REFERENCE_STREAM and ONE_KERNEL_BOUNCE cannot be combined with it", views, 2, w, h, (2, 4), ok,
                  None, f)
        fails(fn + "threshold must be >= 0", views, 2, w, h, (2, 4), aparams(b2pt, float("nan")), None, 0)
        fails(fn + "epsilon must be > 0", views, 2, w, h, (2, 4), aparams(b2pt, 0.1, eps=0.0), None, 0)
        fails(fn + "radius must be in [0,4]", views, 2, w, h, (2, 4), aparams(b2pt, 0.1, radius=5), None, 0)
        fails("Camera width must be greater than zero.", views, 2, 0, h, (2, 4), ok, None, 0)
        big = np.repeat(views[:1], 17, 0)
        fails(fn + "more than 2^30 float4 of device state", big, 17, 8192, 4096, (2, 4), ok, None, 0)
        for lv in (-1, 11):
            fails(fn + "levels must be in [0,10]", views, 2, w, h, (2, 4), ok, dparams(b2pt, lv), 0)
        for name in ("sigmaLum", "sigmaAlbedo", "sigmaNormal", "sigmaDepth"):
            for bad in (0.0, -1.0, float("nan")):
                dp = dparams(b2pt)
                setattr(dp, name, bad)
                fails(fn + name + " must be > 0 (or +inf)", views, 2, w, h, (2, 4), ok, dp, 0)
        fails(fn + "more than 2^24 samples", views, 2, w, h, (2, (1 << 24) + 1), ok, None, 0)
        # nothing ran: the outputs, the statistics, the view image, the canvas and the camera are the ones from before
        assert all((o == 0).all() for o in outs)
        assert bytes(c.stats()) == bytes(st)
        assert L.b2pt_views_device_ptr(c._h) == ptr
        assert np.array_equal(c.render_views(views, w, h, 4, 3), dev)
        assert np.array_equal(c.read_color(), canvas)
        assert call(views, 0, w, h, (2, 4), ok, None, 0) == 0  # nViews == 0 does nothing
        assert all((o == 0).all() for o in outs)
        # NULL parameters are the defaults; a successful call leaves the canvas and camera alone
        assert call(views, 2, w, h, (2, 4), None, None, 0) == 0
        want = c.render_views_adaptive_denoised(views, w, h, (2, 4), 3, b2pt.AdaptiveParams.defaults(),
                                                b2pt.DenoiseParams.defaults(), features=True)
        got = (outs[0], outs[1], outs[4], outs[2], outs[3])
        for x, y in zip(got, want):
            assert np.array_equal(x.reshape(-1).view(np.uint8), y.reshape(-1).view(np.uint8))
        assert np.array_equal(c.read_color(), canvas)
        c.render(2, 3)  # the context's own camera still renders its own canvas
        assert same_bits(c.read_color(), canvas)


def test_driver_matches_binding(b2pt, host_build, tmp_path):
    exe = os.path.join(host_build, "CornellBox_b2pt")
    w, h, tau = 24, 16, 0.15
    args = ["-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", "16", "-hemisphere", "-phicount", "2",
            "-thetacount", "3", "-checkpoints", "2,4,8"]

    def run(name, *extra):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe] + args + list(extra), cwd=d, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        return d, sorted(os.listdir(d))

    ddir, files = run("denoised", "-adaptive-denoise", str(tau))
    adir, plain = run("adaptive", "-adaptive", str(tau))
    order = driver_view_names("hemisphere", hemisphere_positions(2, 3))
    assert len(plain) == 2 * len(order)
    for f in plain:  # the -adaptive files, byte-identical
        assert open(ddir / f, "rb").read() == open(adir / f, "rb").read(), f
    assert files == sorted(plain + ["output-adaptive-denoised-%s.pnm" % t for t in order])
    views = np.stack([view_row(pos) for pos in hemisphere_positions(2, 3)])
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        pnm, counts, den = c.render_views_adaptive_denoised(views, w, h, (2, 4, 8, 16), 5, aparams(b2pt, tau), None,
                                                            b2pt.FLAG_VIEWS_PNM16)
    assert len(np.unique(counts)) > 1
    for v, tail in enumerate(order):
        for stem, img in (("output-adaptive", pnm), ("output-adaptive-denoised", den)):
            body = "".join("%d %d %d\n" % tuple(px) for px in img[v])
            assert open(ddir / ("%s-%s.pnm" % (stem, tail))).read() == "P3\n%d %d 255\n" % (w, h) + body, stem
        assert np.array_equal(read_pfm(ddir / ("output-spp-%s.pfm" % tail), w, h, 1), counts[v].astype(np.float32))
