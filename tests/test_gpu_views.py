"""GPU tests of the view-batched render (b2pt_render_views): the camera loop of generateHemisphere /
fibonacciHemisphere (main.cc:431-561) done as one flat (view, sample, pixel) index space.

Bar: every view's radiance sum is BIT-IDENTICAL to b2pt_set_camera(view) + b2pt_render of the same view (same
per-(pixel, sample) streams, same per-path arithmetic, same sample-order accumulation), whatever the split of the view
list into batches; and -- through the single-view parity tests -- equal to the oracle.
"""
import ctypes
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def hemisphere_views(n_phi, n_theta, fov=40.0):
    """n_phi x n_theta view points in front of the box opening (variations of the main.cc:616-622 camera, every one
    sees the lit interior), tilted up vectors and varying fields of view included."""
    c = np.array([278 / 555.0] * 3, np.float32)
    out = []
    for a in range(n_phi):
        for b in range(n_theta):
            ang = 0.5 * (b - (n_theta - 1) / 2.0) / max(n_theta, 1)  # swing left/right about the y axis
            elev = 0.25 * a
            d = 1078 / 555.0 + 0.2 * a
            pos = c + d * np.array([math.sin(ang) * math.cos(elev), math.sin(elev), -math.cos(ang) * math.cos(elev)])
            up = (0.1 * b, 1, 0.05 * a)
            out.append(np.concatenate([pos, c, np.array(up), [fov + 3 * a + b]]).astype(np.float32))
    return np.stack(out)


def single_renders(ctx, b2pt, views, W, H, spp, depth, flags=0):
    imgs = []
    for v in views:
        ctx.set_camera(b2pt.Camera(W, H, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9])))
        ctx.render(spp, depth, flags)
        imgs.append(ctx.read_color().copy())
    return np.stack(imgs)


def same_bits(a, b):
    return np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("batch_paths", [None, "views2", "one_view", "split_view"])
def test_views_bit_identical_to_single_renders(gpu_ctx, b2pt, batch_paths, monkeypatch):
    W, H, spp, depth = 64, 48, 6, 7
    views = hemisphere_views(2, 3)
    N = W * H
    if batch_paths == "views2":  # 2 views per batch -> 3 batches in flight on separate streams, tail mode
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(2 * N * spp + 5))
    elif batch_paths == "one_view":
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(N * spp))
    elif batch_paths == "split_view":  # a view no longer fits a batch: per-view fallback
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(N * 4))
    got = gpu_ctx.render_views(views, W, H, spp, depth)
    monkeypatch.delenv("B2PT_BATCH_PATHS", raising=False)
    ref = single_renders(gpu_ctx, b2pt, views, W, H, spp, depth)
    assert got.shape == ref.shape == (6, N, 4)
    assert same_bits(got, ref)
    # the views differ from each other (the camera array is really indexed)
    assert got[:, :, :3].max() > 0
    assert not same_bits(got[0], got[1]) and not same_bits(got[1], got[4])


def test_views_match_oracle(gpu_ctx, b2pt, oracle):
    """Directly against the CPU oracle's production stream for two tilted views."""
    W, H, spp, depth = 40, 40, 4, 5
    views = hemisphere_views(2, 2)[1:3]
    got = gpu_ctx.render_views(views, W, H, spp, depth)
    sc = oracle.cornell_scene()
    for k, v in enumerate(views):
        cam = oracle.Camera(W, H, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9]))
        o, _ = oracle.render(sc, cam, spp, depth, mode=oracle.MODE_FORWARD_FAST)
        g3, o3 = got[k][:, :3].astype(np.float64), o[:, :3].astype(np.float64)
        assert np.array_equal(np.isnan(g3), np.isnan(o3))
        ok = ~np.isnan(o3)
        rel = np.abs(g3[ok] - o3[ok]) / np.maximum(np.abs(o3[ok]), 1e-3 * spp)
        assert (rel <= 1e-4).mean() > 0.999


def test_views_normalize_and_state_preserved(gpu_ctx, b2pt):
    W, H, spp, depth = 32, 32, 5, 5
    views = hemisphere_views(1, 3)
    gpu_ctx.set_camera(b2pt.Camera(48, 16))
    gpu_ctx.render(2, 3)
    before = gpu_ctx.read_color().copy()
    got = gpu_ctx.render_views(views, W, H, spp, depth, flags=b2pt.FLAG_VIEWS_NORMALIZE)
    # the context's own camera and canvas are untouched by the view render
    assert same_bits(gpu_ctx.read_color(), before)
    gpu_ctx.render(2, 3)
    assert same_bits(gpu_ctx.read_color(), before)
    for k, v in enumerate(views):
        gpu_ctx.set_camera(b2pt.Camera(W, H, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9])))
        gpu_ctx.render(spp, depth)
        gpu_ctx.normalize(spp)
        assert same_bits(got[k], gpu_ctx.read_color())


def test_views_stats_and_empty(gpu_ctx, b2pt):
    W, H, spp, depth = 32, 24, 3, 4
    views = hemisphere_views(1, 4)
    gpu_ctx.render_views(views, W, H, spp, depth)
    st = gpu_ctx.stats()
    assert st.paths == 4 * W * H * spp
    assert st.batches == 1  # all four views shared every launch
    assert st.launches <= 2 * depth + 2  # k_primary_prep + two per bounce + k_accumulate
    assert gpu_ctx.render_views(np.zeros((0, 10), np.float32), W, H, spp, depth).shape == (0, W * H, 4)
    z = gpu_ctx.render_views(views, W, H, 0, depth)
    assert not z.any()


def test_views_errors(gpu_ctx, b2pt):
    views = hemisphere_views(1, 2)
    with pytest.raises(b2pt.B2ptError):
        gpu_ctx.render_views(views, 32, 32, 2, 3, flags=b2pt.FLAG_REFERENCE_STREAM)
    bad = views.copy()
    bad[1, 9] = 0.0  # Camera.cxx:720
    with pytest.raises(b2pt.B2ptError, match="feild of view"):
        gpu_ctx.render_views(bad, 32, 32, 2, 3)
    with pytest.raises(b2pt.B2ptError):
        gpu_ctx.render_views(views, 0, 32, 2, 3)


def test_contract(b2pt, monkeypatch):
    """b2pt_render_views at the C level: the code and message of every argument fault (the first fault when a call has
    several), nothing touched by a failing call, the context's own camera and canvas untouched by a sweep, the
    normalised image left on the device without a host output, and the statistics of the per-view fallback."""
    L, p = b2pt.lib(), b2pt._p
    views = hemisphere_views(2, 2)
    w, h, spp, depth = 32, 24, 4, 5
    n, V = w * h, len(views)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(b2pt.Camera(48, 16))
        ctx.render(2, 3)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        full = ctx.render_views(views, w, h, spp, depth)
        st = ctx.stats()
        assert st.paths == n * spp * V
        ptr = L.b2pt_views_device_ptr(ctx._h)
        assert ptr
        # the context's own camera and canvas are untouched by the sweep
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])

        def fails(message, nv, vp, W, H, s, flags=0):
            assert L.b2pt_render_views(ctx._h, nv, vp, W, H, s, depth, flags, None) == b2pt.ERR_BAD_VALUE
            assert L.b2pt_last_error() == message

        vp, ref = p(views), b2pt.FLAG_REFERENCE_STREAM
        bad = views.copy()
        bad[2, 9] = 0.0  # Camera.cxx:720
        fails(b"b2pt_render_views: bad view list", V, None, w, h, spp)
        fails(b"b2pt_render_views: bad view list", -1, vp, w, h, spp)
        fails(b"b2pt_render_views: bad view list", V, None, w, h, -1, ref)
        fails(b"negative sample range", V, vp, w, h, -1)
        fails(b"negative sample range", V, p(bad), w, h, -1, ref)
        fails(b"spp must be positive", V, vp, w, h, 0, b2pt.FLAG_VIEWS_PNM16)
        fails(b"REFERENCE_STREAM cannot be combined with a view-batched render", V, vp, w, h, spp, ref)
        fails(b"REFERENCE_STREAM cannot be combined with a view-batched render", V, p(bad), w, h, 0,
              ref | b2pt.FLAG_VIEWS_PNM16)
        fails(b"Camera feild of view must be greater than zero.", V, p(bad), w, h, spp)
        # more than 2^30 output pixels: 17 views of 8192^2 (2^26 pixels each, the largest canvas)
        big = np.ascontiguousarray(np.repeat(views[:1], 17, axis=0))
        fails(b"b2pt_render_views: more than 2^30 output pixels (16 GiB); split the view list", 17, p(big), 8192, 8192,
              spp)
        bigbad = big.copy()
        bigbad[16, 9] = 0.0
        fails(b"Camera feild of view must be greater than zero.", 17, p(bigbad), 8192, 8192, spp)
        # nothing was rendered: same statistics, same device image
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches) == (st.paths, st.launches, st.batches)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        # VIEWS_NORMALIZE without a host output: the normalised images stay on the device
        want = ctx.render_views(views, w, h, spp, depth, flags=b2pt.FLAG_VIEWS_NORMALIZE)
        assert L.b2pt_render_views(ctx._h, V, vp, w, h, spp, depth, b2pt.FLAG_VIEWS_NORMALIZE, None) == 0
        ptr = L.b2pt_views_device_ptr(ctx._h)
        ctx.set_camera(b2pt.Camera(w, h))
        for v in range(V):
            assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * n * 16)) == 0
            assert same_bits(ctx.read_color(), want[v]), v
        assert L.b2pt_set_color_buffer(ctx._h, None) == 0
        # per-view fallback (a view no longer fits a batch): same images, statistics summed over the views
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(n * 2))
        split = ctx.render_views(views, w, h, spp, depth)
        st3 = ctx.stats()
        monkeypatch.delenv("B2PT_BATCH_PATHS")
        assert same_bits(split, full)
        assert st3.paths == n * spp * V and st3.launches > st.launches
        # nViews == 0 renders nothing and leaves no view image
        assert ctx.render_views(np.zeros((0, 10), np.float32), w, h, spp, depth).shape == (0, n, 4)
        assert not L.b2pt_views_device_ptr(ctx._h)


def pnm_integers(rgba_sum, spp, oracle):
    """numpy restatement of save() (main.cc:325-384) after NormalizeFunctor (:253-287, through the C oracle)."""
    n = oracle.normalize(np.ascontiguousarray(rgba_sum, np.float32), spp)[:, :3].astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        p = 255.99 * n
    return np.where(p >= 65535.0, 65535, np.trunc(np.minimum(p, 65535.0))).astype(np.uint16)


def test_read_pnm16_matches_reference_writer_arithmetic(gpu_ctx, b2pt, oracle):
    W, H, spp = 64, 32, 7
    gpu_ctx.set_camera(b2pt.Camera(W, H))
    gpu_ctx.render(spp, 6)
    sums = gpu_ctx.read_color().copy()
    got = gpu_ctx.read_pnm16(spp)
    assert got.shape == (W * H, 3) and np.array_equal(got, pnm_integers(sums, spp, oracle))
    assert got.max() > 255  # the light is not clamped (the reference prints 991 there)
    assert same_bits(gpu_ctx.read_color(), sums)  # the canvas is left un-normalised
    # corner cases of the arithmetic: NaN channels, zeros, exact integer boundaries, huge and infinite sums
    rng = np.random.default_rng(5)
    c = (rng.random((W * H, 4)) * 3 * spp).astype(np.float32)
    c[0] = [np.nan, 1.0, 2.0, 0.0]
    c[1] = [0.0, -0.0, np.nan, 0.0]
    c[2] = [spp, spp * 4.0, spp * 15.0, 0.0]
    c[3] = [np.inf, 1e30, spp * 65535.0, 0.0]
    c[4] = [spp * (1.0 / 255.99) ** 2, spp * (2.0 / 255.99) ** 2, spp * (255.0 / 255.99) ** 2, 0.0]
    gpu_ctx.write_color(c)
    got = gpu_ctx.read_pnm16(spp)
    assert np.array_equal(got, pnm_integers(c, spp, oracle))
    assert list(got[0]) == [0, 96, 136] and list(got[3][:2]) == [65535, 65535]
    with pytest.raises(b2pt.B2ptError):
        gpu_ctx.read_pnm16(0)


def test_views_pnm16_output(gpu_ctx, b2pt, oracle):
    W, H, spp, depth = 48, 40, 5, 6
    views = hemisphere_views(2, 2)
    sums = gpu_ctx.render_views(views, W, H, spp, depth)
    got = gpu_ctx.render_views(views, W, H, spp, depth, flags=b2pt.FLAG_VIEWS_PNM16)
    assert got.dtype == np.uint16 and got.shape == (4, W * H, 3)
    for k in range(4):
        assert np.array_equal(got[k], pnm_integers(sums[k], spp, oracle))


def test_render_replans_when_memory_was_taken_after_planning(b2pt):
    """The batch target is chosen from the memory that is free at a context's first render.  If another consumer takes
    that memory afterwards, the batch buffers no longer fit: the render halves the target until they do, and the
    image keeps its bits (results never depend on the batch split)."""
    torch = pytest.importorskip("torch")
    cams = (b2pt.Camera(96, 96), b2pt.Camera(768, 768))
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(cams[1])
        ctx.render(48, 6)
        want = ctx.read_color().copy()
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(cams[0])
        ctx.render(2, 3)  # plans the batch target now, with the memory still free
        free, _ = torch.cuda.mem_get_info()
        hog = torch.empty(max(int(free) - (3 << 30), 1 << 20), dtype=torch.uint8, device="cuda")  # leave 3 GiB
        try:
            ctx.set_camera(cams[1])
            ctx.render(48, 6)  # 27 Mi paths: 7.4 GB in one batch does not fit any more
            got = ctx.read_color().copy()
            assert ctx.stats().batches > 1
        finally:
            del hog
            torch.cuda.empty_cache()
    assert same_bits(got, want)


def test_destroy_releases_every_device_buffer(b2pt):
    """b2pt_destroy gives back everything a context allocated -- the view canvases, the camera array and the PNM staging
    buffer included (ADVICE round 1: they used to leak; all buffers are owning DevBufs now)."""
    torch = pytest.importorskip("torch")
    torch.cuda.init()
    torch.cuda.synchronize()
    views = hemisphere_views(2, 3)

    def cycle():
        with b2pt.Context(0) as ctx:
            ctx.set_scene(b2pt.Scene.cornell())
            ctx.build_bvh()
            ctx.set_camera(b2pt.Camera(256, 256))
            ctx.render(8, 6)
            ctx.read_pnm16(8)
            ctx.render_views(views, 256, 256, 4, 5, flags=b2pt.FLAG_VIEWS_PNM16)
            ctx.render_views(views, 256, 256, 4, 5)

    cycle()  # first use loads the module and creates the primary context's pools
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(3):
        cycle()
    free1, _ = torch.cuda.mem_get_info()
    assert abs(free0 - free1) < (64 << 20), (free0, free1)
