"""A view sweep rendered and temporally denoised in one call (b2pt_render_views_temporal_denoised, DESIGN.md 8k) on the
GPU: every output is, bit for bit, what the four-call chain render_views_checkpoints -> render_views_features ->
render_views_motion (towards the previous view) -> denoise_views_temporal returns through the binding, on the small
scene path, the binary BVH (host and device builders), the 8-wide BVH, a 700-sphere scene, under a lens and with a seed
offset, at the default parameters and at alpha = 1 and levels = 0, across a denoiser chunk boundary and on the render's
per-view path; afterwards the view image and statistics are the render's and the context's camera and canvas are
untouched; bad calls fail before anything runs."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_features import hemisphere_positions, same_bits, view_row  # noqa: E402

pytestmark = pytest.mark.gpu
W, H = 64, 48
CKPTS = (1, 4, 16)
DEPTH = 5
BUILD = 0x8 | 0x4 | 0x10 | 0x80 | 0x1000  # B2PT_BUILD_FLAGS


def chain(views):
    return np.concatenate([views[:1], views[:-1]])


def ring_views(n, ring=3):
    pos = hemisphere_positions(15, 15)
    return np.stack([view_row(pos[ring * 15 + v]) for v in range(n)])


def four_calls(ctx, views, w, h, ck, depth, flags=0, temporal=None, denoise=None):
    """The chain the one call is defined as: (out, history, (color, moment2, albedo, normal_depth, motion))."""
    pnm = flags & 0x200
    color, m2 = ctx.render_views_checkpoints(views, w, h, ck, depth, flags & ~0x200, moments=True)
    alb, nd = ctx.render_views_features(views, w, h, ck, flags & BUILD)
    mot = ctx.render_views_motion(views, chain(views), w, h, ck, flags & BUILD)
    out, n = ctx.denoise_views_temporal(color, m2, alb, nd, mot, views, w, h, ck, temporal, denoise, pnm, history=True)
    return out, n, (color, m2, alb, nd, mot)


def same_as_chain(ctx, views, w, h, ck, depth, flags=0, temporal=None, denoise=None):
    want, wn, wins = four_calls(ctx, views, w, h, ck, depth, flags, temporal, denoise)
    got, n, ins = ctx.render_views_temporal_denoised(views, w, h, ck, depth, temporal, denoise, flags, history=True,
                                                     inputs=True)
    if flags & 0x200:
        assert got.dtype == np.uint16 and np.array_equal(got, want)
    else:
        assert same_bits(got, want)
    assert same_bits(n, wn)
    for name, a, b in zip(("color", "moment2", "albedo", "normal_depth", "motion"), ins, wins):
        assert same_bits(a, b), name
    return got, n, ins


def tparams(b2pt, **kw):
    p = b2pt.TemporalParams.defaults()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def dparams(b2pt, levels):
    p = b2pt.DenoiseParams.defaults()
    p.levels = levels
    return p


CASES = [  # (scene, build flags, aperture, seed offset)
    ("cornell", 0, 0.0, 0), ("cornell", "FORCE_BVH", 0.0, 0), ("cornell", "FORCE_BVH|GPU_LBVH", 0.0, 0),
    ("cornell", "FORCE_BVH|WIDE_BVH", 0.0, 0), ("spheres", 0, 0.0, 0), ("spheres", "WIDE_BVH", 0.0, 0),
    ("cornell", 0, 0.05, 0), ("cornell", "FORCE_BVH|WIDE_BVH", 0.05, 0), ("spheres", 0, 0.05, 0),
    ("cornell", 0, 0.0, 12345), ("cornell", "FORCE_BVH", 0.05, 777),
]


@pytest.mark.parametrize("scene_name,build,aperture,seed", CASES)
def test_is_the_four_call_chain(b2pt, scene_name, build, aperture, seed):
    flags = 0
    for f in (build.split("|") if build else ()):
        flags |= getattr(b2pt, "FLAG_" + f)
    views = ring_views(8)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell() if scene_name == "cornell" else b2pt.Scene.spheres(700))
        c.seed(seed)
        c.set_lens(aperture, 0)
        out, n, ins = same_as_chain(c, views, W, H, CKPTS, DEPTH, flags)
        assert (n > 1).any()  # views take history
        if (scene_name, build, aperture, seed) == ("cornell", 0, 0.0, 0):
            same_as_chain(c, views, W, H, CKPTS, DEPTH, flags | b2pt.FLAG_VIEWS_PNM16)
            same_as_chain(c, views, W, H, CKPTS, DEPTH, flags, tparams(b2pt, alpha=1.0), dparams(b2pt, 0))
            same_as_chain(c, views, W, H, CKPTS, DEPTH, flags, None, dparams(b2pt, 0))
            same_as_chain(c, views, W, H, CKPTS, DEPTH, flags, tparams(b2pt, alpha=1.0), None)


def test_chunk_boundary_and_determinism(b2pt):
    """256 x 128 views in 2 slices: 128 views per chunk of 2^23 float4, so 131 views carry the history of view 127
    across a chunk boundary."""
    pos = hemisphere_positions(15, 15)
    views = np.stack([view_row(pos[v]) for v in range(131)])
    ck = (1, 2)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        out, n, ins = same_as_chain(c, views, 256, 128, ck, 3)
        again, n2, ins2 = c.render_views_temporal_denoised(views, 256, 128, ck, 3, history=True, inputs=True)
    assert same_bits(out, again) and same_bits(n, n2)
    assert all(same_bits(a, b) for a, b in zip(ins, ins2))
    assert (n[:, 128] > 1).any()  # the history crosses the boundary


def test_per_view_render_path(b2pt):
    """A memory budget that sets the batch target to its 1 Mi-path floor: 256 x 256 at 32 samples no longer fits a
    batch, so render_view_sweep renders view by view."""
    views = ring_views(3, ring=5)
    ck = (4, 32)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        c.set_memory_budget(1)
        same_as_chain(c, views, 256, 256, ck, 3)
        st = c.stats()
        assert st.paths == 256 * 256 * 32 * 3 and st.batches > 1


def test_contract(b2pt):
    L, p = b2pt.lib(), b2pt._p
    views = ring_views(3)
    w, h = 24, 16
    ck = np.array((2, 3), np.int32)
    K, V, n = 2, 3, w * h
    out = np.zeros((K, V, n, 4), np.float32)
    with b2pt.Context(0) as ctx:
        assert L.b2pt_render_views_temporal_denoised(ctx._h, V, p(views), w, h, K, p(ck), 5, None, None, 0, p(out),
                                                     *([None] * 6)) == b2pt.ERR_STATE  # no scene
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.set_camera(b2pt.Camera(48, 16))
        ctx.render(2, 3)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        full = ctx.render_views_checkpoints(views, w, h, (2, 3), 5)
        st = ctx.stats()
        ptr = L.b2pt_views_device_ptr(ctx._h)

        def call(nViews=V, v=views, W_=w, H_=h, K_=K, cks=ck, depth=5, tp=None, prm=None, flags=0, o=out):
            return L.b2pt_render_views_temporal_denoised(ctx._h, nViews, p(v), W_, H_, K_, p(cks), depth,
                                                         None if tp is None else ctypes.byref(tp),
                                                         None if prm is None else ctypes.byref(prm), flags, p(o),
                                                         *([None] * 6))

        def fails(message, **kw):
            assert call(**kw) == b2pt.ERR_BAD_VALUE, kw
            assert message.encode() in L.b2pt_last_error(), (message, L.b2pt_last_error())

        fails("nCheckpoints must be in [1,32]", K_=0)
        fails("checkpoints must be >= 1 and strictly increasing", cks=np.array([3, 3], np.int32))
        fails("bad view list", v=None)
        fails("bad view list", nViews=-1)
        badv = views.copy()
        badv[1, 9] = 0.0
        fails("feild of view must be greater than zero", v=badv)
        fails("W and H must be positive", W_=0)
        fails("maxDepth must be in [1,4096]", depth=0)
        fails("REFERENCE_STREAM and VIEWS_NORMALIZE", flags=b2pt.FLAG_REFERENCE_STREAM)
        fails("REFERENCE_STREAM and VIEWS_NORMALIZE", flags=b2pt.FLAG_VIEWS_NORMALIZE)
        fails("NULL out", o=None)
        fails("more than 2^24 samples", cks=np.array([2, (1 << 24) + 1], np.int32))
        fails("levels must be in [0,10]", prm=dparams(b2pt, 11))
        fails("alpha must be in (0,1]", tp=tparams(b2pt, alpha=0.0))
        fails("minVisible must be in [0,1]", tp=tparams(b2pt, minVisible=float("nan")))
        fails("depthTol must be > 0 (or +inf)", tp=tparams(b2pt, depthTol=0.0))
        # 2K nViews W H float4 of render state above 2^30: 5 views of 8192^2 in 2 slices
        big = np.stack([views[0]] * 5)
        fails("more than 2^30 float4 of render state", nViews=5, v=big, W_=8192, H_=8192)
        assert not out.any()  # nothing ran
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches) == (st.paths, st.launches, st.batches)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        assert same_bits(ctx.read_color(), canvas)

        def view_image_is(want):
            ptr = L.b2pt_views_device_ptr(ctx._h)
            for v in range(V):
                assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * n * 16)) == 0
                assert same_bits(ctx.read_color(), want[v]), v
            assert L.b2pt_set_color_buffer(ctx._h, None) == 0

        ctx.set_camera(b2pt.Camera(w, h))
        view_image_is(full[-1])
        assert call(nViews=0, v=None) == 0 and not out.any()
        # a good call leaves the render's view image and statistics; the context's camera and canvas are untouched
        ctx.render_views_checkpoints(views, 8, 8, (1,), 2)  # something else in the view image first
        ctx.render(1, 2)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        got = ctx.render_views_temporal_denoised(views, w, h, ck, 5)
        assert call() == 0 and same_bits(out, got)
        assert ctx.stats().paths == n * 3 * V
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])
        view_image_is(full[-1])
