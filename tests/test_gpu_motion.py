"""Motion vectors and disocclusion of a view sweep (b2pt_render_views_motion, DESIGN.md 8i) on the GPU: bit-identical to
the restatement on the oracle (tests/motion_ref.c) on every trace path, on a sphere scene and under a lens; exact zeros
and the features' hit counts for identical cameras; independent of chunking and of the checkpoint list; the context is
left alone and bad calls are rejected; the driver's -motion files are the binding's means; and a view warped along its
motion into its neighbour agrees with it within the noise."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_features import (driver_view_names, hemisphere_positions, hemisphere_views, read_pfm, same_bits,  # noqa
                               view_row)
import motion_ref  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
C = 278 / 555.0
FRONT = (C, C, -800 / 555.0)


def right_of(pos, look, delta):
    """pos and look moved by delta along the camera's right axis (the basis' dx: -x for a camera looking along +z)."""
    f = np.asarray(look, np.float64) - np.asarray(pos, np.float64)
    u = np.cross(f / np.linalg.norm(f), (0.0, 1.0, 0.0))
    u /= np.linalg.norm(u)
    return np.asarray(pos) + delta * u, np.asarray(look) + delta * u


def yawed(pos, look, deg):
    a = np.radians(deg)
    d = np.asarray(look, np.float64) - np.asarray(pos, np.float64)
    return np.asarray(pos) + np.array([d[0] * np.cos(a) + d[2] * np.sin(a), d[1], -d[0] * np.sin(a) + d[2] * np.cos(a)])


def camera_pairs():
    """(views, prev_views): hemisphere neighbours, a camera moved so that the tall box hides part of the back wall, a
    rotated camera that sends points off the canvas, and a view compared with itself."""
    hemi = [view_row(p) for p in hemisphere_positions(4, 6)]
    pos, look = right_of(FRONT, (C, C, C), -0.35)
    views = [hemi[8], hemi[15], view_row(FRONT), view_row(FRONT), hemi[20]]
    prev = [hemi[7], hemi[14], view_row(pos, look), view_row(FRONT, yawed(FRONT, (C, C, C), 25.0)), hemi[20]]
    return np.stack(views), np.stack(prev)


def oracle_camera(oracle, row, w, h):
    return oracle.Camera(w, h, pos=row[:3], lookAt=row[3:6], up=tuple(row[6:9]), fov=float(row[9]))


def oracle_scene(oracle, s):
    return oracle.Scene(s.pts, s.quadIds, s.sphPt, s.sphR, s.matIdxQ, s.texIdxQ, s.matIdxS, s.texIdxS, s.matType,
                        s.texType, s.tex, s.lightQuadIds, s.lightSphPt, s.lightSphR, s.lightables, s.refIdx)


def flags_of(b2pt, spec):
    out = 0
    for name in (spec.split("|") if spec else []):
        out |= getattr(b2pt, "FLAG_" + name)
    return out


CASES = [
    ("cornell", 0, 0.0), ("cornell", "FORCE_BVH", 0.0), ("cornell", "FORCE_BVH|GPU_LBVH", 0.0),
    ("cornell", "FORCE_BVH|WIDE_BVH", 0.0), ("spheres", 0, 0.0), ("spheres", "WIDE_BVH", 0.0),
    ("cornell", 0, 0.1), ("cornell", "FORCE_BVH|WIDE_BVH", 0.1), ("spheres", 0, 0.1),
]


@pytest.mark.parametrize("scene_name,build,aperture", CASES)
def test_matches_the_restatement(b2pt, oracle, scene_name, build, aperture):
    w, h, ck, seed = 24, 20, (1, 3), 5
    views, prev = camera_pairs()
    scene = b2pt.Scene.cornell() if scene_name == "cornell" else b2pt.Scene.spheres(700)
    osc = oracle.cornell_scene() if scene_name == "cornell" else oracle_scene(oracle, scene)
    with b2pt.Context(0) as c:
        c.set_scene(scene)
        c.seed(seed)
        c.set_lens(aperture, 0)
        got = c.render_views_motion(views, prev, w, h, ck, flags_of(b2pt, build))
    for v in range(len(views)):
        want = motion_ref.sums(osc, oracle_camera(oracle, views[v], w, h), oracle_camera(oracle, prev[v], w, h), ck,
                               aperture, 0.0, seed)
        assert same_bits(got[:, v], want), v
    if scene_name == "cornell":  # the occluding and off-canvas pairs are not vacuous
        last = got[-1]
        assert (last[2, :, 2] < last[2, :, 3]).sum() > 10 and (last[2, :, 2] > 0).sum() > 100
        assert (last[3, :, 2] < last[3, :, 3]).sum() > 50
        assert np.isfinite(last[..., :2]).all()


def test_identical_cameras(b2pt):
    views, w, h, ck = hemisphere_views(2, 3), 32, 24, (2, 8)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        c.seed(3)
        m = c.render_views_motion(views, views, w, h, ck)
        alb, _ = c.render_views_features(views, w, h, ck)
    assert np.all(m[..., :2] == 0) and not np.signbit(m[..., :2]).any()
    assert same_bits(m[..., 3], alb[..., 3])
    assert np.all(m[..., 2] <= m[..., 3])
    share = np.mean(m[-1, ..., 2] == m[-1, ..., 3])
    print("identical cameras: visible == valid at %.5f of the pixels" % share)
    assert share >= 0.995


def test_chunks_and_checkpoints(b2pt):
    """70 views of 64^2 with K = 32 run in two chunks; they equal per-view calls, and slice k equals a call with the
    first k + 1 checkpoints."""
    pos = hemisphere_positions(7, 10)
    views = np.stack([view_row(p) for p in pos])
    prev = np.concatenate([views[:1], views[:-1]])
    w = h = 64
    ck = tuple(range(1, 33))
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        full = c.render_views_motion(views, prev, w, h, ck)
        for v in range(len(views)):
            assert same_bits(c.render_views_motion(views[v:v + 1], prev[v:v + 1], w, h, ck)[:, 0], full[:, v]), v
        for k in (0, 4, 31):
            part = c.render_views_motion(views, prev, w, h, ck[:k + 1])
            assert same_bits(part[-1], full[k]), k
    assert np.abs(full[-1, ..., 0]).max() > 1


def test_contract(b2pt):
    L, p = b2pt.lib(), b2pt._p
    views = hemisphere_views(2, 3)[:4]
    prev = views[::-1].copy()
    w, h, ck = 32, 24, (1, 3, 4)
    n = w * h
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh()
        ctx.set_camera(b2pt.Camera(48, 16))
        ctx.render(2, 3)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        full = ctx.render_views_checkpoints(views, w, h, ck, 5)
        st = ctx.stats()
        ptr = L.b2pt_views_device_ptr(ctx._h)
        m = ctx.render_views_motion(views, prev, w, h, ck)
        assert same_bits(ctx.render_views_motion(views, prev, w, h, ck), m)  # deterministic

        def fails(message, *args):
            with pytest.raises(b2pt.B2ptError, match=message) as e:
                ctx.render_views_motion(*args)
            assert e.value.code == b2pt.ERR_BAD_VALUE

        fails(r"nCheckpoints must be in \[1,32\]", views, prev, w, h, ())
        fails("checkpoints must be >= 1 and strictly increasing", views, prev, w, h, (2, 2))
        fails(r"more than 2\^24 samples", views, prev, w, h, (1, (1 << 24) + 1))
        for f in (b2pt.FLAG_REFERENCE_STREAM, b2pt.FLAG_VIEWS_NORMALIZE, 1 << 20):
            fails("flags may only hold FORCE_BVH, NO_DEDUP, NO_AA, GPU_LBVH and WIDE_BVH", views, prev, w, h, ck, f)
        bad = views.copy()
        bad[2, 9] = 0.0
        fails("feild of view must be greater than zero", bad, prev, w, h, ck)
        fails("feild of view must be greater than zero", views, bad, w, h, ck)
        fails("width must be greater than zero", views, prev, 0, h, ck)
        vp, pp, c3 = p(views), p(prev), np.array(ck, np.int32)
        out = np.zeros_like(m)
        fn = L.b2pt_render_views_motion
        assert fn(ctx._h, 4, vp, None, w, h, 3, p(c3), 0, p(out)) == b2pt.ERR_BAD_VALUE
        assert b"bad view list" in L.b2pt_last_error()
        assert fn(ctx._h, 4, vp, pp, w, h, 3, p(c3), 0, None) == b2pt.ERR_BAD_VALUE
        assert b"NULL motionOut" in L.b2pt_last_error()
        assert fn(ctx._h, -1, vp, pp, w, h, 3, p(c3), 0, p(out)) == b2pt.ERR_BAD_VALUE
        big = np.arange(1, 18, dtype=np.int32)
        assert fn(ctx._h, 1, vp, pp, 8192, 8192, 17, p(big), 0, p(out)) == b2pt.ERR_BAD_VALUE
        assert b"exceed 2^30 float4" in L.b2pt_last_error()
        assert not out.any()  # nothing ran
        assert fn(ctx._h, 0, None, None, w, h, 3, p(c3), 0, None) == 0
        # the context's statistics, view images, camera and canvas are untouched
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches, st2.segments, st2.tracePath) == \
            (st.paths, st.launches, st.batches, st.segments, st.tracePath)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])
        ctx.set_camera(b2pt.Camera(w, h))
        for v in range(len(views)):
            assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * n * 16)) == 0
            assert same_bits(ctx.read_color(), full[-1][v]), v
        assert L.b2pt_set_color_buffer(ctx._h, None) == 0
    with b2pt.Context(0) as ctx:  # no scene
        with pytest.raises(b2pt.B2ptError) as e:
            ctx.render_views_motion(views, prev, w, h, ck)
        assert e.value.code == b2pt.ERR_STATE


def test_driver_matches_binding(b2pt, tmp_path):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    exe = os.path.join(HOST, "CornellBox_b2pt")
    w, h, spp, aperture = 24, 16, 6, 0.1
    sweep = ["-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", str(spp), "-hemisphere", "-phicount", "2",
             "-thetacount", "3", "-checkpoints", "2,4", "-aperture", str(aperture)]

    def run(name, *extra):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe] + sweep + list(extra), cwd=d, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        return d, sorted(os.listdir(d))

    mdir, files = run("motion", "-features", "-denoise", "-motion")
    pdir, plain = run("plain", "-features", "-denoise")
    order = driver_view_names("hemisphere", hemisphere_positions(2, 3))
    stems = ("output-s2", "output-s4", "output")
    assert files == sorted(plain + ["%s-motion-%s.pfm" % (s, t) for s in stems for t in order])
    for f in plain:  # every other file: byte-identical to a run without -motion
        assert open(mdir / f, "rb").read() == open(pdir / f, "rb").read(), f
    views = np.stack([view_row(pos) for pos in hemisphere_positions(2, 3)])
    prev = np.concatenate([views[:1], views[:-1]])
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        c.set_lens(aperture, 0)
        m = c.render_views_motion(views, prev, w, h, (2, 4, spp))
    for k, stem in enumerate(stems):
        for v, tail in enumerate(order):
            s = m[k, v]
            with np.errstate(invalid="ignore", divide="ignore"):
                want = np.where(s[:, 3:4] > 0, s[:, :3] / s[:, 3:4], np.float32(0)).astype(np.float32)
            assert same_bits(read_pfm(mdir / ("%s-motion-%s.pfm" % (stem, tail)), w, h, 3), want.reshape(-1)), \
                (stem, tail)
    assert np.abs(m[-1, 4, :, 0]).max() > 0.5


def test_warped_view_agrees_with_its_neighbour(b2pt):
    """View v warped along its mean motion into view v-1 agrees with view v-1 at fully visible lambertian pixels, within
    the noise the two images' second moments give."""
    W = H = 128
    spp, depth = 1024, 8
    pos = hemisphere_positions(15, 15)
    a, b = 3 * 15 + 4, 3 * 15 + 5  # neighbours on one ring of the sweep: b is compared with a
    views = np.stack([view_row(pos[a]), view_row(pos[b])])
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        img, m2 = c.render_views_checkpoints(views, W, H, (spp,), depth, moments=True)
        alb, nd = c.render_views_features(views[1:], W, H, (spp,))
        mot = c.render_views_motion(views[1:], views[:1], W, H, (spp,))
    wts = np.array([0.2126, 0.7152, 0.0722])
    mean = np.nan_to_num(img[0].astype(np.float64)[..., :3]) / spp
    sq = np.nan_to_num(m2[0].astype(np.float64)[..., :3]) / spp
    lum = (mean @ wts).reshape(2, H, W)
    var = ((np.maximum(sq - mean ** 2, 0) / (spp - 1)) @ wts ** 2).reshape(2, H, W)
    s = mot[0, 0]
    full = (s[:, 3] == spp) & (s[:, 2] == spp)
    albm = alb[0, 0][:, :3] / spp
    nrm = np.linalg.norm(nd[0, 0][:, :3] / spp, axis=1)
    lambertian = (albm.max(axis=1) <= 0.7301) & (nrm > 0.999)  # every sample on one plane of texture colour
    sel = full & lambertian
    mx, my = s[:, 0] / np.maximum(s[:, 3], 1), s[:, 1] / np.maximum(s[:, 3], 1)
    j, i = np.divmod(np.arange(W * H), W)
    # pixel centre (i + 0.5, j + 0.5) lands at (i + 0.5 + mx, j + 0.5 + my) in view a; bilinear in pixel centres
    x, y = i + mx, j + my
    x0, y0 = np.floor(x).astype(int), np.floor(y).astype(int)
    sel &= (x0 >= 0) & (y0 >= 0) & (x0 + 1 < W) & (y0 + 1 < H)
    idx = np.nonzero(sel)[0]
    fx, fy = x[idx] - x0[idx], y[idx] - y0[idx]

    def bilinear(img2):
        return ((1 - fx) * (1 - fy) * img2[y0[idx], x0[idx]] + fx * (1 - fy) * img2[y0[idx], x0[idx] + 1] +
                (1 - fx) * fy * img2[y0[idx] + 1, x0[idx]] + fx * fy * img2[y0[idx] + 1, x0[idx] + 1])
    warped, wvar = bilinear(lum[0]), bilinear(var[0])
    here = lum[1].reshape(-1)[idx]
    z = np.abs(here - warped) / np.sqrt(var[1].reshape(-1)[idx] + wvar + 1e-12)
    print("warp: %d pixels, mean |motion| %.2f px, mean |z| %.3f, share |z| < 4: %.4f" %
          (idx.size, np.hypot(mx[idx], my[idx]).mean(), z.mean(), (z < 4).mean()))
    assert idx.size > 3000
    assert np.hypot(mx[idx], my[idx]).mean() > 2
    # measured on a B200: 12257 pixels, mean |motion| 2.32 px, mean |z| 0.906, 99.05 % below 4 (deterministic)
    assert (z < 4).mean() > 0.98 and z.mean() < 1.1
