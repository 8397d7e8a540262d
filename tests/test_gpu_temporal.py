"""Temporal accumulation of a view sweep (b2pt_denoise_views_temporal, DESIGN.md 8j) on the GPU: alpha = 1 is
b2pt_denoise_views bit for bit; levels = 0 is the float32 restatement (tests/temporal_ref.py) bit for bit on a ring of
the driver's hemisphere and on synthetic inputs with NaN, off-canvas and exact-integer motion, motion onto and just
past the canvas' first and last columns and rows, and hard guide edges, on canvases from 1 x 1, one column and one row
up to one pixel past the 16 x 16 tile; the default levels agree with denoise_ref applied to the restated history, and
so do ten levels on the synthetic canvases; a view chain that crosses a chunk boundary is still the restatement;
disoccluded pixels take no history; the accumulation lowers the error against a 4096-spp target; bad calls fail before
anything runs; the driver's -temporal files are the binding's pipeline."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_ref as R  # noqa: E402
import temporal_ref as T  # noqa: E402
from test_gpu_denoise import CANVASES, TOL_ALL, rel_err, rel_mse, synthetic  # noqa: E402
from test_gpu_features import driver_view_names, hemisphere_positions, same_bits, view_row  # noqa: E402
from test_gpu_motion import FRONT, right_of  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
C = 278 / 555.0
INF = float("inf")
W, H = 64, 48
CKPTS = (1, 4, 16)


def chain(views):
    """prevViews of a sweep: every view towards the one before it, the first towards itself."""
    return np.concatenate([views[:1], views[:-1]])


def ring_views(n, first=0, ring=3):
    """n consecutive views of one ring of the driver's 15 x 15 hemisphere."""
    pos = hemisphere_positions(15, 15)
    return np.stack([view_row(pos[ring * 15 + first + v]) for v in range(n)])


def tparams(b2pt, **kw):
    p = b2pt.TemporalParams.defaults()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def dparams(b2pt, levels=None):
    p = b2pt.DenoiseParams.defaults()
    if levels is not None:
        p.levels = levels
    return p


@pytest.fixture(scope="module")
def ring(b2pt):
    """8 consecutive views of ring 3 at 64 x 48, checkpoints (1, 4, 16): sums, squares, guides and motion."""
    views = ring_views(8)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        color, m2 = c.render_views_checkpoints(views, W, H, CKPTS, 5, 0, moments=True)
        alb, nd = c.render_views_features(views, W, H, CKPTS)
        mot = c.render_views_motion(views, chain(views), W, H, CKPTS)
    return dict(views=views, color=color, m2=m2, alb=alb, nd=nd, mot=mot)


def run(ctx, s, moments=True, temporal=None, params=None, flags=0, history=True):
    return ctx.denoise_views_temporal(s["color"], s["m2"] if moments else None, s["alb"], s["nd"], s["mot"],
                                      s["views"], W, H, CKPTS, temporal, params, flags, history)


def test_alpha_one_is_denoise_views(b2pt, ring):
    s = ring
    with b2pt.Context(0) as c:  # no scene: neither call needs one
        for levels in (0, 5):
            p = dparams(b2pt, levels)
            out, n = run(c, s, temporal=tparams(b2pt, alpha=1.0), params=p)
            want = c.denoise_views(s["color"], s["m2"], s["alb"], s["nd"], W, H, CKPTS, p)
            assert same_bits(out, want), levels
            assert (n == 1).all()
            pnm = run(c, s, temporal=tparams(b2pt, alpha=1.0), params=p, flags=b2pt.FLAG_VIEWS_PNM16, history=False)
            assert np.array_equal(pnm, c.denoise_views(s["color"], s["m2"], s["alb"], s["nd"], W, H, CKPTS, p,
                                                       b2pt.FLAG_VIEWS_PNM16)), levels


@pytest.mark.parametrize("moments", [True, False])
def test_ring_levels_zero_is_the_restatement(b2pt, ring, moments):
    s = ring
    with b2pt.Context(0) as c:
        out, n = run(c, s, moments, params=dparams(b2pt, 0))
        inf_out, inf_n = run(c, s, moments, temporal=tparams(b2pt, normalTol=INF, albedoTol=INF, depthTol=INF),
                             params=dparams(b2pt, 0))
    q = s["m2"] if moments else None
    x, V, hn = T.temporal(s["color"], q, s["alb"], s["nd"], s["mot"], s["views"], W, H, CKPTS)
    assert same_bits(out[..., :3], x) and same_bits(out[..., 3], V) and same_bits(n, hn)
    x, V, hn = T.temporal(s["color"], q, s["alb"], s["nd"], s["mot"], s["views"], W, H, CKPTS, normal_tol=INF,
                          albedo_tol=INF, depth_tol=INF)
    assert same_bits(inf_out[..., :3], x) and same_bits(inf_out[..., 3], V) and same_bits(inf_n, hn)
    # not vacuous: histories grow along the ring, and the tolerances reject some taps
    assert n[:, -1].max() > 7.9 and (n[:, 1:] == 1).any() and (inf_n != n).any()
    if not moments:
        assert (out[..., 3] == 0).all()


def synthetic_motion(K, V, h, w, ck, seed=0):
    """Motion sums with fractional, exact-integer, off-canvas and NaN motion, NaN sums, no valid sample and partial
    visibility, and motion onto the canvas' edges: exactly onto the last column or row (zero fraction, so the second
    column or row of taps is off the canvas), a little left of or above it (floorf gives -1, so the first is), and a
    little right of or below it (the second is)."""
    rng = np.random.default_rng(seed)
    N = h * w
    j, i = np.divmod(np.arange(N), w)
    M = np.zeros((K, V, N, 4), np.float32)
    for k, c in enumerate(ck):
        cf = np.float32(c)
        mx = rng.uniform(-1.5, 1.5, (V, N)).astype(np.float32)
        my = rng.uniform(-1.5, 1.5, (V, N)).astype(np.float32)
        kind = rng.integers(0, 14, (V, N))
        mx = np.where(kind == 1, np.round(mx), mx)  # exact integers
        my = np.where(kind == 1, np.round(my), my)
        mx = np.where(kind == 2, np.float32(3 * w), mx)  # off the canvas
        my = np.where(kind == 3, np.float32(-1e30), my)
        # every one exact in float32, and so are its sums and i + Sx / Sval
        mx = np.where(kind == 8, (w - 1 - i).astype(np.float32), mx)
        my = np.where(kind == 9, (h - 1 - j).astype(np.float32), my)
        mx = np.where(kind == 10, (-0.125 - i).astype(np.float32), mx)
        my = np.where(kind == 11, (-0.125 - j).astype(np.float32), my)
        mx = np.where(kind == 12, (w - 1 - i + 0.375).astype(np.float32), mx)
        my = np.where(kind == 13, (h - 1 - j + 0.375).astype(np.float32), my)
        M[k, ..., 0] = mx * cf
        M[k, ..., 1] = my * cf
        M[k, ..., 3] = cf
        M[k, ..., 2] = np.where(kind == 4, np.floor(0.3 * cf), cf)
        M[k, ..., 0] = np.where(kind == 5, np.nan, M[k, ..., 0])
        M[k, ..., 3] = np.where(kind == 6, 0, M[k, ..., 3])
        M[k, ..., 2] = np.where((kind == 7) & (rng.random((V, N)) < 0.5), np.nan, M[k, ..., 2])
    return M


@pytest.mark.parametrize("moments", [True, False])
def test_synthetic_levels_zero_is_the_restatement(b2pt, moments):
    """On every canvas of test_gpu_denoise.CANVASES (at least 240 pixels of views in all): levels 0 is the restatement
    bit for bit, and ten levels agree with it within TOL_ALL."""
    names = dict(alpha="alpha", minVisible="min_visible", normalTol="normal_tol", albedoTol="albedo_tol",
                 depthTol="depth_tol")
    with b2pt.Context(0) as c:
        for w, h in CANVASES:
            nv = max(5, 240 // (w * h))
            ck, S, Q, A, ND = synthetic(2, nv, h, w)
            Q = Q if moments else None
            views = np.stack([view_row(FRONT, fov=40.0)] * nv)
            M = synthetic_motion(2, nv, h, w, ck)
            for tp in (dict(), dict(alpha=0.05, minVisible=0.0), dict(normalTol=INF, albedoTol=INF, depthTol=INF)):
                out, n = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, tparams(b2pt, **tp),
                                                  dparams(b2pt, 0), history=True)
                rp = {names[k]: v for k, v in tp.items()}
                x, V, hn = T.temporal(S, Q, A, ND, M, views, w, h, ck, **rp)
                assert same_bits(out[..., :3], x) and same_bits(out[..., 3], V) and same_bits(n, hn), (w, h, tp)
                assert (n[:, 1:] > 1).mean() > 0.1 and (n[:, 1:] == 1).mean() > 0.1, (w, h, tp)
                out = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, tparams(b2pt, **tp), dparams(b2pt, 10))
                x, V = T.filtered(S, Q, A, ND, M, views, w, h, ck, rp, levels=10)
                assert rel_err(out[..., :3], x) < TOL_ALL, (w, h, tp)
                if moments:
                    assert rel_err(out[..., 3:], V[..., None]) < 10 * TOL_ALL, (w, h, tp)


def test_default_levels_against_the_restatement(b2pt, ring):
    s = ring
    with b2pt.Context(0) as c:
        out = run(c, s, history=False)
    x, V = T.filtered(s["color"], s["m2"], s["alb"], s["nd"], s["mot"], s["views"], W, H, CKPTS)
    assert rel_err(out[..., :3], x) < TOL_ALL
    assert rel_err(out[1:, ..., 3:], V[1:, ..., None]) < 10 * TOL_ALL  # c = 1 has no variance


def test_chunk_boundary_and_determinism(b2pt):
    """256 x 128 images in 2 slices: 2^16 float4 per view, 128 views per chunk of 2^23; 131 views cross it, so view 128
    takes its history from the state carried over from the first chunk."""
    h, w, V = 128, 256, 131
    ck = np.array([2, 6], np.int32)
    rng = np.random.default_rng(3)
    N = h * w
    S = (rng.random((2, V, N, 4), np.float32) * ck[:, None, None, None]).astype(np.float32)
    Q = S * S
    A = np.repeat(rng.random((2, V, 1, 4), np.float32) * 0.05 + 0.5, N, 2)
    A[..., 3] = ck[:, None, None]
    ND = np.zeros((2, V, N, 4), np.float32)
    ND[..., 2] = -ck[:, None, None]
    views = np.stack([view_row(FRONT)] * V)
    d = T.centre_directions(views[0], w, h)
    ND[..., 3] = ((np.float32(1) - views[0, 2]) / d[:, 2])[None, None] * ck[:, None, None]
    M = synthetic_motion(2, V, h, w, ck, seed=4)
    with b2pt.Context(0) as c:
        out, n = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, None, dparams(b2pt, 0), history=True)
        again, n2 = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, None, dparams(b2pt, 0), history=True)
        full = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck)
        full2 = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck)
    assert same_bits(out, again) and same_bits(n, n2) and same_bits(full, full2)
    x, Vb, hn = T.temporal(S, Q, A, ND, M, views, w, h, ck)
    assert same_bits(out[..., :3], x) and same_bits(out[..., 3], Vb) and same_bits(n, hn)
    assert (n[:, 128] > 1).mean() > 0.2  # the history crosses the boundary


def test_disocclusion(b2pt):
    """The sideways move of the motion tests: the tall box uncovers part of the back wall.  Pixels whose visible fraction
    is below minVisible start a new history (n = 1, out = m at levels 0)."""
    w, h, ck = 64, 48, (16,)
    pos, look = right_of(FRONT, (C, C, C), -0.35)
    views = np.stack([view_row(pos, look), view_row(FRONT)])
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        color, m2 = c.render_views_checkpoints(views, w, h, ck, 5, 0, moments=True)
        alb, nd = c.render_views_features(views, w, h, ck)
        mot = c.render_views_motion(views, chain(views), w, h, ck)
        out, n = c.denoise_views_temporal(color, m2, alb, nd, mot, views, w, h, ck, None, dparams(b2pt, 0),
                                          history=True)
    m, V0, *_ = R.prep(color, m2, alb, nd, ck)
    s = mot[0, 1]
    hidden = (s[:, 3] > 0) & (s[:, 2] < 0.5 * s[:, 3])
    print("disocclusion: %d pixels below minVisible, %d with history" % (hidden.sum(), (n[0, 1] > 1).sum()))
    assert hidden.sum() > 10 and (n[0, 1] > 1).sum() > 1000
    assert (n[0, 1][hidden] == 1).all()
    assert same_bits(out[0, 1][hidden][:, :3], m[0, 1][hidden]) and same_bits(out[0, 1][hidden][:, 3], V0[0, 1][hidden])


# Measured on a B200 (DESIGN.md 8j); the bounds leave room above the measured ratios.
RATIO_TEMPORAL, RATIO_FILTERED = 0.2, 0.4


def test_quality(b2pt):
    """One ring of 15 views at 128^2, depth 8, checkpoints (4, 16), against a 4096-spp target, rel-MSE of DESIGN.md 8e on
    the lambertian pixels of views >= 5: the temporal result at levels 0 beats the noisy mean where n >= 5, and
    temporal + the default filter beats the filter alone at 4 spp.  The dielectric sphere (view-dependent) is reported
    apart."""
    w = h = 128
    ck, depth = (4, 16), 8
    views = ring_views(15, ring=3)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        color, m2 = c.render_views_checkpoints(views, w, h, ck, depth, 0, moments=True)
        alb, nd = c.render_views_features(views, w, h, ck)
        mot = c.render_views_motion(views, chain(views), w, h, ck)
        target = c.render_views(views, w, h, 4096, depth)[..., :3] / np.float32(4096)
        t0, n = c.denoise_views_temporal(color, m2, alb, nd, mot, views, w, h, ck, None, dparams(b2pt, 0),
                                         history=True)
        tf = c.denoise_views_temporal(color, m2, alb, nd, mot, views, w, h, ck)
        sp = c.denoise_views(color, m2, alb, nd, w, h, ck)
    target = np.nan_to_num(target.astype(np.float64))
    albm = alb[-1][..., :3] / ck[-1]
    nrm = np.linalg.norm(nd[-1][..., :3] / ck[-1], axis=-1)
    lamb = (albm.max(-1) <= 0.7301) & (nrm > 0.999)
    glass = (albm.min(-1) >= 0.999) & (albm.max(-1) <= 1.001) & (alb[-1][..., 3] == ck[-1]) & (target.max(-1) < 5)
    late = np.zeros(lamb.shape, bool)
    late[5:] = True
    report = {}
    for k, cnt in enumerate(ck):
        noisy = np.nan_to_num(color[k, ..., :3].astype(np.float64)) / cnt
        for name, mask in (("lambertian", lamb & late), ("lambertian n>=5", lamb & late & (n[k] >= 5)),
                           ("dielectric", glass & late)):
            if not mask.any():  # the sphere may be hidden from a ring: report nothing rather than an empty mean
                continue
            report[(cnt, name)] = tuple(rel_mse(a[mask][:, :3].astype(np.float64), target[mask])
                                        for a in (noisy, t0[k], sp[k], tf[k]))
    for key, (rn, rt, rs, rtf) in sorted(report.items()):
        print("%2d spp %-16s noisy %.4f temporal %.4f (%.3f) spatial %.4f temporal+spatial %.4f (%.3f of spatial)" %
              (key[0], key[1], rn, rt, rt / rn, rs, rtf, rtf / rs))
    mean_n = n[:, 5:][:, lamb[5:]].mean(-1)
    print("mean history on lambertian pixels of views >= 5: %s" % mean_n)
    g = glass & late
    print("dielectric pixels (albedo 1, not the light) of views >= 5: %d" % g.sum())
    # the independence the V_bar rule assumes: actual squared error over predicted variance, split by |motion|
    s = mot[0]
    speed = np.hypot(s[..., 0], s[..., 1]) / np.maximum(s[..., 3], 1)
    err2 = ((t0[0][..., :3].astype(np.float64) - target) @ R.LUM) ** 2
    for name, mask in (("|motion| < 1 px", speed < 1), ("|motion| >= 1 px", speed >= 1)):
        sel = lamb & late & (n[0] >= 5) & mask
        if sel.sum():
            print("4 spp, n >= 5, %s: %d pixels, mean squared luminance error / mean V_bar = %.3f" %
                  (name, sel.sum(), err2[sel].mean() / t0[0][..., 3][sel].mean()))
    rn, rt, _, _ = report[(4, "lambertian n>=5")]
    _, _, rs, rtf = report[(4, "lambertian")]
    assert rt < RATIO_TEMPORAL * rn, report
    assert rtf < RATIO_FILTERED * rs, report


def test_contract(b2pt, ring):
    L, p = b2pt.lib(), b2pt._p
    s = ring
    color, m2, alb, nd, mot = (np.ascontiguousarray(s[k][:, :3]) for k in ("color", "m2", "alb", "nd", "mot"))
    views = np.ascontiguousarray(s["views"][:3])
    ck = np.array(CKPTS, np.int32)
    out = np.zeros((3, 3, W * H, 4), np.float32)
    hist = np.zeros((3, 3, W * H), np.float32)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.set_camera(b2pt.Camera(48, 16))
        ctx.render(2, 3)
        canvas, hits = ctx.read_color().copy(), ctx.primary_hits()
        full = ctx.render_views_checkpoints(views, 24, 16, (2, 3), 5)
        st = ctx.stats()
        ptr = L.b2pt_views_device_ptr(ctx._h)
        good, gh = ctx.denoise_views_temporal(color, m2, alb, nd, mot, views, W, H, ck, history=True)

        def call(nViews=3, v=views, w=W, h=H, K=3, cks=ck, c=color, q=m2, a=alb, n=nd, m=mot, tp=None, prm=None,
                 flags=0, o=out, ho=hist):
            return L.b2pt_denoise_views_temporal(ctx._h, nViews, p(v), w, h, K, p(cks), p(c), p(q), p(a), p(n), p(m),
                                                 None if tp is None else ctypes.byref(tp),
                                                 None if prm is None else ctypes.byref(prm), flags, p(o), p(ho))

        def fails(message, **kw):
            assert call(**kw) == b2pt.ERR_BAD_VALUE, kw
            assert message.encode() in L.b2pt_last_error(), (message, L.b2pt_last_error())

        # what b2pt_denoise_views rejects
        fails("nCheckpoints must be in [1,32]", K=0)
        fails("checkpoints must be >= 1 and strictly increasing", cks=np.array([1, 4, 4], np.int32))
        for kw in (dict(c=None), dict(a=None), dict(n=None), dict(o=None)):
            fails("color, albedo, normalDepth and out must not be NULL", **kw)
        fails("W and H must be positive", w=0)
        fails("negative view count", nViews=-1)
        fails("levels must be in [0,10]", prm=dparams(b2pt, 11))
        bad = dparams(b2pt)
        bad.sigmaDepth = float("nan")
        fails("must be > 0 (or +inf)", prm=bad)
        for f in (b2pt.FLAG_VIEWS_NORMALIZE, b2pt.FLAG_FORCE_BVH, 1 << 20):
            fails("flags may only hold VIEWS_PNM16", flags=f)
        fails("slices exceed 2^30 float4", nViews=1, w=8192, h=8192, K=17, cks=np.arange(1, 18, dtype=np.int32))
        # and its own
        fails("bad view list", v=None)
        fails("NULL motion", m=None)
        badv = views.copy()
        badv[1, 9] = 0.0
        fails("feild of view must be greater than zero", v=badv)
        for a in (0.0, -0.5, 1.5, float("nan"), INF):
            fails("alpha must be in (0,1]", tp=tparams(b2pt, alpha=a))
        for mv in (-0.1, 1.01, float("nan")):
            fails("minVisible must be in [0,1]", tp=tparams(b2pt, minVisible=mv))
        for name in ("normalTol", "albedoTol", "depthTol"):
            for b in (0.0, -1.0, float("nan"), -INF):
                fails("%s must be > 0 (or +inf)" % name, tp=tparams(b2pt, **{name: b}))
        assert not out.any() and not hist.any()  # nothing ran
        assert call(nViews=0, v=None, m=None) == 0 and not out.any()
        # NULL parameters are the defaults; history may be NULL
        assert call(tp=b2pt.TemporalParams.defaults(), prm=b2pt.DenoiseParams.defaults()) == 0
        assert same_bits(out, good) and same_bits(hist, gh)
        assert call(ho=None) == 0 and same_bits(out, good)
        # the context's statistics, view images, camera and canvas are untouched
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches, st2.segments, st2.tracePath) == \
            (st.paths, st.launches, st.batches, st.segments, st.tracePath)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])
        ctx.set_camera(b2pt.Camera(24, 16))
        for v in range(3):
            assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * 24 * 16 * 16)) == 0
            assert same_bits(ctx.read_color(), full[-1][v]), v
        assert L.b2pt_set_color_buffer(ctx._h, None) == 0
    with b2pt.Context(0) as ctx:  # no scene: the call needs none
        assert same_bits(ctx.denoise_views_temporal(color, m2, alb, nd, mot, views, W, H, ck), good)


def test_driver_temporal(b2pt, tmp_path):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    exe = os.path.join(HOST, "CornellBox_b2pt")
    w, h, spp = 24, 16, 6
    sweep = ["-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", str(spp), "-hemisphere", "-phicount", "2",
             "-thetacount", "3", "-checkpoints", "2,4"]

    def drive(name, *extra):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe] + sweep + list(extra), cwd=d, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        return d, sorted(os.listdir(d))

    tdir, files = drive("temporal", "-features", "-denoise", "-motion", "-temporal")
    pdir, plain = drive("plain", "-features", "-denoise", "-motion")
    order = driver_view_names("hemisphere", hemisphere_positions(2, 3))
    stems = ("output-s2", "output-s4", "output")
    assert files == sorted(plain + ["%s-temporal-%s.pnm" % (s, t) for s in stems for t in order])
    for f in plain:  # every other file: byte-identical to a run without -temporal
        assert open(tdir / f, "rb").read() == open(pdir / f, "rb").read(), f
    views = np.stack([view_row(pos) for pos in hemisphere_positions(2, 3)])
    counts = (2, 4, spp)
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        color, m2 = c.render_views_checkpoints(views, w, h, counts, 5, 0, moments=True)
        alb, nd = c.render_views_features(views, w, h, counts)
        mot = c.render_views_motion(views, chain(views), w, h, counts)
        want, n = c.denoise_views_temporal(color, m2, alb, nd, mot, views, w, h, counts,
                                           flags=b2pt.FLAG_VIEWS_PNM16, history=True)
    assert (n > 1).any()
    for k, stem in enumerate(stems):
        for v, tail in enumerate(order):
            body = "".join("%d %d %d\n" % tuple(px) for px in want[k, v])
            text = "P3\n%d %d 255\n" % (w, h) + body
            assert open(tdir / ("%s-temporal-%s.pnm" % (stem, tail))).read() == text, (stem, tail)
