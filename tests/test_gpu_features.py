"""Denoiser guide buffers of a view sweep (b2pt_render_views_features, k_view_features): per pixel, the first-hit
albedo, hit count, normal and depth of the renderer's own path samples, summed in sample order at every checkpoint.

Bar: every slice is BIT-IDENTICAL to a per-sample reference built from the existing parity hooks (b2pt_create_rays with
the render's seeds pixel + seedOffset + s * GOLDEN, then b2pt_intersect), with the albedo rule applied in numpy and a
sequential float32 sum; hit counts and depth sums equal the oracle's primary hits; results do not depend on the view
chunking or on the trace structure; and the driver's PFM files are the binding's sums through its mean formulas."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
GOLDEN = 0x9E3779B9
C = 278 / 555.0
W, H = 64, 48
CKPTS = (1, 2, 5, 7)


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


@pytest.fixture(scope="module")
def cornell(b2pt):
    """A context of its own (these tests change the seed offset and the trace structure)."""
    scene = b2pt.Scene.cornell()
    ctx = b2pt.Context(0)
    ctx.set_scene(scene)
    ctx.build_bvh()
    yield ctx, scene
    ctx.close()


def hemisphere_views(n_phi, n_theta, fov=40.0):
    """n_phi x n_theta view points in front of the box opening, tilted up vectors and varying fields of view."""
    c = np.array([C] * 3, np.float32)
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


def view_row(pos, lookAt=(C, C, C), up=(0, 1, 0), fov=40.0):
    return np.concatenate([np.asarray(pos, np.float32), np.asarray(lookAt, np.float32), np.asarray(up, np.float32),
                           [fov]]).astype(np.float32)


def camera(b2pt_or_oracle, v, w, h):
    return b2pt_or_oracle.Camera(w, h, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9]))


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def seeds(n, off, s):
    return ((np.arange(n, dtype=np.uint64) + off + s * GOLDEN) % (1 << 32)).astype(np.uint32)


def sample_features(ctx, scene, n, off, s):
    """One path sample of every pixel of the context's camera through the parity hooks: (albedo rgb + hit,
    normal xyz + depth, prim ids, hit records)."""
    _, d, o, _ = ctx.create_rays(seeds(n, off, s))
    prim, rec, mat, texi = ctx.intersect(o, d, 0.001)
    hit = prim >= 0
    a = np.zeros((n, 4), np.float32)
    nd = np.zeros((n, 4), np.float32)
    kind = scene.matType[mat[hit]]
    col = scene.tex[scene.texType[texi[hit]]]
    alb = np.where((kind == 2)[:, None], np.float32(1), np.where((kind == 1)[:, None], np.clip(col, 0, 1), col))
    a[hit, :3] = alb
    a[hit, 3] = 1
    nd[hit, :3] = rec[3:6].T[hit]
    nd[hit, 3] = rec[2][hit]
    return a, nd, prim, rec


def reference(ctx, b2pt, scene, views, w, h, counts, off=0):
    """[K, view, pixel, 4] albedo and normal/depth sums, in sample order from +0.0 (float32 adds, as the kernel)."""
    n = w * h
    K = len(counts)
    ra = np.zeros((K, len(views), n, 4), np.float32)
    rn = np.zeros((K, len(views), n, 4), np.float32)
    for v, row in enumerate(views):
        ctx.set_camera(camera(b2pt, row, w, h))
        sa = np.zeros((n, 4), np.float32)
        sn = np.zeros((n, 4), np.float32)
        k = 0
        for s in range(counts[-1]):
            a, nd, _, _ = sample_features(ctx, scene, n, off, s)
            sa = sa + a
            sn = sn + nd
            if s + 1 == counts[k]:
                ra[k, v], rn[k, v] = sa, sn
                k += 1
    return ra, rn


@pytest.mark.parametrize("w, h, off", [(W, H, 0), (33, 20, 0), (W, H, 0x7654321)])
def test_bit_identical_to_per_sample_reference(cornell, b2pt, w, h, off):
    ctx, scene = cornell
    views = hemisphere_views(2, 3)
    ctx.seed(off)
    try:
        alb, nd = ctx.render_views_features(views, w, h, CKPTS)
        ra, rn = reference(ctx, b2pt, scene, views, w, h, CKPTS, off)
    finally:
        ctx.seed(0)
    assert alb.shape == (4, 6, w * h, 4) and nd.shape == alb.shape and alb.dtype == np.float32
    assert same_bits(alb, ra) and same_bits(nd, rn)
    hits = alb[..., 3]
    assert (hits[-1] == 7).mean() > 0.3 and alb[-1][..., :3].max() > 0 and nd[-1][..., 3].max() > 0
    assert not same_bits(alb[0], alb[1])
    if off:  # the seed offset moves the samples
        alb0, _ = ctx.render_views_features(views, w, h, CKPTS)
        assert not same_bits(alb0, alb)


def test_hits_and_depth_match_oracle(cornell, b2pt, oracle):
    ctx, _ = cornell
    views = hemisphere_views(2, 3)[[0, 4]]
    off = 99
    ctx.seed(off)
    try:
        alb, nd = ctx.render_views_features(views, W, H, CKPTS)
    finally:
        ctx.seed(0)
    sc = oracle.cornell_scene()
    for v, row in enumerate(views):
        cnt = np.zeros(W * H, np.float32)
        dep = np.zeros(W * H, np.float32)
        k = 0
        for s in range(CKPTS[-1]):
            prim, t = oracle.primary_hits(sc, camera(oracle, row, W, H), seed_offset=(off + s * GOLDEN) % (1 << 32))
            cnt = cnt + (prim >= 0).astype(np.float32)
            dep = dep + np.where(prim >= 0, t, np.float32(0)).astype(np.float32)
            if s + 1 == CKPTS[k]:
                assert same_bits(alb[k, v, :, 3], cnt), (v, s)
                assert same_bits(nd[k, v, :, 3], dep), (v, s)
                k += 1


def test_prefix_property_and_determinism(gpu_ctx, b2pt):
    views = hemisphere_views(2, 2)
    alb, nd = gpu_ctx.render_views_features(views, W, H, CKPTS)
    alb2, nd2 = gpu_ctx.render_views_features(views, W, H, CKPTS)
    assert same_bits(alb, alb2) and same_bits(nd, nd2)
    for k, c in enumerate(CKPTS):
        a1, n1 = gpu_ctx.render_views_features(views, W, H, (c,))
        assert a1.shape == (1, 4, W * H, 4)
        assert same_bits(a1[0], alb[k]) and same_bits(n1[0], nd[k]), c


def test_chunk_boundary(cornell, b2pt):
    """128^2 views with 4 checkpoints: 2^23 float4 of staging per output hold 128 views, so 130 views take two chunks."""
    ctx, scene = cornell
    w = h = 128
    n = 130
    i = np.arange(n)
    z = (i + 0.5) * (1.0 / n) - 1.0  # the lower half of a Fibonacci lattice: every view sees into the box
    rad = np.sqrt(1 - z * z)
    az = i * math.pi * (3 - math.sqrt(5))
    views = np.stack([view_row([C + 0.95 * rad[k] * math.cos(az[k]), C + 0.95 * rad[k] * math.sin(az[k]),
                                C + 1.9 * z[k]]) for k in range(n)])
    alb, nd = ctx.render_views_features(views, w, h, CKPTS)
    per_chunk = (1 << 23) // (len(CKPTS) * w * h)
    assert per_chunk == 128
    for v in (0, per_chunk - 1, per_chunk, n - 1):
        a1, n1 = ctx.render_views_features(views[v:v + 1], w, h, CKPTS)
        assert same_bits(alb[:, v], a1[:, 0]) and same_bits(nd[:, v], n1[:, 0]), v
    ra, rn = reference(ctx, b2pt, scene, views[[per_chunk - 1, per_chunk]], w, h, CKPTS)
    assert same_bits(alb[:, per_chunk - 1:per_chunk + 1], ra) and same_bits(nd[:, per_chunk - 1:per_chunk + 1], rn)
    assert not same_bits(alb[:, per_chunk - 1], alb[:, per_chunk])


@pytest.mark.parametrize("flags", ["FORCE_BVH", "FORCE_BVH|GPU_LBVH", "FORCE_BVH|WIDE_BVH"])
def test_bvh_paths_equal_small_scene_path(gpu_ctx, b2pt, flags):
    views = hemisphere_views(2, 3)
    want = gpu_ctx.render_views_features(views, W, H, CKPTS)
    f = 0
    for name in flags.split("|"):
        f |= getattr(b2pt, "FLAG_" + name)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        got = ctx.render_views_features(views, W, H, CKPTS, f)
        assert same_bits(got[0], want[0]) and same_bits(got[1], want[1]), flags
        # the flags chose the structure as a render would: the render's statistics name the BVH path
        ctx.set_camera(b2pt.Camera(16, 16))
        ctx.render(1, 2, f)
        assert ctx.stats().tracePath == 1


def generated_scene(b2pt, seed=7, n_quads=200):
    """About 200 random parallelograms, each inside its own cell of a 6^3 grid of unit cells with gaps around it;
    about a third rotated arbitrarily, the rest axis-aligned; two made non-planar by lifting a corner.  Six spheres
    (four at the centres of quad cells, two in empty cells).  Material and texture indices cycle through the Cornell
    tables, so lambertian, emitter (its colour 15 clamped) and dielectric primitives all occur."""
    rng = np.random.default_rng(seed)
    cells = rng.permutation(216)
    pts, quads = [], []
    for q in range(n_quads):
        c = cells[q]
        centre = np.array([c % 6, (c // 6) % 6, c // 36], np.float64) + 0.5
        a = np.zeros(3)
        b = np.zeros(3)
        if q % 3 == 0:  # rotated: random unit vectors
            a = rng.normal(size=3)
            b = np.cross(a, rng.normal(size=3)) + 0.4 * a
        else:  # axis-aligned rectangle
            u, v = rng.choice(3, 2, replace=False)
            a[u], b[v] = 1.0, 1.0
        a *= rng.uniform(0.2, 0.35) / np.linalg.norm(a)
        b *= rng.uniform(0.2, 0.35) / np.linalg.norm(b)
        v00 = centre - 0.5 * (a + b)
        corners = [v00, v00 + a, v00 + a + b, v00 + b]
        if q in (5, 11):  # non-planar: lift the third corner along the normal
            nrm = np.cross(a, b)
            corners[2] = corners[2] + 0.3 * np.linalg.norm(a) * nrm / np.linalg.norm(nrm)
        base = len(pts)
        pts += [p.astype(np.float32) for p in corners]
        quads.append([q, base, base + 1, base + 2, base + 3])
    sph_cells = list(cells[:4]) + list(cells[n_quads:n_quads + 2])
    sph_pt = []
    for c in sph_cells:
        sph_pt.append(len(pts))
        pts.append((np.array([c % 6, (c // 6) % 6, c // 36], np.float64) + 0.5).astype(np.float32))
    n_sph = len(sph_pt)
    sph_r = np.full(n_sph, 0.2, np.float32)
    cb = b2pt.Scene.cornell()
    args = (np.array(pts, np.float32), np.array(quads, np.int64), np.array(sph_pt, np.int64), sph_r,
            np.arange(n_quads) % 5, np.arange(n_quads) % 4, np.arange(n_sph) % 5, np.arange(n_sph) % 4,
            cb.matType, cb.texType, cb.tex)
    return b2pt.Scene(*args, lightQuadIds=[quads[0]], lightSphPt=[sph_pt[0]], lightSphR=[sph_r[0]])


def test_generated_bvh_scene_matches_per_sample_reference(b2pt):
    w, h = 48, 40
    s = generated_scene(b2pt)
    g = 3.0
    views = np.stack([
        view_row([g, g, -6.0], [g, g, g], (0, 1, 0), 60.0),
        view_row([-4.0, 8.0, -3.5], [g, g, g], (0.2, 1.0, 0.0), 55.0),
        view_row([g + 0.1, g - 0.2, g + 0.3], [0.5, 5.5, 0.5], (0, 0, 1), 90.0),  # inside the grid
    ])
    ck = (1, 3, 4)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(s)
        alb, nd = ctx.render_views_features(views, w, h, ck, b2pt.FLAG_FORCE_BVH)
        ra, rn = reference(ctx, b2pt, s, views, w, h, ck)
        prims = set()
        for row in views:
            ctx.set_camera(camera(b2pt, row, w, h))
            prims |= set(np.unique(sample_features(ctx, s, w * h, 0, 0)[2]).tolist())
    assert same_bits(alb, ra) and same_bits(nd, rn)
    n_quads = len(s.quadIds)
    assert len(prims) > 60 and any(p >= n_quads for p in prims)  # many quads and at least one sphere
    kinds = s.matType[s.matIdxQ]
    assert set(kinds.tolist()) == {0, 1, 2}


def test_glass_sphere_shows_up(cornell, b2pt):
    """The camera of test_gpu_primary aimed at Cornell's glass sphere: the pixels whose samples all hit the sphere
    carry albedo (1,1,1) and the sphere's normals (p - c) / r; the -direct G-buffers of the same view have no sphere."""
    ctx, scene = cornell
    w = h = 64
    view = view_row([-1.5, 0.2, 0.5], [-0.6, 0.16, 0.52], (0, 1, 0), 30.0)[None]
    ck = (1, 4)
    alb, nd = ctx.render_views_features(view, w, h, ck)
    ra, rn = reference(ctx, b2pt, scene, view, w, h, ck)
    assert same_bits(alb, ra) and same_bits(nd, rn)
    sphere = len(scene.quadIds)  # the first sphere's primitive id
    assert scene.matType[scene.matIdxS[0]] == 2  # dielectric
    ctx.set_camera(camera(b2pt, view[0], w, h))
    all_sphere = np.ones(w * h, bool)
    centre = scene.pts[scene.sphPt[0]]
    for s in range(ck[-1]):
        _, _, prim, rec = sample_features(ctx, scene, w * h, 0, s)
        on = prim == sphere
        all_sphere &= on
        p = rec[6:9].T[on]
        assert same_bits(rec[3:6].T[on], (p - centre) / scene.sphR[0])
    assert all_sphere.sum() > 20
    assert np.array_equal(alb[-1, 0][all_sphere], np.full((all_sphere.sum(), 4), 4, np.float32))
    mean_n = nd[-1, 0][all_sphere][:, :3] / 4
    assert (np.abs(np.linalg.norm(mean_n, axis=1) - 1) < 0.05).mean() > 0.9
    _, _, _, dprim = ctx.render_direct_views(view, w, h)
    assert not (dprim == sphere).any()


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
        full = ctx.render_views_checkpoints(views, w, h, ck, depth)
        st = ctx.stats()
        ptr = L.b2pt_views_device_ptr(ctx._h)
        assert ptr
        alb, nd = ctx.render_views_features(views, w, h, ck)
        ctx.render_views_features(views, w, h, ck, b2pt.FLAG_FORCE_BVH | b2pt.FLAG_WIDE_BVH)  # rebuilds, renders nothing

        def fails(message, *args, **kw):
            with pytest.raises(b2pt.B2ptError, match=message) as e:
                ctx.render_views_features(*args, **kw)
            assert e.value.code == b2pt.ERR_BAD_VALUE

        fails(r"nCheckpoints must be in \[1,32\]", views, w, h, ())
        fails(r"nCheckpoints must be in \[1,32\]", views, w, h, range(1, 34))
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (0, 2))
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (2, 2))
        fails("checkpoints must be >= 1 and strictly increasing", views, w, h, (3, 2))
        fails(r"more than 2\^24 samples", views, w, h, (1, (1 << 24) + 1))
        for f in (b2pt.FLAG_REFERENCE_STREAM, b2pt.FLAG_VIEWS_NORMALIZE, b2pt.FLAG_NO_TAIL, 1 << 20):
            fails("flags may only hold FORCE_BVH, NO_DEDUP, NO_AA, GPU_LBVH and WIDE_BVH", views, w, h, ck, f)
        bad = views.copy()
        bad[2, 9] = 0.0
        fails("feild of view must be greater than zero", bad, w, h, ck)
        fails("width must be greater than zero", views, 0, h, ck)
        vp, two = p(views), np.array([1, 2], np.int32)
        assert L.b2pt_render_views_features(ctx._h, 4, vp, w, h, 2, None, 0, None, None) == b2pt.ERR_BAD_VALUE
        assert b"nCheckpoints must be in [1,32]" in L.b2pt_last_error()
        assert L.b2pt_render_views_features(ctx._h, 4, None, w, h, 2, p(two), 0, None, None) == b2pt.ERR_BAD_VALUE
        assert b"bad view list" in L.b2pt_last_error()
        assert L.b2pt_render_views_features(ctx._h, -1, vp, w, h, 2, p(two), 0, None, None) == b2pt.ERR_BAD_VALUE
        # one 8192^2 view (2^26 pixels) in 17 slices is more than 2^30 float4; 16 slices are not (not run here)
        big = np.arange(1, 18, dtype=np.int32)
        assert L.b2pt_render_views_features(ctx._h, 1, vp, 8192, 8192, 17, p(big), 0, None, None) == b2pt.ERR_BAD_VALUE
        assert b"exceed 2^30 float4" in L.b2pt_last_error()
        # NULL outputs: any combination gives the same bits
        c3 = np.array(ck, np.int32)
        assert L.b2pt_render_views_features(ctx._h, 4, vp, w, h, 3, p(c3), 0, None, None) == 0
        only_a, only_nd = np.zeros_like(alb), np.zeros_like(nd)
        assert L.b2pt_render_views_features(ctx._h, 4, vp, w, h, 3, p(c3), 0, p(only_a), None) == 0
        assert L.b2pt_render_views_features(ctx._h, 4, vp, w, h, 3, p(c3), 0, None, p(only_nd)) == 0
        assert same_bits(only_a, alb) and same_bits(only_nd, nd)
        # nViews == 0
        ea, en = ctx.render_views_features(np.zeros((0, 10), np.float32), w, h, ck)
        assert ea.shape == (3, 0, n, 4) and en.shape == (3, 0, n, 4)
        # nothing was rendered: same statistics, same view image pointer
        st2 = ctx.stats()
        assert (st2.paths, st2.launches, st2.batches, st2.segments, st2.tracePath) == \
            (st.paths, st.launches, st.batches, st.segments, st.tracePath)
        assert L.b2pt_views_device_ptr(ctx._h) == ptr
        # the context's own camera and canvas are untouched
        assert same_bits(ctx.read_color(), canvas)
        after = ctx.primary_hits()
        assert np.array_equal(after[0], hits[0]) and same_bits(after[1], hits[1])
        # the library-owned view images still hold the last checkpoint
        ctx.set_camera(b2pt.Camera(w, h))
        for v in range(len(views)):
            assert L.b2pt_set_color_buffer(ctx._h, ctypes.c_void_p(ptr + v * n * 16)) == 0
            assert same_bits(ctx.read_color(), full[-1][v]), v
        assert L.b2pt_set_color_buffer(ctx._h, None) == 0
    with b2pt.Context(0) as ctx:  # no scene
        with pytest.raises(b2pt.B2ptError) as e:
            ctx.render_views_features(views, w, h, ck)
        assert e.value.code == b2pt.ERR_STATE


# ---- the driver: -hemisphere -features / -fibonacci -features
def hemisphere_positions(n_phi, n_theta):
    """generateHemisphere's view points as host/main.cc computes them (float32 arithmetic, cos/sin rounded to float)."""
    f = np.float32
    theta_end = f(2 * 3.14159265358979323846)
    r_theta = f(theta_end / f(n_theta))
    r_phi = f(f(1.0) / f(n_phi))
    r = f(-1078 / 555.0)
    out = []
    phi = f(0)
    while float(phi) < 1.0 - 0.5 * float(r_phi):
        theta = f(0)
        while theta < theta_end:
            ct, st = f(math.cos(float(theta))), f(math.sin(float(theta)))
            sp, cp = f(math.sin(float(phi))), f(math.cos(float(phi)))
            x, y, z = f(f(r * ct) * sp), f(f(r * st) * sp), f(r * cp)
            out.append([f(float(x) + C), f(float(y) + C), f(float(z) + C)])
            theta = f(theta + r_theta)
        phi = f(phi + r_phi)
    return out


def fibonacci_positions(n):
    """fibonacciHemisphere's view points with -viewseed 0 (float z and radius, double azimuth), z < 0 only."""
    offset = np.float32(2.0 / n)
    inc = math.pi * (3.0 - math.sqrt(5.0))
    out = []
    for i in range(n):
        z = np.float32(np.float32(np.float32(i * offset) - np.float32(1)) + np.float32(offset / np.float32(2)))
        rad = np.float32(math.sqrt(1 - float(z) ** 2))
        phi = (i % n) * inc
        x, y = np.float32(math.cos(phi) * float(rad)), np.float32(math.sin(phi) * float(rad))
        if z < 0:
            out.append([np.float32(float(x) + C), np.float32(float(y) + C), np.float32(float(z) + C)])
    return out


def read_pfm(path, w, h, channels):
    data = open(path, "rb").read()
    header = ("PF" if channels == 3 else "Pf") + "\n%d %d\n-1.0\n" % (w, h)
    assert data[:len(header)] == header.encode(), path
    payload = np.frombuffer(data[len(header):], "<f4")
    assert payload.size == w * h * channels, path
    return payload


@pytest.mark.parametrize("sweep", ["hemisphere", "fibonacci"])
@pytest.mark.parametrize("checkpoints", [None, "2,4"])
def test_driver_features(b2pt, host_build, tmp_path, sweep, checkpoints):
    exe = os.path.join(host_build, "CornellBox_b2pt")
    w, h, spp = 24, 16, 6
    args = ["-hemisphere", "-phicount", "2", "-thetacount", "3"] if sweep == "hemisphere" else \
        ["-fibonacci", "-viewcount", "12"]
    if checkpoints:
        args += ["-checkpoints", checkpoints]

    def run(name, *extra):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe, "-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", str(spp)] + args +
                             list(extra), cwd=d, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        assert "views rendered       = 6" in out.stdout
        return d, sorted(os.listdir(d))

    fdir, files = run("features", "-features")
    pdir, plain = run("plain")
    assert len(plain) == 6 * (3 if checkpoints else 1)
    for f in plain:  # the radiance files: byte-identical to a run without -features
        assert open(fdir / f, "rb").read() == open(pdir / f, "rb").read(), f
    tails = sorted(f[len("output-"):-len(".pnm")] for f in plain if not f.startswith("output-s"))
    counts = [int(c) for c in checkpoints.split(",")] + [spp] if checkpoints else [spp]
    stems = ["output-s%d" % c for c in counts[:-1]] + ["output"]
    want = sorted(plain + ["%s-%s-%s.pfm" % (s, b, t) for s in stems for b in ("albedo", "normal", "depth")
                           for t in tails])
    assert files == want

    positions = hemisphere_positions(2, 3) if sweep == "hemisphere" else fibonacci_positions(12)
    views = np.stack([view_row(pos) for pos in positions])
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        alb, nd = ctx.render_views_features(views, w, h, counts)
    order = driver_view_names(sweep, positions)
    assert sorted(order) == tails
    for k, (c, stem) in enumerate(zip(counts, stems)):
        cf = np.float32(c)
        for v, tail in enumerate(order):
            a, q = alb[k, v], nd[k, v]
            want_a = (a[:, :3] / cf).reshape(-1)
            want_n = (q[:, :3] / cf).reshape(-1)
            with np.errstate(invalid="ignore", divide="ignore"):
                want_d = np.where(a[:, 3] > 0, q[:, 3] / a[:, 3], np.float32(0)).astype(np.float32)
            assert same_bits(read_pfm(fdir / ("%s-albedo-%s.pfm" % (stem, tail)), w, h, 3), want_a), (stem, tail)
            assert same_bits(read_pfm(fdir / ("%s-normal-%s.pfm" % (stem, tail)), w, h, 3), want_n), (stem, tail)
            assert same_bits(read_pfm(fdir / ("%s-depth-%s.pfm" % (stem, tail)), w, h, 1), want_d), (stem, tail)
    assert alb[-1][..., 3].max() == spp and np.abs(nd[-1][..., :3]).max() > 0


def driver_view_names(sweep, positions):
    """The <phi>-<theta> part of the driver's file names, in its view order."""
    if sweep == "fibonacci":
        return ["0.0000-%d.0000" % i for i in range(len(positions))]
    f = np.float32
    theta_end = f(2 * 3.14159265358979323846)
    r_theta, r_phi = f(theta_end / f(3)), f(f(1.0) / f(2))
    out = []
    phi = f(0)
    while float(phi) < 1.0 - 0.5 * float(r_phi):
        theta = f(0)
        while theta < theta_end:
            out.append("%.4f-%.4f" % (phi, theta))
            theta = f(theta + r_theta)
        phi = f(phi + r_phi)
    return out
