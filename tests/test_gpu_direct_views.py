"""-direct G-buffers of many views in one call (b2pt_render_direct_views, k_direct_views): the camera sweeps of
generateHemisphere / fibonacciHemisphere (main.cc:386-561) with -direct.

Bar: every view's normals, albedo, depth and primitive ids are BIT-IDENTICAL to b2pt_set_camera(view) +
b2pt_render_direct, whatever the split of the view list into chunks and whichever trace structure the scene is on
(small-scene path, binary BVH from either builder); and -- on Cornell and on a generated scene only the BVH path can
take -- equal to the oracle's brute-force restatement (oracle.direct)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host", "CornellBox_b2pt")
C = 278 / 555.0


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def reference_hemisphere(n_phi, n_theta):
    """generateHemisphere's view points as host/main.cc computes them (float32 arithmetic, cos/sin rounded to float):
    [(phi, theta, pos)] in the driver's order."""
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
            out.append((phi, theta, [f(float(x) + C), f(float(y) + C), f(float(z) + C)]))
            theta = f(theta + r_theta)
        phi = f(phi + r_phi)
    return out


def view_row(pos, lookAt=(C, C, C), up=(0, 1, 0), fov=40.0):
    return np.concatenate([np.asarray(pos, np.float32), np.asarray(lookAt, np.float32), np.asarray(up, np.float32),
                           [fov]]).astype(np.float32)


def sweep_views():
    """A 12-view hemisphere (3 x 4) plus a tilted up vector at fov 55, and a camera inside the box at fov 70."""
    rows = [view_row(p) for _, _, p in reference_hemisphere(3, 4)]
    rows.append(view_row([1.4, 0.9, -1.1], [0.4, 0.5, 0.5], (0.1, 1.0, 0.2), 55.0))
    rows.append(view_row([0.5, 0.5, 0.5], [0.9, 0.1, 0.9], (0, 1, 0), 70.0))
    rows.append(view_row([0.2, 0.8, -0.3], [0.6, 0.3, 0.7], (-0.3, 1.0, 0.1), 70.0))
    return np.stack(rows)


def camera(b2pt_or_oracle, v, W, H):
    return b2pt_or_oracle.Camera(W, H, pos=v[0:3], lookAt=v[3:6], up=tuple(v[6:9]), fov=float(v[9]))


def one_by_one(ctx, b2pt, views, W, H):
    outs = [[], [], [], []]
    for v in views:
        ctx.set_camera(camera(b2pt, v, W, H))
        for k, a in enumerate(ctx.render_direct()):
            outs[k].append(a)
    return [np.stack(o) for o in outs]


def assert_same(got, want, where=""):
    names = ("normals", "albedo", "depth", "prim")
    for k in range(4):
        g, w = got[k], want[k]
        if k < 3:
            g, w = bits(g), bits(w)
        assert g.shape == w.shape, (names[k], where)
        assert np.array_equal(g, w), "%s differs %s" % (names[k], where)


@pytest.mark.parametrize("W,H,which", [(128, 128, "all"), (33, 20, "all"), (128, 128, "single")])
def test_views_equal_one_view_at_a_time(gpu_ctx, b2pt, W, H, which):
    views = sweep_views() if which == "all" else sweep_views()[13:14]
    got = gpu_ctx.render_direct_views(views, W, H)
    want = one_by_one(gpu_ctx, b2pt, views, W, H)
    assert got[0].shape == (len(views), W * H, 4) and got[3].shape == (len(views), W * H)
    assert_same(got, want)
    assert (got[3] >= 0).mean() > 0.3 and (got[3] < 22).all()
    if which == "all":  # the view array is really indexed (the phi = 0 views of the hemisphere share one position)
        assert not np.array_equal(got[3][0], got[3][4]) and not np.array_equal(bits(got[2][5]), bits(got[2][6]))


def test_views_match_oracle(gpu_ctx, b2pt, oracle):
    W = H = 128
    views = sweep_views()[[6, 12, 13]]  # a hemisphere view, the tilted one, the one inside the box
    got = gpu_ctx.render_direct_views(views, W, H)
    sc = oracle.cornell_scene()
    for k, v in enumerate(views):
        on, oa, od, op = oracle.direct(sc, camera(oracle, v, W, H))
        assert_same([g[k] for g in got], (on, oa, od, op), "view %d" % k)


def test_chunk_boundary(gpu_ctx, b2pt):
    """128^2 x 300 views = 4.9 M pixels: more than one chunk of 2^22 pixels (256 views of 128^2)."""
    W = H = 128
    n = 300
    i = np.arange(n)
    z = (i + 0.5) * (1.0 / n) - 1.0  # the lower half of a Fibonacci lattice: every view sees into the box
    rad = np.sqrt(1 - z * z)
    az = i * math.pi * (3 - math.sqrt(5))
    views = np.stack([view_row([C + 1.9 * rad[k] * math.cos(az[k]) * 0.5, C + 1.9 * rad[k] * math.sin(az[k]) * 0.5,
                                C + 1.9 * z[k]]) for k in range(n)])
    got = gpu_ctx.render_direct_views(views, W, H)
    per_chunk = (1 << 22) // (W * H)
    check = sorted({0, per_chunk - 1, per_chunk, n - 1})
    want = one_by_one(gpu_ctx, b2pt, views[check], W, H)
    for j, v in enumerate(check):
        assert_same([g[v] for g in got], [w[j] for w in want], "view %d" % v)


@pytest.mark.parametrize("flags", ["FORCE_BVH", "FORCE_BVH|GPU_LBVH", "FORCE_BVH|WIDE_BVH"])
def test_bvh_path_equals_small_scene_path(gpu_ctx, b2pt, flags):
    """Direct rays on the binary BVH of either builder give the small-scene path's bits.  With the 8-wide tree the
    renders walk, direct rays still walk the binary tree it was collapsed from."""
    W = H = 128
    views = sweep_views()
    want = gpu_ctx.render_direct_views(views, W, H)
    f = 0
    for name in flags.split("|"):
        f |= getattr(b2pt, "FLAG_" + name)
    with b2pt.Context(0) as ctx:
        ctx.set_scene(b2pt.Scene.cornell())
        ctx.build_bvh(f)
        got = ctx.render_direct_views(views, W, H)
        ctx.set_camera(camera(b2pt, views[13], W, H))
        single = ctx.render_direct()
    assert_same(got, want, flags)
    assert_same(single, [w[13] for w in want], flags + " render_direct")


def generated_scene(b2pt, oracle, seed=7, n_quads=200):
    """About 200 random parallelograms, each inside its own cell of a 6^3 grid of unit cells with gaps around it (no two
    quads touch, so exact-t ties between quads of different BVH leaves cannot occur); about a third rotated arbitrarily,
    the rest axis-aligned; two made non-planar by lifting a corner.  Six spheres (four at the centres of quad cells,
    two in empty cells) that the G-buffers must never show.  Returns (b2pt scene, oracle scene)."""
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
            np.arange(n_quads) % 3, np.zeros(n_quads, np.int64), np.zeros(n_sph, np.int64), np.zeros(n_sph, np.int64),
            cb.matType, cb.texType, cb.tex)
    kw = dict(lightQuadIds=[quads[0]], lightSphPt=[sph_pt[0]], lightSphR=[sph_r[0]])
    return b2pt.Scene(*args, **kw), oracle.Scene(*args, **kw)


def test_generated_bvh_scene_matches_oracle(b2pt, oracle):
    W, H = 96, 80
    s, osc = generated_scene(b2pt, oracle)
    g = 3.0
    views = np.stack([
        view_row([g, g, -6.0], [g, g, g], (0, 1, 0), 60.0),
        view_row([-4.0, 8.0, -3.5], [g, g, g], (0.2, 1.0, 0.0), 55.0),
        view_row([9.0, 1.0, 7.5], [g, 2.5, g], (0, 1, 0), 70.0),
        view_row([g + 0.1, g - 0.2, g + 0.3], [0.5, 5.5, 0.5], (0, 0, 1), 90.0),  # inside the grid
        view_row([1.0, 1.0, 1.0], [5.0, 4.0, 6.0], (0, 1, 0), 40.0),
    ])
    with b2pt.Context(0) as ctx:
        ctx.set_scene(s)
        ctx.build_bvh()
        got = ctx.render_direct_views(views, W, H)  # 200 quads: beyond the kernel-parameter path, on the BVH
        ctx.set_camera(camera(b2pt, views[0], W, H))
        single = ctx.render_direct()
    n_quads = len(s.quadIds)
    for k, v in enumerate(views):
        want = oracle.direct(osc, camera(oracle, v, W, H))
        assert_same([a[k] for a in got], want, "view %d" % k)
        assert (got[3][k] < n_quads).all()  # never a sphere
    assert_same(single, [a[0] for a in got], "render_direct")
    hit = got[3][got[3] >= 0]
    assert len(np.unique(hit)) > 60 and np.isin([5, 11], hit).all()  # many quads, the non-planar ones included


def test_contract(gpu_ctx, b2pt):
    L = b2pt.lib()
    views = sweep_views()[:5]
    W, H = 40, 24
    gpu_ctx.set_camera(b2pt.Camera(48, 16))
    before = gpu_ctx.primary_hits()
    before_direct = gpu_ctx.render_direct()
    bad = views.copy()
    bad[3, 9] = 0.0  # Camera.cxx:720
    with pytest.raises(b2pt.B2ptError, match="feild of view must be greater than zero") as e:
        gpu_ctx.render_direct_views(bad, W, H)
    assert e.value.code == b2pt.ERR_BAD_VALUE
    with pytest.raises(b2pt.B2ptError, match="width must be greater than zero") as e:
        gpu_ctx.render_direct_views(views, 0, H)
    assert e.value.code == b2pt.ERR_BAD_VALUE
    empty = gpu_ctx.render_direct_views(np.zeros((0, 10), np.float32), W, H)
    assert [a.shape for a in empty] == [(0, W * H, 4), (0, W * H, 4), (0, W * H), (0, W * H)]
    assert L.b2pt_render_direct_views(gpu_ctx._h, -1, views.ctypes.data_as(ctypes.c_void_p), W, H, None, None, None,
                                      None) == b2pt.ERR_BAD_VALUE
    assert L.b2pt_render_direct_views(gpu_ctx._h, 2, None, W, H, None, None, None, None) == b2pt.ERR_BAD_VALUE
    # NULL outputs: any subset
    full = gpu_ctx.render_direct_views(views, W, H)
    depth = np.zeros((len(views), W * H), np.float32)
    albedo = np.zeros((len(views), W * H, 4), np.float32)
    vp = views.ctypes.data_as(ctypes.c_void_p)
    assert L.b2pt_render_direct_views(gpu_ctx._h, len(views), vp, W, H, None, None, None, None) == 0
    assert L.b2pt_render_direct_views(gpu_ctx._h, len(views), vp, W, H, None, albedo.ctypes.data_as(ctypes.c_void_p),
                                      depth.ctypes.data_as(ctypes.c_void_p), None) == 0
    assert np.array_equal(bits(depth), bits(full[2])) and np.array_equal(bits(albedo), bits(full[1]))
    # the context's own camera and canvas are untouched
    after = gpu_ctx.primary_hits()
    assert np.array_equal(before[0], after[0]) and np.array_equal(bits(before[1]), bits(after[1]))
    assert_same(gpu_ctx.render_direct(), before_direct)
    with b2pt.Context(0) as ctx:  # no scene
        with pytest.raises(b2pt.B2ptError) as e:
            ctx.render_direct_views(views, W, H)
        assert e.value.code == b2pt.ERR_STATE


# ---- the driver: -hemisphere -direct / -fibonacci -direct
def read_pnm(path, W, H):
    toks = open(path).read().split()
    assert toks[:4] == ["P3", str(W), str(H), "255"]
    return np.array(toks[4:], np.int64).reshape(-1, 3)


def save_vec4(c):  # main.cc:331-341
    c = c.copy()
    c[np.isnan(c[:, :3]).any(1)] = 0
    with np.errstate(invalid="ignore", over="ignore"):
        return np.trunc(255.99 * c[:, :3].astype(np.float64))


def assert_files_match_oracle(dirname, suffix, oracle, cam, W, H):
    on, oa, od, _ = oracle.direct(oracle.cornell_scene(), cam)
    n_img = read_pnm(os.path.join(dirname, "normals-" + suffix), W, H)
    a_img = read_pnm(os.path.join(dirname, "albedo-" + suffix), W, H)
    d_img = read_pnm(os.path.join(dirname, "depth-" + suffix), W, H)
    assert np.array_equal(n_img, save_vec4(on).astype(np.int64)), suffix
    fin = np.isfinite(save_vec4(oa)).all(1) & (np.abs(save_vec4(oa)) < 2**31 - 1).all(1)
    assert np.array_equal(a_img[fin], save_vec4(oa)[fin].astype(np.int64)), suffix
    want_d = np.trunc(255.99 * np.sqrt(od).astype(np.float32).astype(np.float64)).astype(np.int64)
    assert np.array_equal(d_img[:, 0], want_d), suffix


def test_driver_hemisphere_direct(b2pt, oracle, tmp_path):
    W, H = 40, 32
    out = subprocess.run([EXE, "-x", str(W), "-y", str(H), "-hemisphere", "-direct", "-phicount", "2", "-thetacount",
                          "3"], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "views rendered       = 6" in out.stdout
    sweep = reference_hemisphere(2, 3)
    names = ["%.4f-%.4f.pnm" % (phi, theta) for phi, theta, _ in sweep]
    want = sorted(b + "-" + n for b in ("normals", "albedo", "depth") for n in names)
    assert sorted(os.listdir(tmp_path)) == want and len(want) == 18
    for k in (0, 4):
        phi, theta, pos = sweep[k]
        assert_files_match_oracle(tmp_path, names[k], oracle, oracle.Camera(W, H, pos=pos), W, H)


def test_driver_fibonacci_direct(b2pt, tmp_path):
    out = subprocess.run([EXE, "-x", "24", "-y", "16", "-fibonacci", "-direct", "-viewcount", "12"], cwd=tmp_path,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "views rendered       = 6" in out.stdout
    want = sorted("%s-0.0000-%d.0000.pnm" % (b, i) for b in ("normals", "albedo", "depth") for i in range(6))
    assert sorted(os.listdir(tmp_path)) == want
    for f in want:
        read_pnm(os.path.join(tmp_path, f), 24, 16)
