"""Thin-lens depth of field (b2pt_set_lens, DESIGN.md 8h) on the GPU: the pinhole is untouched after a lens was set and
removed, lens primary hits are bit-identical to the lens rays restated on the oracle (tests/lens_ref.c) on every trace
path, lens paths follow the restatement's trajectories, the sweeps keep their per-view and per-count identities under
the lens, the image shows defocus where it should and not elsewhere, bad values are rejected, and the driver's
-aperture files are the binding's."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_features import driver_view_names, hemisphere_positions, read_pfm, view_row  # noqa: E402
from test_gpu_parity import channels_within  # noqa: E402
import lens_ref  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
C = 278 / 555.0
APERTURE = 0.1


def oracle_scene(oracle, s):
    return oracle.Scene(s.pts, s.quadIds, s.sphPt, s.sphR, s.matIdxQ, s.texIdxQ, s.matIdxS, s.texIdxS, s.matType,
                        s.texType, s.tex, s.lightQuadIds, s.lightSphPt, s.lightSphR, s.lightables, s.refIdx)


def same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.reshape(-1).view(np.uint8), b.reshape(-1).view(np.uint8))


def context(b2pt, scene, build_flags=0):
    c = b2pt.Context(0)
    c.set_scene(scene)
    c.build_bvh(build_flags)
    return c


def sweep_views():
    """Four views around the box opening with tilted up vectors, other fields of view and off-centre look-at points."""
    rows = []
    for k, (dx, dy, dz) in enumerate([(0, 0, -1.9), (0.5, 0.2, -1.7), (-0.6, -0.1, -1.6), (0.2, 0.5, -1.5)]):
        look = (C + 0.05 * k, C - 0.03 * k, C + 0.1 * k)
        rows.append(view_row((C + dx, C + dy, C + dz), look, (0.05 * k, 1, 0.02 * k), 38.0 + 3 * k))
    return np.stack(rows)


def camera_of(b2pt, row, W, H):
    return b2pt.Camera(W, H, pos=row[:3], lookAt=row[3:6], up=row[6:9], fov=float(row[9]))


def snapshot(b2pt, c):
    """Every path-traced output of a context with the pinhole: render, render_views, checkpoints with moments,
    features, adaptive image and counts, and primary hits."""
    views = sweep_views()
    c.seed(5)
    c.set_camera(b2pt.Camera(64, 48))
    c.render(8, 6)
    out = [c.read_color(), *c.primary_hits()]
    out.append(c.render_views(views, 32, 32, 6, 5))
    out += list(c.render_views_checkpoints(views, 32, 32, (2, 5, 8), 5, moments=True))
    out += list(c.render_views_features(views, 32, 32, (2, 5, 8)))
    img, m2, counts, active = c.render_views_adaptive(views, 32, 32, (2, 4, 8), 5)
    return out + [img, m2, counts, active]


def test_pinhole_after_lens_is_unchanged(b2pt):
    scene = b2pt.Scene.cornell()
    with context(b2pt, scene) as fresh:
        want = snapshot(b2pt, fresh)
    with context(b2pt, scene) as c:
        c.set_lens(0.1, 0)
        c.set_camera(b2pt.Camera(64, 48))
        c.render(2, 3)
        c.set_lens(0, 0)
        got = snapshot(b2pt, c)
    assert len(got) == len(want)
    for k, (x, y) in enumerate(zip(got, want)):
        assert same(x, y), k


PRIMARY_CASES = [
    ("cornell", 0, 0.1, 1.7, 17),          # kernel-parameter path, explicit focus, seed offset
    ("cornell", 0, 0.25, 0.0, 0),          # focus at the look-at point
    ("cornell", "FORCE_BVH", 0.2, 0.0, 3),
    ("cornell", "FORCE_BVH|GPU_LBVH", 0.2, 2.0, 3),
    ("cornell", "FORCE_BVH|WIDE_BVH", 0.2, 0.0, 9),
    ("spheres", 0, 0.15, 0.0, 1),
    ("spheres", "GPU_LBVH", 0.15, 1.2, 1),
    ("spheres", "WIDE_BVH", 0.3, 0.0, 2),
]


def flags_of(b2pt, spec):
    if not spec:
        return 0
    out = 0
    for name in spec.split("|"):
        out |= getattr(b2pt, "FLAG_" + name)
    return out


@pytest.mark.parametrize("scene_name,build,aperture,focus,seed", PRIMARY_CASES)
def test_primary_hits_match_oracle(b2pt, oracle, scene_name, build, aperture, focus, seed):
    scene = b2pt.Scene.cornell() if scene_name == "cornell" else b2pt.Scene.spheres(700)
    osc = oracle.cornell_scene() if scene_name == "cornell" else oracle_scene(oracle, scene)
    row = sweep_views()[2]
    cams = [(b2pt.Camera(64, 48), oracle.Camera(64, 48)),
            (camera_of(b2pt, row, 40, 40),
             oracle.Camera(40, 40, pos=row[:3], lookAt=row[3:6], up=row[6:9], fov=float(row[9])))]
    with context(b2pt, scene, flags_of(b2pt, build)) as c:
        c.seed(seed)
        c.set_lens(aperture, focus)
        for bc, oc in cams:
            c.set_camera(bc)
            prim, t = c.primary_hits()
            oprim, ot = lens_ref.primary_hits(osc, oc, aperture, focus, seed_offset=seed)
            assert np.array_equal(prim, oprim)
            assert same(t, ot)
            c.set_lens(0, 0)
            _, tp = c.primary_hits()
            assert not same(tp, t)
            c.set_lens(aperture, focus)


@pytest.mark.parametrize("W,H,spp,depth", [(128, 128, 10, 5), (96, 64, 48, 50)])
def test_paths_match_oracle(b2pt, oracle, W, H, spp, depth):
    with context(b2pt, b2pt.Scene.cornell()) as c:
        c.set_lens(APERTURE, 0)
        c.set_camera(b2pt.Camera(W, H))
        c.render(spp, depth)
        g, st = c.read_color(), c.stats()
    o, ost = lens_ref.render(oracle.cornell_scene(), oracle.Camera(W, H), APERTURE, 0.0, spp, depth)
    assert st.segments == ost.segments
    assert st.nanSamples == ost.nanSamples
    assert channels_within(g, o, spp) > 0.9995


def test_trace_paths_tail_and_ranges_are_bit_identical(b2pt, monkeypatch):
    """Under the lens: the BVH paths equal the small-scene path, tail mode (many batches) and the other render flags
    equal a plain render, and the two halves of render_range add up to the plain render."""
    W, H, spp, depth = 96, 64, 24, 30
    scene = b2pt.Scene.cornell()

    def run(build=0, flags=0, batch_paths=0, split=None):
        if batch_paths:
            monkeypatch.setenv("B2PT_BATCH_PATHS", str(batch_paths))
        else:
            monkeypatch.delenv("B2PT_BATCH_PATHS", raising=False)
        with context(b2pt, scene, build) as c:
            c.set_lens(APERTURE, 1.9)
            c.seed(11)
            c.set_camera(b2pt.Camera(W, H))
            if split is None:
                c.render(spp, depth, flags)
            else:
                c.clear_color()
                c.render_range(0, split, depth, flags)
                c.render_range(split, spp - split, depth, flags)
            return c.read_color(), c.stats()

    base, st = run()
    assert st.tracePath == 0
    for build in (b2pt.FLAG_FORCE_BVH, b2pt.FLAG_FORCE_BVH | b2pt.FLAG_GPU_LBVH,
                  b2pt.FLAG_FORCE_BVH | b2pt.FLAG_WIDE_BVH):
        img, s = run(build=build, flags=build)
        assert s.tracePath == 1 and s.segments == st.segments
        assert same(img, base), build
    tail, s = run(batch_paths=W * H * 3)
    assert s.batches > 2 and s.tailDepth < depth
    assert same(tail, base)
    for flags in (b2pt.FLAG_NO_TAIL, b2pt.FLAG_NO_OVERLAP, b2pt.FLAG_NO_PRIMARY_MASKS, b2pt.FLAG_ONE_KERNEL_BOUNCE):
        img, _ = run(flags=flags)
        assert same(img, base), flags
    halves, _ = run(split=10)
    assert same(halves, base)


def test_reference_stream_is_rejected_under_a_lens(b2pt):
    with context(b2pt, b2pt.Scene.cornell()) as c:
        c.set_camera(b2pt.Camera(32, 32))
        c.render(2, 3, b2pt.FLAG_REFERENCE_STREAM)
        before = c.read_color()
        c.set_lens(APERTURE, 0)
        for call in (lambda: c.render(2, 3, b2pt.FLAG_REFERENCE_STREAM),
                     lambda: c.render_range(0, 2, 3, b2pt.FLAG_REFERENCE_STREAM)):
            with pytest.raises(b2pt.B2ptError) as e:
                call()
            assert e.value.code == b2pt.ERR_BAD_VALUE
        # render clears the canvas before it renders; render_range fails before it touches anything
        c.set_lens(0, 0)
        c.render(2, 3, b2pt.FLAG_REFERENCE_STREAM)
        assert same(c.read_color(), before)


def test_bad_lens_values_leave_the_lens_alone(b2pt):
    with context(b2pt, b2pt.Scene.cornell()) as c:
        c.set_camera(b2pt.Camera(48, 32))
        c.set_lens(0.2, 1.5)
        want = c.primary_hits()
        for a, f in ((float("nan"), 0), (float("inf"), 0), (-0.1, 0), (-float("inf"), 1), (0.1, float("nan")),
                     (0.1, float("inf")), (0.1, -float("inf"))):
            with pytest.raises(b2pt.B2ptError) as e:
                c.set_lens(a, f)
            assert e.value.code == b2pt.ERR_BAD_VALUE
            got = c.primary_hits()
            assert same(got[0], want[0]) and same(got[1], want[1])


def test_sweeps_under_the_lens(b2pt, monkeypatch):
    views, W, H, spp = sweep_views(), 48, 32, 8
    with context(b2pt, b2pt.Scene.cornell()) as c:
        c.seed(4)
        c.set_lens(APERTURE, 0)
        imgs = c.render_views(views, W, H, spp, 6)
        for v in range(len(views)):  # view v is set_camera(v) + render under the same lens
            c.set_camera(camera_of(b2pt, views[v], W, H))
            c.render(spp, 6)
            assert same(c.read_color(), imgs[v]), v
        ck, m2 = c.render_views_checkpoints(views, W, H, (2, 5, spp), 6, moments=True)
        for k, n in enumerate((2, 5, spp)):
            assert same(ck[k], c.render_views(views, W, H, n, 6)), n
        # one view at a time (a whole view larger than a batch): the per-view records
        monkeypatch.setenv("B2PT_BATCH_PATHS", str(W * H * spp // 2))
        assert same(c.render_views(views, W, H, spp, 6), imgs)
        monkeypatch.delenv("B2PT_BATCH_PATHS")
        # adaptive: every pixel is render_views at its own count; the denoised call's guides are the features there
        rounds = (2, 4, 8)
        p = b2pt.AdaptiveParams.defaults()
        p.threshold = 0.1
        img, _, counts, active = c.render_views_adaptive(views, W, H, rounds, 6, p)
        assert len(np.unique(counts)) > 1
        for n in rounds:
            ref = c.render_views(views, W, H, n, 6)
            sel = counts == n
            assert same(img[sel], ref[sel]), n
        img2, counts2, _, alb, nd = c.render_views_adaptive_denoised(views, W, H, rounds, 6, p, None, features=True)
        assert same(img2, img) and same(counts2, counts)
        falb, fnd = c.render_views_features(views, W, H, rounds)
        for k, n in enumerate(rounds):
            sel = counts == n
            assert same(alb[sel], falb[k][sel]) and same(nd[sel], fnd[k][sel]), n
        # the lens changes the image
        c.set_lens(0, 0)
        assert not same(c.render_views(views, W, H, spp, 6), imgs)


def feature_reference(oracle, osc, orow, W, H, nsamples, seed):
    """Sums of (albedo, hit) and (normal, t) over samples 0..n-1 of the restated lens rays, in sample order."""
    cam = oracle.Camera(W, H, pos=orow[:3], lookAt=orow[3:6], up=orow[6:9], fov=float(orow[9]))
    alb = np.zeros((W * H, 4), np.float32)
    nd = np.zeros((W * H, 4), np.float32)
    one = np.float32(1)
    for p in range(W * H):
        for s in range(nsamples):
            o, d, _, _ = lens_ref.raygen(cam, APERTURE, 0.0, p, (p + seed + s * 0x9E3779B9) & 0xFFFFFFFF)
            prim, rec, hid = oracle.closest_hit(osc, o, d)
            if prim < 0:
                continue
            kind = osc.matType[hid[0]]
            col = osc.tex[osc.texType[hid[1]]]
            a = np.ones(3, np.float32) if kind == 2 else (np.clip(col, 0, 1) if kind == 1 else col)
            alb[p] += np.array([a[0], a[1], a[2], one], np.float32)
            nd[p] += np.array([rec[3], rec[4], rec[5], rec[2]], np.float32)
    return alb, nd


@pytest.mark.parametrize("scene_name,build", [("cornell", 0), ("cornell", "FORCE_BVH|WIDE_BVH"), ("spheres", 0),
                                              ("spheres", "WIDE_BVH")])
def test_features_match_oracle_lens_rays(b2pt, oracle, scene_name, build):
    W, H, seed = 16, 12, 6
    views = sweep_views()[1:3]
    scene = b2pt.Scene.cornell() if scene_name == "cornell" else b2pt.Scene.spheres(700)
    osc = oracle.cornell_scene() if scene_name == "cornell" else oracle_scene(oracle, scene)
    with context(b2pt, scene) as c:
        c.seed(seed)
        c.set_lens(APERTURE, 0)
        alb, nd = c.render_views_features(views, W, H, (1, 3), flags_of(b2pt, build))
    for v in range(len(views)):
        for k, n in enumerate((1, 3)):
            ra, rn = feature_reference(oracle, osc, views[v], W, H, n, seed)
            assert same(alb[k, v], ra), (v, n)
            assert same(nd[k, v], rn), (v, n)


def luminance(img, spp):
    m = np.nan_to_num(img[:, :3].astype(np.float64)) / spp
    return m @ np.array([0.2126, 0.7152, 0.0722])


def test_lens_image_shows_defocus(b2pt, oracle):
    """Cornell box with the focus on the back wall: the back wall agrees with the pinhole image within the noise, and
    the edges of the boxes in front of it (out of focus) lose their sharpness."""
    W = H = 128
    spp, depth, aperture = 1024, 8, 0.2
    osc = oracle.cornell_scene()
    pts, quads = osc.pts, osc.quadIds[:, 1:]
    back = [q for q in range(len(quads)) if np.all(pts[quads[q], 2] == np.float32(555 / 555.0))]
    assert len(back) == 1
    focus = float(np.float32(1.0) - np.float32(-800 / 555.0))  # the back wall plane, along the view direction
    out = {}
    with context(b2pt, b2pt.Scene.cornell()) as c:
        c.set_camera(b2pt.Camera(W, H))
        for name, a in (("pin", 0.0), ("lens", aperture)):
            c.set_lens(a, focus)
            (img,), (m2,) = c.render_views_checkpoints(
                np.stack([view_row((C, C, -800 / 555.0))]), W, H, (spp,), depth, moments=True)
            out[name] = (img[0], m2[0])
        c.set_lens(0, 0)
        prim, t = c.primary_hits()
    ids = prim.reshape(H, W)
    # back-wall pixels at least 4 pixels away from anything else
    wall = ids == back[0]
    interior = wall.copy()
    for dy in range(-4, 5):
        for dx in range(-4, 5):
            interior &= np.roll(np.roll(wall, dy, 0), dx, 1)
    interior[:4, :] = interior[-4:, :] = interior[:, :4] = interior[:, -4:] = False
    assert interior.sum() > 1000
    lum, var = {}, {}
    for name, (img, m2) in out.items():
        mean = np.nan_to_num(img[:, :3].astype(np.float64)) / spp
        sq = np.nan_to_num(m2[:, :3].astype(np.float64)) / spp
        lum[name] = (mean @ np.array([0.2126, 0.7152, 0.0722])).reshape(H, W)
        var[name] = (np.maximum(sq - mean ** 2, 0) / (spp - 1) @ np.array([0.2126, 0.7152, 0.0722]) ** 2).reshape(H, W)
    z = (lum["lens"] - lum["pin"]) / np.sqrt(var["lens"] + var["pin"] + 1e-12)
    inside = np.abs(z[interior])
    print("back wall: %d pixels, mean |z| %.3f, share |z| < 4: %.4f" % (inside.size, inside.mean(), (inside < 4).mean()))
    # measured on a B200: 1787 pixels, mean |z| 1.088, 99.66 % below 4 (the render is deterministic)
    assert (inside < 4).mean() > 0.99 and inside.mean() < 1.25
    # edges of the foreground: neighbouring pixels whose primary hits differ, one of them much nearer than the wall
    tt = t.reshape(H, W)
    near = (ids >= 0) & (ids != back[0]) & (tt < focus - 0.4)
    edge = np.zeros_like(near)
    for ax in (0, 1):
        diff = (ids != np.roll(ids, 1, ax)) & (near | np.roll(near, 1, ax))
        edge |= diff | np.roll(diff, -1, ax)
    edge[:2, :] = edge[-2:, :] = edge[:, :2] = edge[:, -2:] = False

    def laplacian(L):
        return np.abs(4 * L - np.roll(L, 1, 0) - np.roll(L, -1, 0) - np.roll(L, 1, 1) - np.roll(L, -1, 1))
    lp, ll = laplacian(lum["pin"])[edge].mean(), laplacian(lum["lens"])[edge].mean()
    print("foreground edges: %d pixels, mean |laplacian| pinhole %.4f, lens %.4f, ratio %.3f" %
          (edge.sum(), lp, ll, ll / lp))
    assert edge.sum() > 200
    assert ll < 0.4 * lp  # measured on a B200: 2087 pixels, 0.2471 against 0.0434, ratio 0.176


def test_driver_matches_binding(b2pt, tmp_path):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    exe = os.path.join(HOST, "CornellBox_b2pt")
    w, h, spp, aperture = 24, 16, 8, 0.15
    sweep = ["-x", str(w), "-y", str(h), "-raydepth", "5", "-samplecount", str(spp), "-hemisphere", "-phicount", "2",
             "-thetacount", "3"]

    def run(name, args, rc=0):
        d = tmp_path / name
        d.mkdir()
        out = subprocess.run([exe] + args, cwd=d, capture_output=True, text=True, timeout=300)
        assert out.returncode == rc, out.stdout + out.stderr
        return d, sorted(os.listdir(d)), out.stderr

    lens, files, _ = run("lens", sweep + ["-checkpoints", "2,4", "-features", "-aperture", str(aperture)])
    adaptive, afiles, _ = run("adaptive", sweep + ["-checkpoints", "2,4", "-adaptive", "0.1", "-aperture",
                                                    str(aperture), "-focusdist", "1.8"])
    single, _, _ = run("single", ["-x", str(w), "-y", str(h), "-samplecount", str(spp), "-aperture", str(aperture)])
    plain, pfiles, _ = run("plain", sweep + ["-checkpoints", "2,4"])
    zero, zfiles, _ = run("zero", sweep + ["-checkpoints", "2,4", "-aperture", "0"])
    _, _, err = run("direct", ["-direct", "-aperture", "0.1"], rc=1)
    assert "-direct" in err
    assert zfiles == pfiles
    for f in pfiles:  # a zero aperture writes the pinhole's bytes
        assert open(zero / f, "rb").read() == open(plain / f, "rb").read(), f
    order = driver_view_names("hemisphere", hemisphere_positions(2, 3))
    views = np.stack([view_row(pos) for pos in hemisphere_positions(2, 3)])

    def body(img):
        return "P3\n%d %d 255\n" % (w, h) + "".join("%d %d %d\n" % tuple(px) for px in img)
    with context(b2pt, b2pt.Scene.cornell()) as c:
        pin = c.render_views_checkpoints(views, w, h, (2, 4, spp), 5, b2pt.FLAG_VIEWS_PNM16)
        c.set_lens(aperture, 0)
        ck = c.render_views_checkpoints(views, w, h, (2, 4, spp), 5, b2pt.FLAG_VIEWS_PNM16)
        alb, _ = c.render_views_features(views, w, h, (2, 4, spp))
        c.set_lens(aperture, 1.8)
        p = b2pt.AdaptiveParams.defaults()
        p.threshold = 0.1
        apnm, _, counts, _ = c.render_views_adaptive(views, w, h, (2, 4, spp), 5, p, b2pt.FLAG_VIEWS_PNM16)
        c.set_lens(aperture, 0)
        c.set_camera(b2pt.Camera(w, h))
        c.render(spp, 5)
        one = c.read_pnm16(spp)
    for v, tail in enumerate(order):
        for k, stem in enumerate(("output-s2", "output-s4", "output")):
            assert open(lens / ("%s-%s.pnm" % (stem, tail))).read() == body(ck[k, v]), (stem, tail)
            assert open(plain / ("%s-%s.pnm" % (stem, tail))).read() == body(pin[k, v]), (stem, tail)
        got = read_pfm(lens / ("output-albedo-%s.pfm" % tail), w, h, 3).reshape(-1, 3)
        assert np.array_equal(got, (alb[2, v][:, :3] / np.float32(spp)).astype(np.float32))
        assert open(adaptive / ("output-adaptive-%s.pnm" % tail)).read() == body(apnm[v]), tail
        assert np.array_equal(read_pfm(adaptive / ("output-spp-%s.pfm" % tail), w, h, 1), counts[v].astype(np.float32))
    assert not all(np.array_equal(ck[2, v], pin[2, v]) for v in range(len(order)))
    assert open(single / "output.pnm").read() == body(one.reshape(-1, 3))
