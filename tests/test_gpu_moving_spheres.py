"""Moved spheres (b2pt_update_spheres, b2pt_refit_bvh) against the tree-free brute-force oracle, on every trace path.

A context is built once and then taken through a sequence of moves: small jitters, one sphere carried out of the
scene's original bounds (the LBVH's Morton box), a radius grown 3x and radii shrunk to 0.002 (the cancellation regime of
DESIGN.md 5), eight successive small moves and a move back to the start.  After every move each consumer of the trace
structures must see the moved scene:

* primary_hits and intersect: ids and t bit-identical to oracle.primary_hits / oracle.closest_hit on the moved scene;
* render and the view sweeps (render_views, render_views_checkpoints with moments, render_views_features,
  render_views_adaptive): bit-identical to a fresh context built on the moved scene, and the render also within 1e-4
  of the oracle's on all but a few paths;
* render_direct_views: bit-identical to oracle.direct, and to the unmoved output (-direct does not see spheres).

Call orders: update -> refit -> consumer, update -> consumer (the trace structures follow the update by themselves, and
the result equals the refitted one), two updates -> one refit, and on the 8-wide tree (which refit refuses)
update -> consumer.  The consumer that comes first after an update rotates over render, the view sweeps and primary
hits, so that both ways a trace brings the structures up to date (ensure_built_for, ensure_trace) meet a stale tree.  A move back to the original positions gives the untouched context's output bit for bit."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H, SPP, DEPTH = 64, 48, 4, 6
VW, VH = 32, 24
CHECKPOINTS = [1, 4]
ROUNDS = [2, 4, 8]
CAM_POS = np.array([278 / 555.0, 278 / 555.0, -800 / 555.0], np.float32)
FAR_POINT = np.array([0.5, 0.45, -0.3], np.float32)  # in front of the open box / the sphere field, outside both


def _oracle_scene(oracle, s):
    return oracle.Scene(s.pts, s.quadIds, s.sphPt, s.sphR, s.matIdxQ, s.texIdxQ, s.matIdxS, s.texIdxS, s.matType,
                        s.texType, s.tex, s.lightQuadIds, s.lightSphPt, s.lightSphR, s.lightables, s.refIdx)


def moved_scene(b2pt, s, centers, radii):
    """The scene b2pt_update_spheres(centers, radii) turns `s` into.  A light sphere is a scene sphere named by its
    point id: it moves with it, and its radius (the light list's own copy, lightSphR) follows the sphere's."""
    pts = s.pts.copy()
    pts[s.sphPt] = centers
    light_r = s.lightSphR.copy()
    for l, pid in enumerate(s.lightSphPt):
        owners = np.nonzero(s.sphPt == pid)[0]
        if len(owners):
            light_r[l] = radii[owners[-1]]
    return b2pt.Scene(pts, s.quadIds, s.sphPt, radii, s.matIdxQ, s.texIdxQ, s.matIdxS, s.texIdxS, s.matType, s.texType,
                      s.tex, s.lightQuadIds, s.lightSphPt, light_r, s.lightables, s.refIdx)


def view_rows():
    """The default camera (so that view 0 of -direct is oracle.direct's image) and an oblique one."""
    c = 278 / 555.0
    return np.array([[*CAM_POS, c, c, c, 0, 1, 0, 40.0],
                     [1.3, 0.8, -1.0, 0.45, 0.3, 0.5, 0.1, 1.0, 0.2, 55.0]], np.float32)


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def same(a, b):
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def sweeps(ctx, flags, views):
    """Every view-sweep consumer, with the context's build flags (other build flags would rebuild the structures)."""
    out = {"views": ctx.render_views(views, VW, VH, SPP, DEPTH, flags)}
    out["ckpt"], out["m2"] = ctx.render_views_checkpoints(views, VW, VH, CHECKPOINTS, DEPTH, flags, moments=True)
    out["albedo"], out["normal_depth"] = ctx.render_views_features(views, VW, VH, CHECKPOINTS, flags)
    for k, a in zip(("ad_image", "ad_m2", "ad_counts", "ad_active"),
                    ctx.render_views_adaptive(views, VW, VH, ROUNDS, DEPTH, None, flags)):
        out[k] = a
    return out


CONSUMERS = ("primary", "render", "views", "checkpoints", "features", "adaptive", "direct")


def consumers(ctx, b2pt, flags, views, first="primary"):
    """Every consumer of the trace structures, `first` first: after an update without a refit, that call is the one
    that meets the structures as the update left them (primary hits and -direct bring them up to date through
    ensure_trace, the renders and view sweeps through ensure_built_for)."""
    ctx.set_camera(b2pt.Camera(W, H))
    out = {}

    def primary():
        out["prim"], out["t"] = ctx.primary_hits()

    def render():
        ctx.render(SPP, DEPTH, flags)
        out["render"] = ctx.read_color().copy()
        st = ctx.stats()
        out["segments"] = np.array([st.segments, st.tracePath])

    def views_():
        out["views"] = ctx.render_views(views, VW, VH, SPP, DEPTH, flags)

    def checkpoints():
        out["ckpt"], out["m2"] = ctx.render_views_checkpoints(views, VW, VH, CHECKPOINTS, DEPTH, flags, moments=True)

    def features():
        out["albedo"], out["normal_depth"] = ctx.render_views_features(views, VW, VH, CHECKPOINTS, flags)

    def adaptive():
        for k, a in zip(("ad_image", "ad_m2", "ad_counts", "ad_active"),
                        ctx.render_views_adaptive(views, VW, VH, ROUNDS, DEPTH, None, flags)):
            out[k] = a

    def direct():
        for k, a in zip(("d_normals", "d_albedo", "d_depth", "d_prim"), ctx.render_direct_views(views, W, H)):
            out[k] = a

    calls = dict(zip(CONSUMERS, (primary, render, views_, checkpoints, features, adaptive, direct)))
    calls[first]()
    for name in CONSUMERS:
        if name != first:
            calls[name]()
    return out


def assert_same_outputs(got, want, what):
    assert got.keys() == want.keys()
    for k in want:
        assert same(got[k], want[k]), "%s: %s differs" % (what, k)


def probe_rays(oracle, ocam, centers, radii, picked, rng):
    """Camera rays; rays from the camera aimed at sphere centres and at tangent points with impact parameter
    r (1 +- 1e-6 .. 1e-3); the same tangents from an origin just in front of the sphere; rays starting inside."""
    O, D = [], []
    cam = CAM_POS.astype(np.float64)
    for p in rng.choice(W * H, 96, replace=False):
        d, _ = oracle.raygen(ocam, int(p), int(p))
        O.append(cam), D.append(d)
    for i in picked:
        c, r = centers[i].astype(np.float64), float(radii[i])
        w = (c - cam) / np.linalg.norm(c - cam)
        u = np.cross(w, rng.normal(size=3))
        u /= np.linalg.norm(u)
        O.append(cam), D.append(c - cam)
        back = max(3 * r, 0.02)
        for eps in (1e-6, 1e-5, 1e-4, 1e-3):
            for sgn in (1.0, -1.0):
                tp = c + u * r * (1 + sgn * eps)
                O.append(cam), D.append(tp - cam)
                O.append(tp - back * w), D.append(w)
        for _ in range(2):
            e, f = rng.normal(size=3), rng.normal(size=3)
            O.append(c + 0.3 * r * e / np.linalg.norm(e)), D.append(f / np.linalg.norm(f))
    return np.asarray(O, np.float32), np.asarray(D, np.float32)


def check_against_references(ctx, b2pt, oracle, base, flags, centers, radii, got, untouched, views, picked, rng,
                             what):
    s = moved_scene(b2pt, base, centers, radii)
    osc, ocam = _oracle_scene(oracle, s), oracle.Camera(W, H)
    # primary hits: brute force over every primitive, index order
    oprim, ot = oracle.primary_hits(osc, ocam)
    assert np.array_equal(got["prim"], oprim), "%s: primary ids (%d differ)" % (what, int((got["prim"] != oprim).sum()))
    assert np.array_equal(bits(got["t"]), bits(ot)), what + ": primary t"
    # intersect, ray by ray
    o, d = probe_rays(oracle, ocam, centers, radii, picked, rng)
    prim, rec, _, _ = ctx.intersect(o, d)
    for k in range(len(o)):
        p, orec, _ = oracle.closest_hit(osc, o[k], d[k])
        assert prim[k] == p, (what, "intersect ray", k, int(prim[k]), p)
        if p >= 0:
            assert rec[2, k].view(np.uint32) == np.float32(orec[2]).view(np.uint32), (what, "intersect t", k)
    # render and the view sweeps: bit-identical to a fresh context built on the moved scene (the trace paths do not
    # depend on the tree, so a stale or badly refitted one shows up here bit for bit)
    with b2pt.Context(0) as fresh:
        fresh.set_scene(s)
        fresh.build_bvh(flags)
        fresh.set_camera(b2pt.Camera(W, H))
        fresh.render(SPP, DEPTH, flags)
        st = fresh.stats()
        want = {"render": fresh.read_color().copy(), "segments": np.array([st.segments, st.tracePath])}
        want.update(sweeps(fresh, flags, views))
    assert_same_outputs({k: got[k] for k in want}, want, what + " (against a fresh context)")
    # render against the oracle's trajectories and radiance: the same segments, the same NaN masks and 1e-4 on
    # 99.95 % of the channels while no sphere is smaller than 0.003.  A 1-ulp difference between CUDA's sincosf and glibc's
    # sinf/cosf in a sampled direction now and then sends a path past a sphere of radius ~0.002 on one side and into
    # it on the other (DESIGN.md 5), a path that changes one pixel.  Measured: one segment in 15 000 after jitters of
    # the generated scenes (radii 0.001-0.003 from the generator), on the kernel-parameter path too, which has no
    # tree; one in 41 453 on the Cornell box with its sphere shrunk to 0.002, the same on all four trace paths.  There
    # the shrunk light sphere's pdf (1 - cos theta_max) also cancels, and the few ulp by which radiance-only arithmetic
    # may differ decide between a finite value and a NaN (9 channels measured); without a shrunk radius a diverging path
    # may flip one pixel's mask.  Among 20 000 spheres a handful of
    # paths diverge (test_gpu_spheres.py::test_gpu_lbvh_builder_matches_oracle).
    tiny = bool((s.sphR <= 0.003).any())
    shrunk = bool((s.sphR < base.sphR).any())
    n = len(s.sphR)
    orad, ost = oracle.render(osc, ocam, SPP, DEPTH, mode=oracle.MODE_FORWARD_FAST)
    g = got["render"][:, :3].astype(np.float64)
    ref = orad[:, :3].astype(np.float64)
    seg = int(got["segments"][0])
    if not tiny:
        seg_tol, nan_tol = 0, 0
    elif n <= 700:
        seg_tol, nan_tol = 4, (12 if shrunk else 3)
    else:
        seg_tol, nan_tol = 2e-3 * ost.segments, None
    assert abs(seg - ost.segments) <= seg_tol, (what, seg, ost.segments)
    nan_g, nan_o = np.isnan(g), np.isnan(ref)
    if nan_tol is not None:
        assert (nan_g != nan_o).sum() <= nan_tol, (what, "NaN masks", int((nan_g != nan_o).sum()))
    ok = ~(nan_g | nan_o)
    rel = np.abs(g[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), 1e-3 * SPP)
    frac = float((rel < 1e-4).mean())
    assert frac >= (0.9995 if n <= 700 else 0.99), (what, frac)
    # -direct: the oracle, and the unmoved output (it sees quads only)
    on, oa, od, op = oracle.direct(osc, ocam)
    for k, ref_k in zip(("d_normals", "d_albedo", "d_depth", "d_prim"), (on, oa, od, op)):
        assert same(got[k][0], ref_k), "%s: -direct %s differs from the oracle" % (what, k)
        assert same(got[k], untouched[k]), "%s: -direct %s changed with the spheres" % (what, k)


CASES = {
    "cornell-small": ("cornell", 0),
    "cornell-bvh": ("cornell", 0x8),
    "cornell-lbvh": ("cornell", 0x8 | 0x80),
    "cornell-wide": ("cornell", 0x8 | 0x1000),
    "spheres6-small": (6, 0),
    "spheres700-sah": (700, 0),
    "spheres700-lbvh": (700, 0x80),
    "spheres700-wide": (700, 0x8 | 0x1000),
    "spheres20000-sah": (20000, 0),
    "spheres20000-lbvh": (20000, 0x80),
}


@pytest.mark.parametrize("case", list(CASES))
def test_moved_spheres_match_oracle(b2pt, oracle, case, monkeypatch):
    monkeypatch.setenv("B2PT_VALIDATE_BVH", "1")  # every build and refit checks its boxes against the primitives
    which, flags = CASES[case]
    assert flags == flags & (b2pt.FLAG_FORCE_BVH | b2pt.FLAG_GPU_LBVH | b2pt.FLAG_WIDE_BVH)
    base = b2pt.Scene.cornell() if which == "cornell" else b2pt.Scene.spheres(which)
    wide = bool(flags & b2pt.FLAG_WIDE_BVH)
    n = len(base.sphPt)
    rng = np.random.default_rng(sum(map(ord, case)))
    c0, r0 = base.pts[base.sphPt].copy(), base.sphR.copy()
    views = view_rows()

    def jitter(c, amount):
        return (c + rng.uniform(-amount, amount, size=c.shape)).astype(np.float32)

    far = n // 2
    grown, shrunk = 0, min(1, n - 1)  # sphere 0 is a light sphere in both scenes
    c_far = c0.copy()
    c_far[far] = FAR_POINT
    r_resized = r0.copy()
    r_resized[grown] *= 3
    if shrunk != grown:
        r_resized[shrunk] = 0.002
    r_tiny = np.full_like(r0, 0.002)
    # (label, centres, radii or None (keep), order, the consumer called first after the update, spheres the intersect
    # probes aim at).  Without a refit (and on the 8-wide tree, which has none) the first consumers rotate over both
    # ways in which a trace brings the structures up to date.
    moves = [("jitter 0.003", jitter(c0, 0.003), None, "refit", "render", []),
             ("jitter 0.02", jitter(c0, 0.02), None, "twice", "checkpoints", []),
             ("one sphere out of the scene bounds", c_far, r0, "norefit", "render", [far]),
             ("radius x3 and 0.002", c_far, r_resized, "norefit", "features", [far, grown, shrunk]),
             ("every radius 0.002", c0, r_tiny, "norefit", "views", [grown])]

    with b2pt.Context(0) as ctx:
        ctx.set_scene(base)
        ctx.build_bvh(flags)
        untouched = consumers(ctx, b2pt, flags, views)
        assert untouched["segments"][1] == (1 if (flags or n > 8) else 0)  # the trace path the case names
        radii = r0
        for label, centers, new_radii, order, first, picked in moves:
            what = "%s, %s" % (case, label)
            if order == "twice":  # a first update no trace sees
                ctx.update_spheres(jitter(c0, 0.05))
            ctx.update_spheres(centers, new_radii)
            radii = radii if new_radii is None else new_radii
            if wide:
                got = consumers(ctx, b2pt, flags, views, first)
            else:
                before_refit = consumers(ctx, b2pt, flags, views, first) if order == "norefit" else None
                ctx.refit_bvh()
                got = consumers(ctx, b2pt, flags, views)
                if before_refit is not None:
                    assert_same_outputs(before_refit, got, what + " (no refit against refit)")
            picked = sorted(set(picked) | set(rng.choice(n, min(n, 16), replace=False).tolist()))
            check_against_references(ctx, b2pt, oracle, base, flags, centers, radii, got, untouched, views, picked,
                                     rng, what)
        # eight successive small moves: refitted after every other one, and primary hits first after the others; the
        # last one is left to the consumers
        centers, radii = c0.copy(), r0.copy()
        ctx.update_spheres(centers, radii)
        for step in range(8):
            centers = jitter(centers, 0.003)
            ctx.update_spheres(centers)
            if step == 7:
                break
            if not wide and step % 2 == 0:
                ctx.refit_bvh()
            prim, t = ctx.primary_hits()
            oprim, ot = oracle.primary_hits(_oracle_scene(oracle, moved_scene(b2pt, base, centers, radii)),
                                            oracle.Camera(W, H))
            assert np.array_equal(prim, oprim) and np.array_equal(bits(t), bits(ot)), (case, "small move", step)
        got = consumers(ctx, b2pt, flags, views, "adaptive")
        check_against_references(ctx, b2pt, oracle, base, flags, centers, radii, got, untouched, views,
                                 sorted(rng.choice(n, min(n, 16), replace=False).tolist()), rng,
                                 case + ", eight small moves")
        # and back, without a refit: the untouched context's output, bit for bit
        ctx.update_spheres(c0, r0)
        assert_same_outputs(consumers(ctx, b2pt, flags, views, "render"), untouched, case + ", moved back")


def test_error_contract(b2pt):
    L = b2pt.lib()

    def fails(code, text, rc):
        assert rc == code, (rc, b2pt.lib().b2pt_last_error())
        assert text in L.b2pt_last_error().decode()

    s = b2pt.Scene.spheres(100)
    c = np.ascontiguousarray(s.pts[s.sphPt])
    cp = c.ctypes.data_as(C.c_void_p)
    with b2pt.Context(0) as ctx:
        fails(b2pt.ERR_STATE, "b2pt_update_spheres before b2pt_set_scene", L.b2pt_update_spheres(ctx._h, cp, None))
        fails(b2pt.ERR_STATE, "b2pt_update_spheres before b2pt_set_scene", L.b2pt_update_spheres(ctx._h, None, None))
        fails(b2pt.ERR_STATE, "b2pt_refit_bvh before b2pt_build_bvh", L.b2pt_refit_bvh(ctx._h))
        ctx.set_scene(s)
        fails(b2pt.ERR_STATE, "b2pt_refit_bvh before b2pt_build_bvh", L.b2pt_refit_bvh(ctx._h))
        ctx.build_bvh(0)
        ctx.set_camera(b2pt.Camera(W, H))
        p0, t0 = ctx.primary_hits()
        fails(b2pt.ERR_BAD_VALUE, "null sphere centres", L.b2pt_update_spheres(ctx._h, None, None))
        fails(b2pt.ERR_BAD_VALUE, "null sphere centres",
              L.b2pt_update_spheres(ctx._h, None, s.sphR.ctypes.data_as(C.c_void_p)))
        p1, t1 = ctx.primary_hits()
        assert np.array_equal(p0, p1) and same(t0, t1)  # a refused update changes nothing
        # the 8-wide tree is rebuilt, not refitted: the refusal leaves the context tracing the moved scene
        ctx.build_bvh(b2pt.FLAG_FORCE_BVH | b2pt.FLAG_WIDE_BVH)
        moved = (c + np.float32(0.01)).astype(np.float32)
        ctx.update_spheres(moved)
        fails(b2pt.ERR_UNSUPPORTED, "b2pt_refit_bvh refits the binary tree", L.b2pt_refit_bvh(ctx._h))
        p2, t2 = ctx.primary_hits()
        with b2pt.Context(0) as fresh:
            fresh.set_scene(moved_scene(b2pt, s, moved, s.sphR))
            fresh.build_bvh(b2pt.FLAG_FORCE_BVH | b2pt.FLAG_WIDE_BVH)
            fresh.set_camera(b2pt.Camera(W, H))
            p3, t3 = fresh.primary_hits()
        assert np.array_equal(p2, p3) and same(t2, t3)
        assert not np.array_equal(p0, p2)
        ctx.build_bvh(0)
        ctx.refit_bvh()
