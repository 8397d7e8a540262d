"""The thin lens of b2pt_set_lens restated on top of the C oracle (tests/lens_ref.c; include/b2pt.h, DESIGN.md 8h),
checked without a GPU: lens origins lie on the lens disk, every lens ray passes through the point where the pinhole ray
meets the plane of focus, each ray consumes 2 + 2k draws, the disk is sampled uniformly, and aperture 0 is the oracle's
pinhole bit for bit (rays, draws, primary hits and the committed oracle renders)."""
import os
import sys

import numpy as np
import pytest
from scipy import stats

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import lens_ref  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
C = 278 / 555.0


def cameras(oracle):
    """The default Cornell camera and two off-axis views with tilted up vectors and other canvases."""
    return [
        oracle.Camera(64, 48),
        oracle.Camera(33, 17, pos=(C + 0.7, C + 0.4, C - 1.6), up=(0.2, 1, 0.1), fov=55.0),
        oracle.Camera(40, 40, pos=(C - 1.2, C - 0.3, C - 1.1), lookAt=(C, C + 0.1, C + 0.2), up=(0, 0.9, 0.3),
                      fov=30.0),
    ]


def focus_of(cam, focus):
    if focus > 0:
        return focus
    return float(np.linalg.norm(cam.lookAt.astype(np.float64) - cam.pos.astype(np.float64)))


@pytest.mark.parametrize("aperture,focus", [(0.05, 0.0), (0.3, 0.0), (0.2, 1.1), (1.0, 3.0)])
def test_lens_rays_geometry_and_draws(oracle, aperture, focus):
    rng = np.random.default_rng(7)
    for cam in cameras(oracle):
        nlook, dx, dy = (x.astype(np.float64) for x in cam.basis())
        pos = cam.pos.astype(np.float64)
        r, f = aperture / 2.0, focus_of(cam, focus)
        n = cam.W * cam.H
        for _ in range(300):
            p = int(rng.integers(n))
            seed = int(rng.integers(1 << 32))
            o, d, state, draws = lens_ref.raygen(cam, aperture, focus, p, seed)
            o, d = o.astype(np.float64), d.astype(np.float64)
            # the origin lies on the lens disk: in the plane through pos normal to nlook, within r of pos
            assert abs(np.dot(o - pos, nlook)) <= 1e-6
            assert np.linalg.norm(o - pos) <= r * (1 + 1e-6) + 1e-7
            # the ray passes through F, where the pinhole ray of the same jitter meets the plane of focus
            d0, s0 = oracle.raygen(cam, p, seed)
            d0 = d0.astype(np.float64)
            F = pos + d0 * (f / np.dot(d0, nlook))
            off = F - o
            assert np.linalg.norm(off - np.dot(off, d) * d) <= 1e-5 * f
            assert abs(np.linalg.norm(d) - 1) < 1e-6
            # 2 jitter draws, then k >= 1 pairs; the state is the chain after exactly that many draws
            assert draws >= 4 and draws % 2 == 0 and draws <= 2 + 32
            assert oracle.wang_chain(seed, draws)[-1] == state
            assert oracle.wang_chain(seed, 2)[-1] == s0


def test_rejected_pairs_are_drawn_again(oracle):
    """Some streams reject their first pairs: k counts every pair drawn, and the accepted pair is the first inside."""
    cam = oracle.Camera(16, 16)
    seen = set()
    for seed in range(2000):
        _, _, state, draws = lens_ref.raygen(cam, 0.5, 0.0, 5, seed)
        k = (draws - 2) // 2
        seen.add(k)
        u = oracle.randf_chain(seed, draws)
        pairs = [(2 * np.float32(u[2 + 2 * j]) - np.float32(1), 2 * np.float32(u[3 + 2 * j]) - np.float32(1))
                 for j in range(k)]
        inside = [np.float32(a * a) + np.float32(b * b) < 1 for a, b in pairs]
        assert inside[-1] and not any(inside[:-1])
    assert {1, 2, 3} <= seen


def test_aperture_zero_is_the_pinhole(oracle):
    for cam in cameras(oracle):
        for p in (0, 7, cam.W * cam.H - 1):
            for seed in (0, 12345, 0xFFFFFFFF):
                o, d, state, draws = lens_ref.raygen(cam, 0.0, 0.8, p, seed)
                d0, s0 = oracle.raygen(cam, p, seed)
                assert draws == 2 and state == s0
                assert np.array_equal(d.view(np.uint32), d0.view(np.uint32))
                assert np.array_equal(o.view(np.uint32), cam.pos.view(np.uint32))


def test_disk_is_uniform(oracle):
    """1e5 lens origins of one pixel over consecutive streams: chi-square on 10 bins of a^2 + b^2 (uniform on a
    uniform disk) and on 10 bins of the angle."""
    aperture = 1.0
    cam = oracle.Camera(8, 8)
    _, dx, dy = (x.astype(np.float64) for x in cam.basis())
    u, v = dx / np.linalg.norm(dx), dy / np.linalg.norm(dy)
    pos = cam.pos.astype(np.float64)
    n = 100000
    ab = np.zeros((n, 2))
    for s in range(n):
        o, _, _, _ = lens_ref.raygen(cam, aperture, 0.0, 27, 0x1234567 + s * 0x9E3779B9 & 0xFFFFFFFF)
        e = o.astype(np.float64) - pos
        ab[s] = (np.dot(e, u) / (aperture / 2), np.dot(e, v) / (aperture / 2))
    rho2 = np.clip((ab ** 2).sum(1), 0, 1 - 1e-12)
    ang = np.arctan2(ab[:, 1], ab[:, 0])
    h1 = np.histogram(rho2, bins=10, range=(0, 1))[0]
    h2 = np.histogram(ang, bins=10, range=(-np.pi, np.pi))[0]
    assert h1.sum() == n and h2.sum() == n
    assert stats.chisquare(h1).pvalue > 1e-3, h1
    assert stats.chisquare(h2).pvalue > 1e-3, h2


def test_aperture_zero_is_todays_oracle(oracle):
    """With a zero aperture, whatever the focus distance, the restatement is the oracle's pinhole: the committed
    production-stream render (128^2, 10 spp, depth 5) with its segment count, and the primary hits."""
    sc = oracle.cornell_scene()
    cam = oracle.Camera(128, 128)
    img, st = lens_ref.render(sc, cam, 0.0, 0.9, 10, 5)
    assert np.array_equal(img[:, :3], np.load(os.path.join(GOLD, "config1_fast_rgb.npy")), equal_nan=True)
    want, wst = oracle.render(sc, cam, 10, 5, mode=oracle.MODE_FORWARD_FAST)
    assert np.array_equal(img, want, equal_nan=True)
    assert (st.segments, st.rngDraws, st.nanSamples) == (wst.segments, wst.rngDraws, wst.nanSamples)
    for seed in (0, 9):
        got, want = lens_ref.primary_hits(sc, cam, 0.0, 0.9, seed), oracle.primary_hits(sc, cam, seed)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))


def test_lens_render_and_hits_follow_the_lens_rays(oracle):
    """Under a lens: the render differs from the pinhole's, sample ranges are independent streams, and the primary hits
    are the oracle's closest hits of the restated lens rays (t from the lens origin)."""
    sc = oracle.cornell_scene()
    cam = oracle.Camera(32, 32)
    img, st = lens_ref.render(sc, cam, 0.1, 0.0, 3, 4, seed_offset=5)
    pinhole, pst = oracle.render(sc, cam, 3, 4, mode=oracle.MODE_FORWARD_FAST, seed_offset=5)
    assert not np.array_equal(img, pinhole)
    assert st.paths == pst.paths and st.aliveAtDepth[0] == 32 * 32 * 3
    a, _ = lens_ref.render(sc, cam, 0.1, 0.0, 1, 4, seed_offset=5)
    b, _ = lens_ref.render(sc, cam, 0.1, 0.0, 2, 4, sample_begin=1, seed_offset=5)
    ok = ~np.isnan(img)
    assert np.allclose((a + b)[ok], img[ok], rtol=1e-5, atol=1e-6)
    prim, t = lens_ref.primary_hits(sc, cam, 0.1, 0.0, seed_offset=3)
    for p in (0, 100, 517, 1023):
        o, d, _, _ = lens_ref.raygen(cam, 0.1, 0.0, p, p + 3)
        want, rec, _ = oracle.closest_hit(sc, o, d)
        assert prim[p] == want
        assert t[p] == (rec[2] if want >= 0 else np.finfo(np.float32).max)
