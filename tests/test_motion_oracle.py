"""The motion vectors of b2pt_render_views_motion restated on top of the C oracle (tests/motion_ref.c; include/b2pt.h,
DESIGN.md 8i), checked without a GPU: the projection of a sample's hit gives back its jittered pixel coordinate,
identical cameras give exactly zero motion, a sideways translation gives the pinhole's parallax, a camera the tall box
blocks sees both visible and occluded back-wall points, a rotated camera sends some points off the canvas, and the sums
are the per-sample values added in sample order."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import motion_ref  # noqa: E402

C = 278 / 555.0
W = H = 48
FOV = 40.0


def camera(oracle, pos=(C, C, -800 / 555.0), look=(C, C, C), fov=FOV):
    return oracle.Camera(W, H, pos=pos, lookAt=look, fov=fov)


def shifted(oracle, cam, delta):
    """cam translated by delta along its own right axis (dx / |dx|), look-at point too."""
    _, dx, _ = cam.basis()
    u = dx.astype(np.float64) / np.linalg.norm(dx.astype(np.float64))
    return oracle.Camera(cam.W, cam.H, pos=cam.pos + delta * u, lookAt=cam.lookAt + delta * u, up=cam.up, fov=cam.fov)


def samples(oracle, cam, prev, n=1, seed_offset=0):
    """Sample s < n of every pixel: list of (pixel, s, valid, values)."""
    osc = oracle.cornell_scene()
    out = []
    for p in range(cam.W * cam.H):
        for s in range(n):
            seed = (p + seed_offset + s * 0x9E3779B9) & 0xFFFFFFFF
            valid, r = motion_ref.sample(osc, cam, prev, p, seed)
            out.append((p, seed, valid, r))
    return out


def back_wall(cam, r):
    """The hit lies on the back wall (z = 1) of a camera looking along +z."""
    return abs(float(cam.pos[2]) + float(r["w"]) - 1.0) < 1e-4


def test_projection_gives_back_the_jittered_pixel(oracle):
    cams = [camera(oracle), camera(oracle, pos=(C + 0.6, C + 0.3, C - 1.7), look=(C - 0.1, C, C + 0.2), fov=55.0)]
    for cam in cams:
        hits = 0
        for p, seed, valid, r in samples(oracle, cam, cam):
            if not r["hit"]:
                continue
            hits += 1
            assert valid
            ru, rv = oracle.randf_chain(seed, 2)
            i, j = p % W, p // W
            assert abs(float(r["x"]) - (i + (1.0 - float(ru)))) < 1e-3
            assert abs(float(r["y"]) - (j + float(rv))) < 1e-3
        assert hits > 1000


def test_identical_cameras_give_zero_motion(oracle):
    osc = oracle.cornell_scene()
    for cam in (camera(oracle), camera(oracle, pos=(C - 0.5, C + 0.2, C - 1.5), fov=50.0)):
        m = motion_ref.sums(osc, cam, cam, (1, 4))
        assert np.all(m[..., :2] == 0)
        assert not np.signbit(m[..., :2]).any()
        assert np.all(m[..., 2] <= m[..., 3])
        assert np.mean(m[1, :, 2] == m[1, :, 3]) > 0.995
        # valid counts every hit: the primary hits of the restated rays
        prim, _ = oracle.primary_hits(osc, cam)
        assert np.array_equal(m[0, :, 3] > 0, prim >= 0)


@pytest.mark.parametrize("delta", [0.04, -0.07])
def test_sideways_translation_gives_pinhole_parallax(oracle, delta):
    cam = camera(oracle)
    prev = shifted(oracle, cam, delta)
    scale = W / (2 * np.tan(np.radians(FOV) / 2))
    n = 0
    for _, _, valid, r in samples(oracle, cam, prev):
        if not (valid and back_wall(cam, r)):
            continue
        n += 1
        want = -delta * scale / float(r["w"])  # w: the distance to the wall along the view axis, not t
        assert abs((float(r["xp"]) - float(r["x"])) - want) < 1e-3
        assert abs(float(r["yp"]) - float(r["y"])) < 1e-3
    assert n > 200


def test_the_tall_box_occludes_part_of_the_back_wall(oracle):
    cam = camera(oracle)
    prev = shifted(oracle, cam, -0.35)  # to the camera's left: the tall box now covers back-wall points seen from cam
    seen = hidden = 0
    for _, _, valid, r in samples(oracle, cam, prev):
        if not (valid and back_wall(cam, r)):
            continue
        on = 0 <= r["xp"] < W and 0 <= r["yp"] < H
        if on and r["visible"] == 1:
            seen += 1
        elif on:
            hidden += 1
    assert seen > 100 and hidden > 20, (seen, hidden)


def test_a_rotated_camera_sends_points_off_the_canvas(oracle):
    cam = camera(oracle)
    a = np.radians(25.0)
    d = cam.lookAt.astype(np.float64) - cam.pos.astype(np.float64)
    look = cam.pos + np.array([d[0] * np.cos(a) + d[2] * np.sin(a), d[1], -d[0] * np.sin(a) + d[2] * np.cos(a)])
    prev = camera(oracle, look=look)
    off = on = 0
    for _, _, valid, r in samples(oracle, cam, prev):
        if not valid:
            continue
        assert np.isfinite(r["xp"] - r["x"]) and np.isfinite(r["yp"] - r["y"])
        if not (0 <= r["xp"] < W and 0 <= r["yp"] < H):
            off += 1
            assert r["visible"] == 0
        else:
            on += 1
    assert off > 100 and on > 100, (off, on)


def test_sums_add_the_samples_in_order(oracle):
    osc = oracle.cornell_scene()
    cam = camera(oracle)
    prev = shifted(oracle, cam, 0.1)
    ck, seed_offset = (1, 3, 5), 7
    m = motion_ref.sums(osc, cam, prev, ck, seed_offset=seed_offset)
    want = np.zeros((len(ck), W * H, 4), np.float32)
    acc = np.zeros((W * H, 4), np.float32)
    per = samples(oracle, cam, prev, n=ck[-1], seed_offset=seed_offset)
    for idx, (p, _, valid, r) in enumerate(per):
        s = idx % ck[-1]
        if valid:
            acc[p] += np.array([r["xp"] - r["x"], r["yp"] - r["y"], r["visible"], 1], np.float32)
        if s + 1 in ck:
            want[ck.index(s + 1), p] = acc[p]
    assert np.array_equal(m.view(np.uint32), want.view(np.uint32))
    assert np.any(m[-1, :, 0] != 0)
