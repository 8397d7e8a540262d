"""b2pt_denoise_views_temporal and b2pt_temporal_defaults are part of the C-ABI (declared in include/b2pt.h, exported by
libb2pt.so, bound in SIGNATURES and by Context.denoise_views_temporal), the defaults are the documented values, the
driver rejects bad -temporal uses before it touches a GPU, and the restatement (tests/temporal_ref.py) holds its own
invariants (no GPU needed)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_ref as R  # noqa: E402
import temporal_ref as T  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
C = 278 / 555.0
f = np.float32


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


def test_symbols_are_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_denoise_views_temporal\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,\s*"
                     r"const\s+float\s*\*\s*views\s*,", hdr)
    assert re.search(r"\bvoid\s+b2pt_temporal_defaults\s*\(\s*b2pt_temporal_params\s*\*\s*p\s*\)", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    for name in ("b2pt_denoise_views_temporal", "b2pt_temporal_defaults"):
        assert any(l.split()[-1] == name and " T " in l for l in out.splitlines()), name
        assert name in b2pt.SIGNATURES
    assert len(b2pt.SIGNATURES["b2pt_denoise_views_temporal"][1]) == 17
    assert callable(getattr(b2pt.Context, "denoise_views_temporal", None))


def test_defaults(b2pt):
    p = b2pt.TemporalParams.defaults()
    assert (p.alpha, p.minVisible, p.normalTol, p.albedoTol, p.depthTol) == \
        (f(0.1), f(0.5), f(0.3), f(0.03), f(0.05))
    assert T.DEFAULTS == dict(alpha=0.1, min_visible=0.5, normal_tol=0.3, albedo_tol=0.03, depth_tol=0.05)


@pytest.mark.parametrize("args, message", [
    (["-hemisphere", "-direct", "-temporal"], "-temporal cannot be combined with -direct"),
    (["-temporal", "-direct"], "-temporal cannot be combined with -direct"),
    (["-temporal"], "-temporal needs -hemisphere"),
    (["-fibonacci", "-temporal"], "-temporal cannot be combined with -fibonacci"),
    (["-hemisphere", "-fibonacci", "-temporal"], "-temporal cannot be combined with -fibonacci"),
    (["-hemisphere", "-checkpoints", "2", "-adaptive", "0.1", "-temporal"],
     "-temporal cannot be combined with -adaptive or -adaptive-denoise"),
    (["-hemisphere", "-checkpoints", "2", "-adaptive-denoise", "0.1", "-temporal"],
     "-temporal cannot be combined with -adaptive or -adaptive-denoise"),
])
def test_driver_rejects_bad_temporal(host_build, tmp_path, args, message):
    out = subprocess.run([os.path.join(host_build, "CornellBox_b2pt"), "-x", "8", "-y", "8", "-samplecount", "6"] + args,
                         cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert out.returncode == 1, out.stdout + out.stderr
    assert message in out.stderr
    assert os.listdir(tmp_path) == []


# ---- the restatement's own invariants, on synthetic sums of a static camera (identical views, zero motion) ----------
W, H = 12, 9


def still_sweep(V, K=2, seed=0):
    """V identical views of a box seen head on: noisy colour sums, one plane of guides at the depth a pixel-centre ray
    of the camera travels to z = 1 (so the depth test passes), every sample valid and visible, zero motion."""
    rng = np.random.default_rng(seed)
    ck = np.array([2, 5][:K], np.int32)
    row = np.array([C, C, -800 / 555.0, C, C, C, 0, 1, 0, 40], f)
    views = np.stack([row] * V)
    N = W * H
    d = T.centre_directions(row, W, H)
    depth = (f(1) - row[2]) / d[:, 2]
    S = np.zeros((K, V, N, 4), f)
    Q, A, ND, M = (np.zeros_like(S) for _ in range(4))
    for k, c in enumerate(ck):
        samples = rng.exponential(1.0, (V, N, c, 3)).astype(f)
        S[k, ..., :3] = samples.sum(2)
        Q[k, ..., :3] = (samples ** 2).sum(2)
        A[k, ..., :3] = 0.5 * c
        A[k, ..., 3] = c
        ND[k, ..., 2] = -c
        ND[k, ..., 3] = depth * c
        M[k, ..., 2] = c
        M[k, ..., 3] = c
    return ck, views, S, Q, A, ND, M


def test_alpha_one_is_the_prep():
    ck, views, S, Q, A, ND, M = still_sweep(4)
    x, V, n = T.temporal(S, Q, A, ND, M, views, W, H, ck, alpha=1.0)
    m, V0, *_ = R.prep(S, Q, A, ND, ck)
    assert np.array_equal(x.view(np.uint32), m.view(np.uint32))
    assert np.array_equal(V.view(np.uint32), V0.view(np.uint32))
    assert (n == 1).all()


def test_history_grows_by_one_per_view_under_zero_motion():
    ck, views, S, Q, A, ND, M = still_sweep(6)
    x, V, n = T.temporal(S, Q, A, ND, M, views, W, H, ck, alpha=0.01)
    for v in range(6):
        assert (n[:, v] == v + 1).all(), v
    # with alpha below 1/n the blend is the running mean of the views' means
    m, V0, *_ = R.prep(S, Q, A, ND, ck)
    assert np.allclose(x[:, -1], m.mean(1), rtol=1e-5)
    assert np.allclose(V[:, -1], V0.sum(1) / 36, rtol=1e-4)


@pytest.mark.parametrize("case", ["nan", "nan-sum", "off-canvas", "huge", "no-valid", "hidden"])
def test_no_history(case):
    ck, views, S, Q, A, ND, M = still_sweep(3)
    if case == "nan":
        M[:, 1:, ::3, 0] = np.nan
    elif case == "nan-sum":
        M[:, 1:, ::3, 2] = np.nan
    elif case == "off-canvas":
        M[:, 1:, ::3, 0] = 2.0 * W * M[:, 1:, ::3, 3]
    elif case == "huge":
        M[:, 1:, ::3, 1] = 1e30
    elif case == "no-valid":
        M[:, 1:, ::3] = 0
    else:  # visible fraction below minVisible
        M[:, 1:, ::3, 2] = np.floor(0.4 * M[:, 1:, ::3, 3])
    x, V, n = T.temporal(S, Q, A, ND, M, views, W, H, ck)
    m, V0, *_ = R.prep(S, Q, A, ND, ck)
    sel = np.zeros(W * H, bool)
    sel[::3] = True
    assert (n[:, 1:, sel] == 1).all() and (n[:, 1:, ~sel] > 1).all()
    assert np.array_equal(x[:, 1:, sel], m[:, 1:, sel]) and np.array_equal(V[:, 1:, sel], V0[:, 1:, sel])


def test_a_tap_at_zero_fraction_carries_no_weight():
    """Exact-integer motion of one pixel to the left: the tap at fu = 0 is the only one with weight, so the column
    after it and the row above it do not matter."""
    ck, views, S, Q, A, ND, M = still_sweep(2)
    M[:, 1, :, 0] = -M[:, 1, :, 3]
    M[:, 1, :, 1] = 0
    x, V, n = T.temporal(S, Q, A, ND, M, views, W, H, ck)
    S2 = S.copy()
    S2[:, 0, :, :3] *= 3  # change view 0 everywhere, then compare per pixel with the shifted source
    x2, _, _ = T.temporal(S2, Q, A, ND, M, views, W, H, ck)
    assert not np.array_equal(x[:, 1], x2[:, 1])
    # the result at (i, j) depends on view 0 at (i - 1, j) only: poison every other pixel of view 0's colour
    j, i = np.divmod(np.arange(W * H), W)
    for col in range(1, W):
        S3 = S.copy()
        keep = (i == col - 1)
        S3[:, 0, ~keep, :3] = 1e6
        x3, _, _ = T.temporal(S3, Q, A, ND, M, views, W, H, ck)
        at = np.nonzero(i == col)[0]
        assert np.array_equal(x3[:, 1, at], x[:, 1, at]), col
    assert (n[:, 1][:, i == 0] == 1).all() and (n[:, 1][:, i > 0] == 2).all()  # column 0 maps off the canvas
