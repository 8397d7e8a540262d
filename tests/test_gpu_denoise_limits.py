"""The sweep denoisers at their launch and chunk limits (b2pt_denoise_views, b2pt_denoise_views_temporal,
b2pt_render_views_temporal_denoised), against tests/denoise_ref.py and tests/temporal_ref.py.

Bar: 30000 views of 2 x 2 pixels in 3 slices are 90000 images in one chunk, so each k_atrous level runs in two launches
of at most 65535 images and the second starts at image 65535, inside slice 2: every image agrees with the restatement
at one and five levels, the views on both sides of that boundary are bit for bit the view filtered alone, and the
temporal call is the restatement bit for bit at levels 0 and agrees with it at the default levels.  32 slices of
512 x 513 are more than one chunk of 2^23 float4, so every view is a chunk of its own: levels 0 is the prep bit for bit
on every slice and the default levels agree with the restatement; the temporal call, whose views take their history
from the state carried across chunks, is the restatement bit for bit at levels 0 and agrees with it at the default
levels; and the one-call render and temporal denoise is the four-call chain bit for bit."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_ref as R  # noqa: E402
import temporal_ref as T  # noqa: E402
from test_gpu_denoise import TOL_ALL, TOL_ONE, rel_err  # noqa: E402
from test_gpu_features import same_bits, view_row  # noqa: E402
from test_gpu_motion import FRONT  # noqa: E402
from test_gpu_temporal import dparams, synthetic_motion  # noqa: E402
from test_gpu_temporal_denoised import ring_views, same_as_chain  # noqa: E402

pytestmark = pytest.mark.gpu
# Slice 0 has one sample, so it has no variance and no colour term: an image filtered with another slice's count
# changes both.  2 x 2 x 3 float4 per view: all 30000 views are one chunk, and image 65535 is view 5535 of slice 2.
SPLIT_CK, SPLIT_VIEWS, SPLIT_W, SPLIT_H = (1, 5, 9), 30000, 2, 2
SPLIT_AT = 65535 - 2 * SPLIT_VIEWS
# 32 slices of 512 x 513 are 8,404,992 float4 > 2^23: one view per chunk
BIG_CK, BIG_W, BIG_H = tuple(range(1, 33)), 512, 513


def sums(ck, nv, h, w, seed):
    """Inputs of the denoisers built directly as sums over ck[k] samples (no per-sample draws): colour sums S and sums
    of squares Q >= S^2 / c with a few NaNs, and the guide sums of a plane facing FRONT, its albedo split into two blocks,
    with 5 % of the pixels missed.  Every view of FRONT sees the same guides, so the temporal step takes history."""
    rng = np.random.default_rng(seed)
    K, N = len(ck), h * w
    c = np.asarray(ck, np.float32).reshape(K, 1, 1, 1)
    S = rng.random((K, nv, N, 4), np.float32)
    S *= c
    Q = rng.random((K, nv, N, 4), np.float32)
    Q *= 2
    Q += 1
    Q *= S
    Q *= S
    Q /= c
    S.reshape(-1, 4)[::97, 0] = np.nan
    Q.reshape(-1, 4)[::89, 1] = np.nan
    hits = np.where(rng.random((K, nv, N), np.float32) < 0.05, np.float32(0), c[..., 0])
    i = np.arange(N) % w
    A = np.empty((K, nv, N, 4), np.float32)
    A[..., :3] = np.where(i < w // 2, np.float32(0.5), np.float32(0.2))[:, None] * hits[..., None]
    A[..., 3] = hits
    d = T.centre_directions(view_row(FRONT), w, h)
    ND = np.zeros((K, nv, N, 4), np.float32)
    ND[..., 2] = -hits
    ND[..., 3] = ((np.float32(1) - np.float32(FRONT[2])) / d[:, 2]) * hits
    return np.array(ck, np.int32), S, Q, A, ND


@pytest.fixture(scope="module")
def split(b2pt):
    ck, S, Q, A, ND = sums(SPLIT_CK, SPLIT_VIEWS, SPLIT_H, SPLIT_W, 1)
    M = synthetic_motion(len(ck), SPLIT_VIEWS, SPLIT_H, SPLIT_W, ck, seed=2)
    views = np.stack([view_row(FRONT)] * SPLIT_VIEWS)
    return ck, S, Q, A, ND, M, views


def test_second_atrous_launch(b2pt, split):
    ck, S, Q, A, ND, _, _ = split
    w, h = SPLIT_W, SPLIT_H
    with b2pt.Context(0) as c:
        for levels, tol in ((1, TOL_ONE), (5, TOL_ALL)):
            out = c.denoise_views(S, Q, A, ND, w, h, ck, dparams(b2pt, levels))
            x, V = R.denoise(S, Q, A, ND, w, h, ck, levels)
            assert rel_err(out[..., :3], x) < tol, levels
            assert rel_err(out[1:, ..., 3:], V[1:, ..., None]) < 10 * tol, levels  # c = 1 has no variance
            for v in (SPLIT_AT - 1, SPLIT_AT):
                one = c.denoise_views(S[:, v:v + 1], Q[:, v:v + 1], A[:, v:v + 1], ND[:, v:v + 1], w, h, ck,
                                      dparams(b2pt, levels))
                assert same_bits(one[:, 0], out[:, v]), (levels, v)


def test_second_atrous_launch_temporal(b2pt, split):
    ck, S, Q, A, ND, M, views = split
    w, h = SPLIT_W, SPLIT_H
    with b2pt.Context(0) as c:
        out, n = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, None, dparams(b2pt, 0), history=True)
        full = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck)
    x, V, hn = T.temporal(S, Q, A, ND, M, views, w, h, ck)
    assert same_bits(out[..., :3], x) and same_bits(out[..., 3], V) and same_bits(n, hn)
    assert (n[2, SPLIT_AT:] > 1).mean() > 0.1
    x, V = T.filtered(S, Q, A, ND, M, views, w, h, ck)
    assert rel_err(full[..., :3], x) < TOL_ALL
    assert rel_err(full[1:, ..., 3:], V[1:, ..., None]) < 10 * TOL_ALL


def test_one_view_per_chunk(b2pt):
    ck, S, Q, A, ND = sums(BIG_CK, 3, BIG_H, BIG_W, 3)
    w, h = BIG_W, BIG_H
    with b2pt.Context(0) as c:
        out = c.denoise_views(S, Q, A, ND, w, h, ck, dparams(b2pt, 0))
        for k in range(len(ck)):
            m, V0, *_ = R.prep(S[k:k + 1], Q[k:k + 1], A[k:k + 1], ND[k:k + 1], ck[k:k + 1])
            assert same_bits(out[k, ..., :3], m[0]) and same_bits(out[k, ..., 3], V0[0]), k
        del out
        out = c.denoise_views(S, Q, A, ND, w, h, ck)
    v = 1
    for k in (0, 1, 31):
        x, V = R.denoise(S[k:k + 1, v:v + 1], Q[k:k + 1, v:v + 1], A[k:k + 1, v:v + 1], ND[k:k + 1, v:v + 1], w, h,
                         ck[k:k + 1])
        assert rel_err(out[k:k + 1, v:v + 1, :, :3], x) < TOL_ALL, k
        if k:
            assert rel_err(out[k:k + 1, v:v + 1, :, 3:], V[..., None]) < 10 * TOL_ALL, k


def test_one_view_per_chunk_temporal(b2pt):
    """Views 1 and 2 read their history from the carry: view 1 from view 0's state, view 2 from view 1's, whose own
    history came from the carry before it."""
    ck, S, Q, A, ND = sums(BIG_CK, 3, BIG_H, BIG_W, 4)
    w, h = BIG_W, BIG_H
    M = synthetic_motion(len(ck), 3, h, w, ck, seed=5)
    views = np.stack([view_row(FRONT)] * 3)
    with b2pt.Context(0) as c:
        out, n = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck, None, dparams(b2pt, 0), history=True)
        for k in range(len(ck)):
            sl = slice(k, k + 1)
            x, V, hn = T.temporal(S[sl], Q[sl], A[sl], ND[sl], M[sl], views, w, h, ck[sl])
            assert same_bits(out[sl, ..., :3], x) and same_bits(out[sl, ..., 3], V) and same_bits(n[sl], hn), k
        assert (n[:, 1] > 1).mean() > 0.2 and (n[:, 2] > 2).mean() > 0.05
        del out, n
        out = c.denoise_views_temporal(S, Q, A, ND, M, views, w, h, ck)
    # the levels read the unfiltered history: one slice shows it (the float64 levels take 20 s a slice)
    sl = slice(31, 32)
    x, V = T.filtered(S[sl], Q[sl], A[sl], ND[sl], M[sl], views, w, h, ck[sl])
    assert rel_err(out[sl, ..., :3], x) < TOL_ALL
    assert rel_err(out[sl, ..., 3:], V[..., None]) < 10 * TOL_ALL


def test_one_view_per_chunk_render(b2pt):
    """The one call stages every view after the first from the render's device state at its own offset."""
    with b2pt.Context(0) as c:
        c.set_scene(b2pt.Scene.cornell())
        out, n, ins = same_as_chain(c, ring_views(2), BIG_W, BIG_H, BIG_CK, 3)
    assert (n[:, 1] > 1).any()
