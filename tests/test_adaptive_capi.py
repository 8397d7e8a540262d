"""b2pt_render_views_adaptive is part of the C-ABI (declared, exported, bound with the right arity and struct layout),
the driver rejects bad -adaptive uses before it touches a GPU, and the numpy restatement of the selection rule the GPU
tests replay behaves as stated (no GPU needed)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import adaptive_ref as R  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
f32 = np.float32


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


def test_adaptive_entry_points_are_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_render_views_adaptive\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,", hdr)
    assert re.search(r"\bvoid\s+b2pt_adaptive_defaults\s*\(\s*b2pt_adaptive_params\s*\*\s*p\s*\)", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert {"b2pt_render_views_adaptive", "b2pt_adaptive_defaults"} <= exported
    assert len(b2pt.SIGNATURES["b2pt_render_views_adaptive"][1]) == 14
    assert len(b2pt.SIGNATURES["b2pt_adaptive_defaults"][1]) == 1


def test_params_struct_matches_the_header(b2pt, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b2pt.h"\nint main(void){printf("%zu %zu %zu %zu\\n",'
                   ' sizeof(b2pt_adaptive_params), offsetof(b2pt_adaptive_params, threshold), offsetof('
                   'b2pt_adaptive_params, epsilon), offsetof(b2pt_adaptive_params, radius));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    P = b2pt.AdaptiveParams
    assert got == [ctypes.sizeof(P)] + [getattr(P, f).offset for f, _ in P._fields_]


def test_defaults_run_on_the_host(b2pt):
    p = b2pt.AdaptiveParams.defaults()
    assert (p.threshold, p.epsilon, p.radius) == (f32(0.02), f32(0.01), 1)


SWEEP = ["-hemisphere", "-phicount", "2", "-thetacount", "3"]


@pytest.mark.parametrize("args, message", [
    (SWEEP + ["-adaptive", "0.1"], "-adaptive needs -checkpoints"),
    (["-adaptive", "0.1"], "-adaptive needs -hemisphere or -fibonacci"),
    (SWEEP + ["-direct", "-adaptive", "0.1"], "-adaptive cannot be combined with -direct"),
    (SWEEP + ["-checkpoints", "2", "-features", "-adaptive", "0.1"], "-adaptive cannot be combined with -features or -denoise"),
    (SWEEP + ["-checkpoints", "2", "-denoise", "-adaptive", "0.1"], "-adaptive cannot be combined with -features or -denoise"),
    (SWEEP + ["-checkpoints", "2", "-adaptive", "-0.5"], "-adaptive takes a threshold >= 0, got '-0.5'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive", "abc"], "-adaptive takes a threshold >= 0, got 'abc'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive", "0.1x"], "-adaptive takes a threshold >= 0, got '0.1x'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive", "nan"], "-adaptive takes a threshold >= 0, got 'nan'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive"], "-adaptive takes a threshold >= 0, got ''"),
])
def test_driver_rejects_bad_adaptive(host_build, tmp_path, args, message):
    out = subprocess.run([os.path.join(host_build, "CornellBox_b2pt"), "-x", "8", "-y", "8", "-samplecount", "6"] + args,
                         cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert out.returncode == 1, out.stdout + out.stderr
    assert message in out.stderr
    assert os.listdir(tmp_path) == []


def sums(mean, var, c):
    """Sums and sums of squares of c samples with per-channel mean and (population) variance, float32 [..., 4]."""
    mean = np.asarray(mean, np.float64)
    S = np.zeros(mean.shape[:-1] + (4,), f32)
    Q = np.zeros_like(S)
    S[..., :3] = mean * c
    Q[..., :3] = (mean ** 2 + var) * c
    return S, Q


def test_threshold_edges():
    rng = np.random.default_rng(1)
    mean = rng.uniform(0, 2, (2, 50, 3))
    S, Q = sums(mean, rng.uniform(0, 0.5, (2, 50, 1)), 8)
    S[0, :5, :3] = 0  # black pixels of zero variance
    Q[0, :5, :3] = 0
    assert R.unconverged(S, Q, 8, 0.0, 0.01).all()  # tau = 0 converges nothing, not even zero variance
    assert not R.unconverged(S, Q, 8, np.inf, 0.01).any()  # tau = +inf converges everything finite
    assert not R.unconverged(S[0, :5], Q[0, :5], 8, 1e-6, 0.01).any()


def test_relative_error_test_follows_its_formula():
    # one grey pixel of c samples with mean 0.5 and population variance var: V0 = var / (c - 1)
    c, mean, var = 16, 0.5, 0.04
    S, Q = sums([[mean] * 3], var, c)
    V0 = var / (c - 1)
    rel = np.sqrt(V0) / (mean + 0.01)
    assert R.unconverged(S, Q, c, rel * 0.99, 0.01).all()
    assert not R.unconverged(S, Q, c, rel * 1.01, 0.01).any()


def test_nan_luminance_is_unconverged():
    S = np.array([[np.inf, -np.inf, 0, 0]], f32)  # L = inf - inf = NaN
    Q = np.array([[np.inf, np.inf, 0, 0]], f32)
    assert R.unconverged(S, Q, 4, np.inf, 0.01).all()
    S2 = np.array([[np.nan, 0.5, 0.5, 0]], f32)  # a NaN channel counts as 0, as in the denoiser
    Q2 = np.array([[np.nan, 1.0, 1.0, 0]], f32)
    assert R.unconverged(S2, Q2, 4, 0.01, 0.01).all() == R.unconverged(
        np.array([[0, 0.5, 0.5, 0]], f32), np.array([[0, 1.0, 1.0, 0]], f32), 4, 0.01, 0.01).all()


@pytest.mark.parametrize("radius", [0, 1, 2, 4])
def test_dilation_is_a_chebyshev_square_inside_one_view(radius):
    W, H = 11, 9
    u = np.zeros((3, H * W), bool)
    u[1, 4 * W + 5] = True  # view 1, (i, j) = (5, 4)
    u[2, 0] = True  # view 2, corner
    d = R.dilate(u, W, H, radius).reshape(3, H, W)
    j, i = np.mgrid[:H, :W]
    assert not d[0].any()
    assert (d[1] == ((abs(i - 5) <= radius) & (abs(j - 4) <= radius))).all()
    assert (d[2] == ((i <= radius) & (j <= radius))).all()


def test_replay_stops_pixels_for_good():
    rng = np.random.default_rng(2)
    W, H, V = 16, 12, 2
    rounds = (2, 4, 8, 16)
    mean = rng.uniform(0, 1, (V, H * W, 3))
    var = rng.uniform(0, 1, (V, H * W, 1)) ** 4
    S = np.stack([sums(mean, var, c)[0] for c in rounds])
    Q = np.stack([sums(mean, var, c)[1] for c in rounds])
    lum = mean @ np.array([0.2126, 0.7152, 0.0722])
    tau = float(np.quantile(np.sqrt(var[..., 0] / (rounds[0] - 1)) / (lum + 0.01), 0.9))  # a tenth go on after round 0
    for radius in (0, 1):
        counts, active = R.replay(S, Q, rounds, W, H, tau, 0.01, radius)
        assert active[0] == V * H * W
        assert all(active[k] >= active[k + 1] for k in range(len(rounds) - 1))
        assert active[1:].sum() > 0 and (counts == rounds[0]).any()
        for k in range(1, len(rounds)):  # pixels sampled in round k are those that reached rounds[k]
            assert active[k] == (counts >= rounds[k]).sum()
    c0, _ = R.replay(S, Q, rounds, W, H, tau, 0.01, 0)
    c2, _ = R.replay(S, Q, rounds, W, H, tau, 0.01, 2)
    assert (c2 >= c0).all() and (c2 > c0).any()  # a wider radius only adds samples
    assert (R.replay(S, Q, rounds, W, H, 0.0, 0.01, 1)[0] == rounds[-1]).all()
    assert (R.replay(S, Q, rounds, W, H, np.inf, 0.01, 1)[0] == rounds[0]).all()
