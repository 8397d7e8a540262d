"""b2pt_denoise_views is part of the C-ABI (declared, exported, bound with the right arity and struct layout), the
driver rejects bad -denoise uses before it touches a GPU, and the float64 restatement of the filter the GPU tests
compare against behaves as an edge-avoiding denoiser should (no GPU needed)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_ref as R  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


def test_denoise_entry_points_are_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_denoise_views\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,", hdr)
    assert re.search(r"\bvoid\s+b2pt_denoise_defaults\s*\(\s*b2pt_denoise_params\s*\*\s*p\s*\)", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert {"b2pt_denoise_views", "b2pt_denoise_defaults"} <= exported
    assert len(b2pt.SIGNATURES["b2pt_denoise_views"][1]) == 13
    assert len(b2pt.SIGNATURES["b2pt_denoise_defaults"][1]) == 1


def test_params_struct_matches_the_header(b2pt, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b2pt.h"\nint main(void){printf("%zu %zu %zu %zu '
                   '%zu %zu\\n", sizeof(b2pt_denoise_params), offsetof(b2pt_denoise_params, levels), offsetof('
                   'b2pt_denoise_params, sigmaLum), offsetof(b2pt_denoise_params, sigmaAlbedo), offsetof('
                   'b2pt_denoise_params, sigmaNormal), offsetof(b2pt_denoise_params, sigmaDepth));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    P = b2pt.DenoiseParams
    assert got == [ctypes.sizeof(P)] + [getattr(P, f).offset for f, _ in P._fields_]


def test_defaults_run_on_the_host(b2pt):
    p = b2pt.DenoiseParams.defaults()
    assert (p.levels, p.sigmaLum, p.sigmaNormal, p.sigmaDepth) == (5, 4.0, np.float32(0.3), 2.0)
    assert p.sigmaAlbedo == np.float32(0.1)


@pytest.mark.parametrize("args, message", [
    (["-denoise"], "-denoise needs -hemisphere or -fibonacci"),
    (["-hemisphere", "-direct", "-denoise"], "-denoise cannot be combined with -direct"),
    (["-fibonacci", "-denoise", "-direct"], "-denoise cannot be combined with -direct"),
    (["-denoise", "-direct"], "-denoise cannot be combined with -direct"),
])
def test_driver_rejects_bad_denoise(host_build, tmp_path, args, message):
    out = subprocess.run([os.path.join(host_build, "CornellBox_b2pt"), "-x", "8", "-y", "8", "-samplecount", "6"] + args,
                         cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert out.returncode == 1, out.stdout + out.stderr
    assert message in out.stderr
    assert os.listdir(tmp_path) == []


def flat_inputs(K, V, H, W, c, rgb, albedo=(0.5, 0.5, 0.5), normal=(0.0, 0.0, -1.0), depth=2.0, var=0.0):
    """Sums of c samples whose mean is rgb (broadcast to [K,V,H*W,3]), a per-channel sample variance var, and constant
    guides of c hitting samples."""
    N = H * W
    rgb = np.broadcast_to(np.asarray(rgb, np.float64), (K, V, N, 3))
    S = np.zeros((K, V, N, 4), np.float32)
    S[..., :3] = rgb * c
    Q = np.zeros_like(S)
    Q[..., :3] = (rgb ** 2 + var * (c - 1) / c) * c
    A = np.zeros_like(S)
    A[..., :3] = np.asarray(albedo) * c
    A[..., 3] = c
    ND = np.zeros_like(S)
    ND[..., :3] = np.asarray(normal) * c
    ND[..., 3] = depth * c
    return S, Q, A, ND


def test_restatement_keeps_a_constant_image_constant():
    S, Q, A, ND = flat_inputs(1, 3, 12, 10, 8, (0.3, 0.6, 0.9), var=0.01)
    x, V = R.denoise(S, Q, A, ND, 10, 12, [8], levels=4)
    assert np.allclose(x, [0.3, 0.6, 0.9], rtol=0, atol=1e-6)
    m, V0, *_ = R.prep(S, Q, A, ND, [8])
    assert (V > 0).all() and (V < V0).all()  # averaging equal variances lowers them


def test_restatement_lowers_the_variance_of_white_noise_on_flat_guides():
    rng = np.random.default_rng(3)
    H = W = 48
    c = 16
    noise = rng.normal(0.5, 0.1, (1, 1, H * W, 3))
    S, Q, A, ND = flat_inputs(1, 1, H, W, c, noise, var=0.1 ** 2 * c)
    x, V = R.denoise(S, Q, A, ND, W, H, [c])
    assert x.var() < 0.1 * noise.var()
    assert abs(x.mean() - noise.mean()) < 1e-3
    m, V0, *_ = R.prep(S, Q, A, ND, [c])
    assert V.mean() < 0.1 * V0.mean()  # the filtered variance follows the averaging


def test_restatement_does_not_mix_regions_of_different_albedo():
    rng = np.random.default_rng(4)
    H, W, c = 24, 32, 8
    left = (np.arange(H * W) % W) < W // 2
    rgb = np.where(left[:, None], 0.2, 0.8) + rng.normal(0, 0.02, (H * W, 3))
    alb = np.where(left[:, None], 0.1, 0.9)  # 8 sigma_a apart: exp(-64 * 3) per tap
    S, Q, A, ND = flat_inputs(1, 1, H, W, c, rgb[None, None], var=0.02 ** 2 * c)
    A[..., :3] = (alb * c)[None, None]
    x, _ = R.denoise(S, Q, A, ND, W, H, [c])
    assert np.abs(x[0, 0][left] - 0.2).max() < 0.05
    assert np.abs(x[0, 0][~left] - 0.8).max() < 0.05
    # without the albedo guide (and the other guides flat) the two sides blur into each other at the edge
    xb, _ = R.denoise(S, None, A, ND, W, H, [c], sigma_albedo=np.inf)
    edge = (np.arange(H * W) % W) == W // 2 - 1
    assert np.abs(xb[0, 0][edge] - 0.2).min() > 0.1
