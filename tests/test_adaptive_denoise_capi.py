"""b2pt_render_views_adaptive_denoised is part of the C-ABI (declared, exported, bound with the right arity) and the
driver rejects bad -adaptive-denoise uses before it touches a GPU (no GPU needed)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")


@pytest.fixture(scope="module")
def host_build(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    return HOST


def test_entry_point_is_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_render_views_adaptive_denoised\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,"
                     r"[^;]*const\s+b2pt_adaptive_params\s*\*\s*adaptive\s*,\s*const\s+b2pt_denoise_params\s*\*\s*"
                     r"denoise\s*,\s*uint32_t\s+flags\s*,[^;]*void\s*\*\s*denoisedOut\s*\)\s*;", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert "b2pt_render_views_adaptive_denoised" in exported
    args = b2pt.SIGNATURES["b2pt_render_views_adaptive_denoised"][1]
    assert len(args) == 16
    assert args[8]._type_ is b2pt.AdaptiveParams and args[9]._type_ is b2pt.DenoiseParams


SWEEP = ["-hemisphere", "-phicount", "2", "-thetacount", "3"]


@pytest.mark.parametrize("args, message", [
    (SWEEP + ["-adaptive-denoise", "0.1"], "-adaptive-denoise needs -checkpoints"),
    (["-checkpoints", "2", "-adaptive-denoise", "0.1"], "-checkpoints needs -hemisphere or -fibonacci"),
    (["-adaptive-denoise", "0.1"], "-adaptive-denoise needs -hemisphere or -fibonacci"),
    (SWEEP + ["-direct", "-adaptive-denoise", "0.1"], "-adaptive-denoise cannot be combined with -direct"),
    (SWEEP + ["-checkpoints", "2", "-features", "-adaptive-denoise", "0.1"],
     "-adaptive-denoise cannot be combined with -features or -denoise"),
    (SWEEP + ["-checkpoints", "2", "-denoise", "-adaptive-denoise", "0.1"],
     "-adaptive-denoise cannot be combined with -features or -denoise"),
    (SWEEP + ["-checkpoints", "2", "-adaptive", "0.1", "-adaptive-denoise", "0.1"],
     "-adaptive-denoise cannot be combined with -adaptive"),
    (SWEEP + ["-checkpoints", "2", "-adaptive-denoise", "-0.5"], "-adaptive-denoise takes a threshold >= 0, got '-0.5'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive-denoise", "abc"], "-adaptive-denoise takes a threshold >= 0, got 'abc'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive-denoise", "nan"], "-adaptive-denoise takes a threshold >= 0, got 'nan'"),
    (SWEEP + ["-checkpoints", "2", "-adaptive-denoise"], "-adaptive-denoise takes a threshold >= 0, got ''"),
])
def test_driver_rejects_bad_adaptive_denoise(host_build, tmp_path, args, message):
    out = subprocess.run([os.path.join(host_build, "CornellBox_b2pt"), "-x", "8", "-y", "8", "-samplecount", "6"] + args,
                         cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert out.returncode == 1, out.stdout + out.stderr
    assert message in out.stderr
    assert os.listdir(tmp_path) == []
