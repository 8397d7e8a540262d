"""b2pt_render_views_motion is part of the C-ABI (declared in include/b2pt.h, exported by libb2pt.so, bound in
SIGNATURES and by Context.render_views_motion), and the driver rejects bad -motion uses before it touches a GPU (no GPU
needed)."""
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


def test_render_views_motion_is_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_render_views_motion\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,\s*"
                     r"const\s+float\s*\*\s*views\s*,\s*const\s+float\s*\*\s*prevViews\s*,", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    assert any(l.split()[-1] == "b2pt_render_views_motion" and " T " in l for l in out.splitlines())
    assert "b2pt_render_views_motion" in b2pt.SIGNATURES
    assert len(b2pt.SIGNATURES["b2pt_render_views_motion"][1]) == 10
    assert callable(getattr(b2pt.Context, "render_views_motion", None))


@pytest.mark.parametrize("args, message", [
    (["-hemisphere", "-direct", "-motion"], "-motion cannot be combined with -direct"),
    (["-motion", "-direct"], "-motion cannot be combined with -direct"),
    (["-motion"], "-motion needs -hemisphere"),
    (["-fibonacci", "-motion"], "-motion cannot be combined with -fibonacci"),
    (["-hemisphere", "-fibonacci", "-motion"], "-motion cannot be combined with -fibonacci"),
    (["-hemisphere", "-checkpoints", "2", "-adaptive", "0.1", "-motion"],
     "-motion cannot be combined with -adaptive or -adaptive-denoise"),
    (["-hemisphere", "-checkpoints", "2", "-adaptive-denoise", "0.1", "-motion"],
     "-motion cannot be combined with -adaptive or -adaptive-denoise"),
])
def test_driver_rejects_bad_motion(host_build, tmp_path, args, message):
    out = subprocess.run([os.path.join(host_build, "CornellBox_b2pt"), "-x", "8", "-y", "8", "-samplecount", "6"] + args,
                         cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert out.returncode == 1, out.stdout + out.stderr
    assert message in out.stderr
    assert os.listdir(tmp_path) == []
