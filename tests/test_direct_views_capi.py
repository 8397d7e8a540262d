"""b2pt_render_direct_views is part of the C-ABI: declared in include/b2pt.h and exported by libb2pt.so (no GPU needed)."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_render_direct_views_is_declared_and_exported(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    assert re.search(r"\bint\s+b2pt_render_direct_views\s*\(\s*b2pt_ctx\s*\*\s*ctx\s*,\s*int\s+nViews\s*,", hdr)
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    assert any(l.split()[-1] == "b2pt_render_direct_views" and " T " in l for l in out.splitlines())
    assert "b2pt_render_direct_views" in b2pt.SIGNATURES
