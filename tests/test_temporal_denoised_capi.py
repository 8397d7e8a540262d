"""b2pt_render_views_temporal_denoised is part of the C-ABI (declared in include/b2pt.h, exported by libb2pt.so, bound
in SIGNATURES with its 18 arguments and by Context.render_views_temporal_denoised), and the driver, whose -temporal
files it now produces, still builds (no GPU needed)."""
import inspect
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "raytracingtherestofyourlife_b200", "host")
NAME = "b2pt_render_views_temporal_denoised"


def test_symbol_is_declared_exported_and_bound(b2pt):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2pt.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+%s\s*\(([^)]*)\)\s*;" % NAME, hdr)
    assert m, "not declared"
    params = [p.strip() for p in m.group(1).split(",")]
    assert len(params) == 18
    assert re.fullmatch(r"b2pt_ctx\s*\*\s*ctx", params[0])
    assert re.fullmatch(r"void\s*\*\s*out", params[11])
    assert re.fullmatch(r"float\s*\*\s*motionOut", params[17])
    out = subprocess.check_output(["nm", "-D", "--defined-only", b2pt.LIB_PATH], text=True)
    assert any(l.split()[-1] == NAME and " T " in l for l in out.splitlines())
    res, args = b2pt.SIGNATURES[NAME]
    assert len(args) == 18
    sig = inspect.signature(b2pt.Context.render_views_temporal_denoised)
    assert list(sig.parameters) == ["self", "views", "W", "H", "checkpoints", "max_depth", "temporal", "denoise",
                                    "flags", "history", "inputs"]
    assert [sig.parameters[k].default for k in ("temporal", "denoise", "flags", "history", "inputs")] == \
        [None, None, 0, False, False]


def test_driver_builds(b2pt):
    import runpy
    runpy.run_path(os.path.join(HOST, "build_host.py"), run_name="__test_build__")["build_host"]()
    assert os.access(os.path.join(HOST, "CornellBox_b2pt"), os.X_OK)
