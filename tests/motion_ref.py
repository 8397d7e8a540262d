"""ctypes binding of tests/motion_ref.c: the motion vectors of b2pt_render_views_motion restated on top of the CPU oracle
(test infrastructure only).  The library is compiled from motion_ref.c, which includes tests/lens_ref.c and through it
oracle/b2pt_oracle.c unchanged, with the oracle's own flags, into a per-user cache directory outside the source tree
(keyed by the sources' contents)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "motion_ref.c"), os.path.join(HERE, "lens_ref.c"),
           os.path.join(ROOT, "oracle", "b2pt_oracle.c"), os.path.join(ROOT, "oracle", "b2pt_oracle.h")]
CC = "/usr/bin/gcc"  # the oracle Makefile's compiler and flags: no FMA contraction
CFLAGS = ["-std=gnu11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
          "-Wno-unused-function"]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), "b2pt_motion_ref_%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "libmotion_ref_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(lib):
        tmp = lib + ".%d.tmp" % os.getpid()
        subprocess.check_call([CC] + CFLAGS + ["-o", tmp, SOURCES[0], "-lm"])
        os.replace(tmp, lib)
    return lib


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.motion_sample.restype = C.c_int
        L.motion_sample.argtypes = [C.POINTER(O._Scene), C.POINTER(O._Camera), C.POINTER(O._Camera), C.c_float,
                                    C.c_float, C.c_int64, C.c_uint32, C.c_void_p]
        L.motion_sums.restype = C.c_int
        L.motion_sums.argtypes = [C.POINTER(O._Scene), C.POINTER(O._Camera), C.POINTER(O._Camera), C.c_float,
                                  C.c_float, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def sample(scene, cam, prev, idx, seed, aperture=0.0, focus=0.0):
    """One sample of pixel idx from RNG state seed: (valid, dict of x, y, xp, yp, w, wp, visible, hit, t)."""
    out = np.zeros(9, np.float32)
    ss, cs, ps = scene.c_struct(), cam.c_struct(), prev.c_struct()
    valid = lib().motion_sample(C.byref(ss), C.byref(cs), C.byref(ps), aperture, focus, idx, seed & 0xFFFFFFFF,
                                _p(out))
    names = ("x", "y", "xp", "yp", "w", "wp", "visible", "hit", "t")
    return bool(valid), dict(zip(names, out))


def sums(scene, cam, prev, checkpoints, aperture=0.0, focus=0.0, seed_offset=0):
    """float32 [K, H*W, 4]: the (sum m.x, sum m.y, sum visible, sum valid) of one view, as b2pt_render_views_motion
    computes them."""
    c = np.ascontiguousarray(checkpoints, np.int32).reshape(-1)
    out = np.zeros((len(c), cam.W * cam.H, 4), np.float32)
    ss, cs, ps = scene.c_struct(), cam.c_struct(), prev.c_struct()
    rc = lib().motion_sums(C.byref(ss), C.byref(cs), C.byref(ps), aperture, focus, seed_offset, len(c), _p(c), _p(out))
    if rc != 0:
        raise RuntimeError("motion_sums failed: %d" % rc)
    return out
