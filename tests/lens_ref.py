"""ctypes binding of tests/lens_ref.c: the thin lens of b2pt_set_lens restated on top of the CPU oracle (test
infrastructure only).  The library is compiled from lens_ref.c, which includes oracle/b2pt_oracle.c unchanged, with the
oracle's own flags, into a per-user cache directory outside the source tree (keyed by the sources' contents)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "lens_ref.c"), os.path.join(ROOT, "oracle", "b2pt_oracle.c"),
           os.path.join(ROOT, "oracle", "b2pt_oracle.h")]
CC = "/usr/bin/gcc"  # the oracle Makefile's compiler and flags: no FMA contraction
CFLAGS = ["-std=gnu11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
          "-Wno-unused-function"]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), "b2pt_lens_ref_%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "liblens_ref_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(lib):
        tmp = lib + ".%d.tmp" % os.getpid()
        subprocess.check_call([CC] + CFLAGS + ["-o", tmp, SOURCES[0], "-lm"])
        os.replace(tmp, lib)
    return lib


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.lens_raygen.restype = C.c_int
        L.lens_raygen.argtypes = [C.POINTER(O._Camera), C.c_float, C.c_float, C.c_int64, C.POINTER(C.c_uint32),
                                  C.c_void_p, C.c_void_p]
        L.lens_primary_hits.restype = C.c_int
        L.lens_primary_hits.argtypes = [C.POINTER(O._Scene), C.POINTER(O._Camera), C.c_float, C.c_float, C.c_uint32,
                                        C.c_int, C.c_void_p, C.c_void_p]
        L.lens_render.restype = C.c_int
        L.lens_render.argtypes = [C.POINTER(O._Scene), C.POINTER(O._Camera), C.c_float, C.c_float, C.c_int, C.c_int,
                                  C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.POINTER(O.Stats)]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def raygen(cam, aperture, focus, idx, seed):
    """The primary ray of pixel idx (an oracle.Camera) from RNG state seed: (origin, direction, state after the ray,
    draws consumed)."""
    s = C.c_uint32(seed & 0xFFFFFFFF)
    o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
    cs = cam.c_struct()
    n = lib().lens_raygen(C.byref(cs), aperture, focus, idx, C.byref(s), _p(o), _p(d))
    return o, d, int(s.value), int(n)


def primary_hits(scene, cam, aperture, focus, seed_offset=0, flags=0):
    n = cam.W * cam.H
    prim, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
    ss, cs = scene.c_struct(), cam.c_struct()
    assert lib().lens_primary_hits(C.byref(ss), C.byref(cs), aperture, focus, seed_offset, flags, _p(prim), _p(t)) == 0
    return prim, t


def render(scene, cam, aperture, focus, spp, max_depth, sample_begin=0, seed_offset=0, flags=0, threads=0):
    """Oracle mode 3 through the lens: (rgba_sum[H*W, 4] float32, oracle.Stats)."""
    rgba = np.zeros((cam.W * cam.H, 4), np.float32)
    st = O.Stats()
    ss, cs = scene.c_struct(), cam.c_struct()
    rc = lib().lens_render(C.byref(ss), C.byref(cs), aperture, focus, spp, sample_begin, max_depth, seed_offset, flags,
                           threads, _p(rgba), C.byref(st))
    if rc != 0:
        raise RuntimeError("lens_render failed: %d" % rc)
    return rgba, st
