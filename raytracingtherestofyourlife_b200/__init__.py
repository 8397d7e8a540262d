"""raytracingtherestofyourlife_b200 -- Python harness over libb2pt.so (the C-ABI in include/b2pt.h).

The product is the shared library: hand-written sm_100a kernels behind a C-ABI, with a C++ facade
(host/) that keeps the reference's MapperPathTracer / PathTracer / Camera / ChannelBuffer / Ray API.
This module is the thin ctypes binding tests and bench.py use; torch only supplies device memory,
streams and torch.distributed.  There is NO CPU fallback: if libb2pt.so is missing or no B200 is
present, calls raise.
"""
import ctypes as C
import os

import numpy as np

from . import _build

__all__ = ["lib", "Scene", "Camera", "Context", "B2ptError", "Stats", "FLAG_REFERENCE_STREAM",
           "FLAG_KILL_ZERO_THROUGHPUT", "FLAG_NO_DEDUP", "FLAG_FORCE_BVH", "FLAG_NO_AA", "FLAG_NO_TAIL", "FLAG_NO_OVERLAP", "FLAG_GPU_LBVH", "LIB_PATH"]

LIB_PATH = _build.LIB
FLAG_REFERENCE_STREAM = 0x1
FLAG_KILL_ZERO_THROUGHPUT = 0x2
FLAG_NO_DEDUP = 0x4
FLAG_FORCE_BVH = 0x8
FLAG_NO_AA = 0x10
FLAG_NO_TAIL = 0x20
FLAG_NO_OVERLAP = 0x40
FLAG_GPU_LBVH = 0x80
FLAG_VIEWS_NORMALIZE = 0x100
FLAG_VIEWS_PNM16 = 0x200
FLAG_NO_PRIMARY_MASKS = 0x400
FLAG_ONE_KERNEL_BOUNCE = 0x800
FLAG_WIDE_BVH = 0x1000
FLAG_NO_RAY_SORT = 0x2000
FLAG_SPLIT_TRACE = 0x4000

ERR_BAD_VALUE, ERR_CUDA, ERR_STATE, ERR_ALLOC, ERR_UNSUPPORTED = -1, -2, -3, -4, -5


class B2ptError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("b2pt error %d: %s" % (code, msg))
        self.code = code


class Stats(C.Structure):
    _fields_ = [("paths", C.c_int64), ("segments", C.c_int64), ("nanSamples", C.c_int64), ("launches", C.c_int64),
                ("queueBytes", C.c_int64), ("renderMs", C.c_double), ("batches", C.c_int32),
                ("samplesPerBatch", C.c_int32), ("tracePath", C.c_int32), ("bvhNodes", C.c_int32),
                ("tracedQuads", C.c_int32), ("tracedSpheres", C.c_int32), ("tailDepth", C.c_int32),
                ("loopDepth", C.c_int32)]


_lib = None
_vp, _i64, _i32, _f = C.c_void_p, C.c_int64, C.c_int, C.c_float

# name -> (restype, argtypes); mirrors include/b2pt.h one to one (tests/test_capi_symbols.py checks it)
SIGNATURES = {
    "b2pt_version": (_i32, []),
    "b2pt_create": (_vp, [_i32, C.POINTER(_i32)]),
    "b2pt_destroy": (None, [_vp]),
    "b2pt_last_error": (C.c_char_p, []),
    "b2pt_set_stream": (_i32, [_vp, _vp]),
    "b2pt_set_scene": (_i32, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32,
                              _vp, _i32, _vp, _i32, _vp, _vp, _i32, _i32, _f]),
    "b2pt_build_bvh": (_i32, [_vp]),
    "b2pt_update_spheres": (_i32, [_vp, _vp, _vp]),
    "b2pt_refit_bvh": (_i32, [_vp]),
    "b2pt_set_camera": (_i32, [_vp, _vp, _vp, _vp, _f, _i32, _i32]),
    "b2pt_seed": (_i32, [_vp, C.c_uint32]),
    "b2pt_set_memory_budget": (_i32, [_vp, _i64]),
    "b2pt_render": (_i32, [_vp, _i32, _i32, C.c_uint32]),
    "b2pt_render_range": (_i32, [_vp, _i32, _i32, _i32, C.c_uint32]),
    "b2pt_render_views": (_i32, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, C.c_uint32, _vp]),
    "b2pt_views_device_ptr": (_vp, [_vp]),
    "b2pt_plan_batches": (_i32, [_i64, _i64, _i64, _i32, _vp, _vp]),
    "b2pt_clear_color": (_i32, [_vp]),
    "b2pt_set_color_buffer": (_i32, [_vp, _vp]),
    "b2pt_color_device_ptr": (_vp, [_vp]),
    "b2pt_read_color": (_i32, [_vp, _vp]),
    "b2pt_write_color": (_i32, [_vp, _vp]),
    "b2pt_normalize": (_i32, [_vp, _i32]),
    "b2pt_read_pnm16": (_i32, [_vp, _i32, _vp]),
    "b2pt_synchronize": (_i32, [_vp]),
    "b2pt_get_stats": (_i32, [_vp, C.POINTER(Stats)]),
    "b2pt_build_bvh_ex": (_i32, [_vp, C.c_uint32]),
    "b2pt_get_bounce_profile": (_i32, [_vp, _i32, _vp, _vp]),
    "b2pt_get_stage_profile": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "b2pt_primary_hits": (_i32, [_vp, _vp, _vp]),
    "b2pt_render_direct": (_i32, [_vp] * 5),
    "b2pt_render_direct_views": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "b2pt_create_rays": (_i32, [_vp] * 9),
    "b2pt_intersect": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp]),
    "b2pt_allreduce": (_i32, [C.POINTER(_vp), _i32]),
    "b2pt_scene_cornell": (_i32, [_vp] * 11),
    "b2pt_scene_spheres": (_i32, [_i64] + [_vp] * 11),
    "b2pt_bvh_selfcheck": (_i32, [_i64, _vp]),
}


def lib():
    """Load libb2pt.so (built in-tree by _build.build_lib / __graft_entry__.build). Raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libb2pt.so not built at %s -- run `python -c 'import __graft_entry__ as g; g.build()'`; "
                              "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _check(rc):
    if rc != 0:
        raise B2ptError(rc, lib().b2pt_last_error().decode())


class Scene:
    """Plain-array scene: the inputs MapperPathTracer::RenderCells receives (cell set, coordinates, material
    tables) plus the light lists hard-coded at MapperPathTracer.cxx:141-148."""

    def __init__(self, pts, quadIds, sphPt, sphR, matIdxQ, texIdxQ, matIdxS, texIdxS, matType, texType, tex,
                 lightQuadIds, lightSphPt, lightSphR, lightables=2, refIdx=1.5):
        f32, i64, i32 = np.float32, np.int64, np.int32
        self.pts = np.ascontiguousarray(pts, f32).reshape(-1, 3)
        self.quadIds = np.ascontiguousarray(quadIds, i64).reshape(-1, 5)
        self.sphPt = np.ascontiguousarray(sphPt, i64).reshape(-1)
        self.sphR = np.ascontiguousarray(sphR, f32).reshape(-1)
        self.matIdxQ = np.ascontiguousarray(matIdxQ, i64).reshape(-1)
        self.texIdxQ = np.ascontiguousarray(texIdxQ, i64).reshape(-1)
        self.matIdxS = np.ascontiguousarray(matIdxS, i64).reshape(-1)
        self.texIdxS = np.ascontiguousarray(texIdxS, i64).reshape(-1)
        self.matType = np.ascontiguousarray(matType, i32).reshape(-1)
        self.texType = np.ascontiguousarray(texType, i32).reshape(-1)
        self.tex = np.ascontiguousarray(tex, f32).reshape(-1, 3)
        self.lightQuadIds = np.ascontiguousarray(lightQuadIds, i64).reshape(-1, 5)
        self.lightSphPt = np.ascontiguousarray(lightSphPt, i64).reshape(-1)
        self.lightSphR = np.ascontiguousarray(lightSphR, f32).reshape(-1)
        self.lightables = int(lightables)
        self.refIdx = float(refIdx)

    def nbytes(self):
        return sum(a.nbytes for a in (self.pts, self.quadIds, self.sphPt, self.sphR, self.matIdxQ, self.texIdxQ,
                                      self.matIdxS, self.texIdxS, self.matType, self.texType, self.tex,
                                      self.lightQuadIds, self.lightSphPt, self.lightSphR))

    @staticmethod
    def cornell():
        """CornellBox::buildDataSet (CornellBox.cpp:141-418) through the library's host-side builder."""
        f32, i64, i32 = np.float32, np.int64, np.int32
        pts, quadIds = np.zeros((89, 3), f32), np.zeros((22, 5), i64)
        sphPt, sphR = np.zeros(1, i64), np.zeros(1, f32)
        mq, tq, ms, ts = np.zeros(22, i64), np.zeros(22, i64), np.zeros(1, i64), np.zeros(1, i64)
        matType, texType, tex = np.zeros(5, i32), np.zeros(5, i32), np.zeros((4, 3), f32)
        _check(lib().b2pt_scene_cornell(_p(pts), _p(quadIds), _p(sphPt), _p(sphR), _p(mq), _p(tq), _p(ms), _p(ts),
                                        _p(matType), _p(texType), _p(tex)))
        return Scene(pts, quadIds, sphPt, sphR, mq, tq, ms, ts, matType, texType, tex,
                     lightQuadIds=[[0, 8, 9, 10, 11]], lightSphPt=[48], lightSphR=[sphR[0]])

    @staticmethod
    def spheres(n):
        """BASELINE.json configs[3]: n random lambertian spheres, one emissive quad, one floor quad."""
        f32, i64, i32 = np.float32, np.int64, np.int32
        pts, quadIds = np.zeros((n + 8, 3), f32), np.zeros((2, 5), i64)
        sphPt, sphR = np.zeros(n, i64), np.zeros(n, f32)
        mq, tq, ms, ts = np.zeros(2, i64), np.zeros(2, i64), np.zeros(n, i64), np.zeros(n, i64)
        matType, texType, tex = np.zeros(5, i32), np.zeros(5, i32), np.zeros((4, 3), f32)
        _check(lib().b2pt_scene_spheres(n, _p(pts), _p(quadIds), _p(sphPt), _p(sphR), _p(mq), _p(tq), _p(ms), _p(ts),
                                        _p(matType), _p(texType), _p(tex)))
        return Scene(pts, quadIds, sphPt, sphR, mq, tq, ms, ts, matType, texType, tex,
                     lightQuadIds=[[0, n, n + 1, n + 2, n + 3]], lightSphPt=[0], lightSphR=[sphR[0]])


def bvh_selfcheck(n_spheres):
    """Host-only: (binary nodes, binary depth, wide nodes, wide depth) of the validated trees over n random spheres."""
    st = np.zeros(4, np.int64)
    _check(lib().b2pt_bvh_selfcheck(n_spheres, _p(st)))
    return tuple(int(x) for x in st)


def plan_batches(units, unit_paths, max_paths_per_batch=1 << 27, sets=4):
    """(units per batch, number of batches) of the library's batch split (b2pt_plan_batches; host logic, no GPU)."""
    per, nb = C.c_int64(0), C.c_int64(0)
    _check(lib().b2pt_plan_batches(units, unit_paths, max_paths_per_batch, sets, C.byref(per), C.byref(nb)))
    return per.value, nb.value


class Camera:
    """main.cc:616-622 defaults (pos (278,278,-800)/555, look-at box centre, fov 40)."""

    def __init__(self, W, H, pos=None, lookAt=None, up=(0, 1, 0), fov=40.0):
        f = np.float32
        self.pos = np.array(pos if pos is not None else [278 / 555.0, 278 / 555.0, -800 / 555.0], f)
        self.lookAt = np.array(lookAt if lookAt is not None else [278 / 555.0, 278 / 555.0, 278 / 555.0], f)
        self.up = np.array(up, f)
        self.fov, self.W, self.H = float(fov), int(W), int(H)


class Context:
    """One libb2pt context (one GPU)."""

    def __init__(self, device=0):
        err = C.c_int(0)
        self._h = lib().b2pt_create(device, C.byref(err))
        if not self._h:
            raise B2ptError(err.value, lib().b2pt_last_error().decode())
        self.device = device
        self._keep = None
        self.W = self.H = 0

    def close(self):
        if getattr(self, "_h", None):
            lib().b2pt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream_ptr):
        _check(lib().b2pt_set_stream(self._h, cuda_stream_ptr))

    def set_scene(self, s):
        _check(lib().b2pt_set_scene(
            self._h, _p(s.pts), len(s.pts), _p(s.quadIds), len(s.quadIds), _p(s.sphPt), _p(s.sphR), len(s.sphPt),
            _p(s.matIdxQ), _p(s.texIdxQ), _p(s.matIdxS), _p(s.texIdxS), _p(s.matType), len(s.matType), _p(s.texType),
            len(s.texType), _p(s.tex), len(s.tex), _p(s.lightQuadIds), len(s.lightQuadIds), _p(s.lightSphPt),
            _p(s.lightSphR), len(s.lightSphPt), s.lightables, s.refIdx))

    def build_bvh(self, flags=0):
        _check(lib().b2pt_build_bvh_ex(self._h, flags))

    def update_spheres(self, centers, radii=None):
        c = np.ascontiguousarray(centers, np.float32).reshape(-1, 3)
        r = None if radii is None else np.ascontiguousarray(radii, np.float32).reshape(-1)
        _check(lib().b2pt_update_spheres(self._h, _p(c), _p(r)))

    def refit_bvh(self):
        _check(lib().b2pt_refit_bvh(self._h))

    def set_camera(self, cam):
        _check(lib().b2pt_set_camera(self._h, _p(cam.pos), _p(cam.lookAt), _p(cam.up), cam.fov, cam.W, cam.H))
        self.W, self.H = cam.W, cam.H

    def set_memory_budget(self, nbytes):
        _check(lib().b2pt_set_memory_budget(self._h, nbytes))

    def seed(self, offset):
        _check(lib().b2pt_seed(self._h, offset))

    def render(self, spp, max_depth, flags=0):
        _check(lib().b2pt_render(self._h, spp, max_depth, flags))

    def render_range(self, begin, count, max_depth, flags=0):
        _check(lib().b2pt_render_range(self._h, begin, count, max_depth, flags))

    def render_views(self, views, W, H, spp, max_depth, flags=0, out=None):
        """b2pt_render_views: `views` is [nViews, 10] float32 (pos, lookAt, up, fovDeg); returns the [nViews, H*W, 4]
        radiance sums (un-normalised unless FLAG_VIEWS_NORMALIZE), each bit-identical to set_camera + render."""
        v = np.ascontiguousarray(views, np.float32).reshape(-1, 10)
        pnm = bool(flags & FLAG_VIEWS_PNM16)  # uint16 [nViews, H*W, 3]: the integers of the reference's P3 writer
        dt, ch = (np.uint16, 3) if pnm else (np.float32, 4)
        if out is None:
            out = np.empty((v.shape[0], W * H, ch), dt)
        assert out.dtype == dt and out.flags.c_contiguous and out.size == v.shape[0] * W * H * ch
        _check(lib().b2pt_render_views(self._h, v.shape[0], _p(v), W, H, spp, max_depth, flags, _p(out)))
        return out

    def clear_color(self):
        _check(lib().b2pt_clear_color(self._h))

    def set_color_tensor(self, t):
        """Attach a torch CUDA tensor of shape [H*W,4] float32 as the radiance sum (torch owns the memory)."""
        if t is None:
            _check(lib().b2pt_set_color_buffer(self._h, None))
            self._keep = None
            return
        assert t.is_cuda and t.is_contiguous() and t.numel() == self.W * self.H * 4 and t.element_size() == 4
        _check(lib().b2pt_set_color_buffer(self._h, t.data_ptr()))
        self._keep = t

    def read_color(self, out=None):
        if out is None:
            out = np.zeros((self.W * self.H, 4), np.float32)
        _check(lib().b2pt_read_color(self._h, out.ctypes.data_as(C.c_void_p) if isinstance(out, np.ndarray) else out))
        return out

    def write_color(self, rgba):
        rgba = np.ascontiguousarray(rgba, np.float32)
        _check(lib().b2pt_write_color(self._h, _p(rgba)))

    def read_pnm16(self, spp):
        """uint16 [H*W, 3]: int(255.99 * sqrt(de_nan(sum)/spp)), what the reference's save() prints (main.cc:325-384)."""
        out = np.zeros((self.W * self.H, 3), np.uint16)
        _check(lib().b2pt_read_pnm16(self._h, spp, _p(out)))
        return out

    def normalize(self, spp):
        _check(lib().b2pt_normalize(self._h, spp))

    def synchronize(self):
        _check(lib().b2pt_synchronize(self._h))

    def stats(self):
        st = Stats()
        _check(lib().b2pt_get_stats(self._h, C.byref(st)))
        return st

    def bounce_profile(self, n=16):
        """[(ms, rays_in)] of the first bounce launches of the last render's first batch (CUDA events)."""
        ms, rays = np.zeros(n, np.float32), np.zeros(n, np.int64)
        k = lib().b2pt_get_bounce_profile(self._h, n, _p(ms), _p(rays))
        if k < 0:
            _check(k)
        return [(float(ms[i]), int(rays[i])) for i in range(k)]

    def stage_profile(self, n=16):
        """[(trace_ms, shade_ms, rays_in)] of the same launches, split into the k_trace and k_shade launch."""
        tr, sh, rays = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.int64)
        k = lib().b2pt_get_stage_profile(self._h, n, _p(tr), _p(sh), _p(rays))
        if k < 0:
            _check(k)
        return [(float(tr[i]), float(sh[i]), int(rays[i])) for i in range(k)]

    def primary_hits(self):
        n = self.W * self.H
        prim, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
        _check(lib().b2pt_primary_hits(self._h, _p(prim), _p(t)))
        return prim, t

    def render_direct(self):
        """-direct G-buffers (b2pt_render_direct): (normals[N,4], albedo[N,4], depth[N], prim[N])."""
        n = self.W * self.H
        normals, albedo = np.zeros((n, 4), np.float32), np.zeros((n, 4), np.float32)
        depth, prim = np.zeros(n, np.float32), np.zeros(n, np.int32)
        _check(lib().b2pt_render_direct(self._h, _p(normals), _p(albedo), _p(depth), _p(prim)))
        return normals, albedo, depth, prim

    def render_direct_views(self, views, W, H):
        """b2pt_render_direct_views: `views` is [nViews, 10] float32 (pos, lookAt, up, fovDeg); returns
        (normals[V,H*W,4], albedo[V,H*W,4], depth[V,H*W], prim[V,H*W]), view v bit-identical to set_camera + render_direct."""
        v = np.ascontiguousarray(views, np.float32).reshape(-1, 10)
        nv, n = v.shape[0], W * H
        normals, albedo = np.zeros((nv, n, 4), np.float32), np.zeros((nv, n, 4), np.float32)
        depth, prim = np.zeros((nv, n), np.float32), np.zeros((nv, n), np.int32)
        _check(lib().b2pt_render_direct_views(self._h, nv, _p(v), W, H, _p(normals), _p(albedo), _p(depth), _p(prim)))
        return normals, albedo, depth, prim

    def create_rays(self, seeds):
        n = self.W * self.H
        seeds = np.ascontiguousarray(seeds, np.uint32).copy()
        d = [np.zeros(n, np.float32) for _ in range(6)]
        pix = np.zeros(n, np.int64)
        _check(lib().b2pt_create_rays(self._h, _p(seeds), _p(d[0]), _p(d[1]), _p(d[2]), _p(d[3]), _p(d[4]), _p(d[5]),
                                      _p(pix)))
        return seeds, np.stack(d[:3], 1), np.stack(d[3:], 1), pix

    def intersect(self, o, d, tmin=0.001, tmax=float(np.finfo(np.float32).max)):
        o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
        n = len(o)
        cols = [np.ascontiguousarray(a) for a in (o[:, 0], o[:, 1], o[:, 2], d[:, 0], d[:, 1], d[:, 2])]
        prim, mat, texi = (np.zeros(n, np.int32) for _ in range(3))
        rec = np.zeros((9, n), np.float32)
        _check(lib().b2pt_intersect(self._h, n, *[_p(c) for c in cols], tmin, tmax, _p(prim), _p(rec), _p(mat),
                                    _p(texi)))
        return prim, rec, mat, texi
