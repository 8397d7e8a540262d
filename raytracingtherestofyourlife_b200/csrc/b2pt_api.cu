// b2pt_api.cu -- the C-ABI of libb2pt.so (include/b2pt.h): contexts, scene/camera set-up, BVH build,
// the wavefront render loop and the stage-level entry points.  Host code only; kernels live in
// b2pt_kernels.cu.  There is no CPU fallback anywhere in this file: without a usable CUDA device every
// computing entry point returns B2PT_ERR_CUDA.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <limits>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/b2pt.h"
#include "b2pt_bvh.h"
#include "b2pt_kernels.h"
#include "b2pt_lbvh.h"
#include "b2pt_types.h"
#include "b2pt_wide.h"

namespace
{

thread_local std::string g_lastError;

int fail(int code, const char* fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_lastError = buf;
  return code;
}

#define CU(call)                                                                                                       \
  do                                                                                                                   \
  {                                                                                                                    \
    cudaError_t e__ = (call);                                                                                          \
    if (e__ != cudaSuccess)                                                                                            \
      return fail(B2PT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);         \
  } while (0)

// Owning device allocation: freed by the destructor (on the device that is current then -- every owner binds its
// context's device first), movable, not copyable, so a buffer cannot be forgotten on an error path.
template <class T>
struct DevBuf
{
  T* p = nullptr;
  size_t cap = 0; // elements
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept
    : p(o.p)
    , cap(o.cap)
  {
    o.p = nullptr;
    o.cap = 0;
  }
  DevBuf& operator=(DevBuf&& o) noexcept
  {
    if (this != &o)
    {
      release();
      p = o.p, cap = o.cap;
      o.p = nullptr, o.cap = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  cudaError_t reserve(size_t n)
  {
    if (n <= cap)
      return cudaSuccess;
    if (p)
      cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, n * sizeof(T));
    if (e == cudaSuccess)
      cap = n;
    return e;
  }
  void release()
  {
    if (p)
      cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// host float helpers: same operation order as the reference's vtkm::Vec math (no FMA contraction)
struct H3
{
  float x, y, z;
};
inline H3 hsub(H3 a, H3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
inline float hdot(H3 a, H3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
inline H3 hcross(H3 a, H3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
inline H3 hscale(H3 a, float s) { return { a.x * s, a.y * s, a.z * s }; }
inline H3 hnormalize(H3 a) { return hscale(a, 1.0f / std::sqrt(hdot(a, a))); }
inline void hst(float* d, H3 a)
{
  d[0] = a.x;
  d[1] = a.y;
  d[2] = a.z;
}

} // namespace

struct b2pt_ctx
{
  int device = 0;
  cudaStream_t ownStream = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t evStart = nullptr, evStop = nullptr;
  static constexpr int kProfDepths = 16;
  cudaEvent_t evBounce[kProfDepths + 1] = {}; // batch 0: event before each of the first bounces + one after
  cudaEvent_t evMid[kProfDepths + 1] = {};    // batch 0: event between k_trace and k_shade of those bounces
  int profDepths = 0;
  int64_t profPaths = 0;
  b2pt::LaunchCfg cfg{};

  // scene (host)
  bool haveScene = false, haveBvh = false, haveCamera = false;
  int64_t nQuads = 0, nSph = 0;
  std::vector<B2Quad> quads; // by original index
  std::vector<B2Sphere> sph;
  std::vector<int64_t> sphPointIds, lightSphPointIds; // point id of every sphere / light sphere (b2pt_update_spheres)
  std::vector<B2GateBox> gates; // leaf boxes of non-planar quads (B2Quad::gate indexes this, 1-based)
  std::vector<B2GateBox> boxes; // leaf box of every quad (AABBSurface.h), by original index
  B2Lights lights{};
  // trace structures
  bool useBvh = false;
  B2SmallScene small{};
  B2BvhScene bvh{};
  DevBuf<B2BvhNode> dNodes;
  DevBuf<uint4> dWide; // 8-wide compressed nodes, 5 x uint4 each
  DevBuf<int32_t> dParent; // b2pt_refit_bvh: parent of every binary node (-1 root, -2 not in the tree)
  DevBuf<int> dArrived;
  bool haveParents = false;
  DevBuf<int32_t> dSlots;
  DevBuf<int32_t> dBinSlots; // B2PT_FLAG_WIDE_BVH: the slots in the binary tree's leaf order (direct rays walk that tree)
  DevBuf<float4> dLeafSph;
  DevBuf<B2Quad> dQuads;
  DevBuf<B2Sphere> dSph;
  DevBuf<B2GateBox> dGates;
  int32_t tracedQuads = 0, tracedSph = 0, bvhNodes = 0;
  float sortLo[3] = { 0.f, 0.f, 0.f }, sortHi[3] = { 1.f, 1.f, 1.f }; // scene box (cells of the ray sort)
  uint32_t builtFlags = 0;
  size_t treeSlots = 0;   // primitives in the binary tree (B2PT_VALIDATE_BVH)
  bool treeStale = false; // b2pt_update_spheres moved spheres since the BVH was last built or refitted

  // camera
  B2Camera cam{};
  float camLookAt[3] = { 0.f, 0.f, 0.f }, camUpN[3] = { 0.f, 1.f, 0.f }; // look-at point, up as Camera::SetUp stores it
  uint32_t seedOffset = 0;

  // buffers
  DevBuf<float4> colorOwn;
  float4* colorExt = nullptr;
  int64_t colorPixels = 0;
  // Sets of per-batch buffers: consecutive sample batches run on up to kMaxSets streams, so the poorly occupied tail of
  // batch b overlaps the full-grid head of batch b+1 (set = batch % nSets; sets are allocated on first use)
  static constexpr int kMaxSets = 4;
  struct BatchBufs
  {
    DevBuf<uint4> queue[3];   // two-kernel pipeline: the compact ray queue (three 16-byte planes)
    DevBuf<uint4> bins[2][3]; // sorted hit bins: 4 bins x pathsPerBatch records per plane; the one-kernel pipeline
                              // ping-pongs between two sets, the two-kernel pipeline uses set 0
    DevBuf<uint32_t> binCode[2];
    DevBuf<uint32_t> regionCounts; // qCount[numWarps] + two sets of bin counts [4*numWarps]
    DevBuf<float4> rad;
    DevBuf<uint32_t> sortKeys, sortPerm, sortHist; // BVH scenes: spatial sort of the ray queue (b2pt_kernels.cu)
    DevBuf<unsigned char> sortTemp;
    DevBuf<uint2> hits; // split BVH bounce: closest hit per queue entry (k_bvh_hits -> k_resolve_hits)
    void release_all()
    {
      for (auto& q : queue)
        q.release();
      for (auto& set : bins)
        for (auto& p : set)
          p.release();
      for (auto& c : binCode)
        c.release();
      regionCounts.release();
      rad.release();
      sortKeys.release(), sortPerm.release(), sortHist.release(), sortTemp.release();
      hits.release();
    }
  } bufs[kMaxSets];
  cudaStream_t extra[kMaxSets] = {}; // own non-blocking streams of sets 1.. (set 0 runs on `stream`)
  cudaEvent_t evFork = nullptr, evJoin[kMaxSets] = {}, evAcc[kMaxSets] = {};
  DevBuf<uint32_t> counters;
  DevBuf<uint32_t> binTotals; // tail mode: per batch, per depth, per bin record counts
  DevBuf<uint32_t> seeds;
  DevBuf<unsigned long long> nanCounter;
  std::vector<uint32_t> hCounters;
  // view-batched render (b2pt_render_views): camera bases and the [nViews][W*H] radiance sums
  DevBuf<B2Camera> dViews;
  DevBuf<float4> viewColor;
  DevBuf<uint16_t> pnm; // packed PNM integers (b2pt_read_pnm16, B2PT_FLAG_VIEWS_PNM16)
  // b2pt_render_views_checkpoints: [K-1][nViews][W*H] prefix sums and [K][nViews][W*H] sums of squares
  DevBuf<float4> ckptSnap, ckptMoment;
  // b2pt_render_views_features: [K][chunk views][W*H] staging of one chunk's sums
  DevBuf<float4> featAlbedo, featNormalDepth;
  // b2pt_denoise_views: [K][chunk views][W*H] staging of one chunk: the ping-pong (x, V) images (the colour sums and
  // sums of squares arrive in them) and the two guides
  DevBuf<float4> dnX[2], dnGuideA, dnGuideNZ;
  // b2pt_render_views_adaptive: per canvas entry the sample count, the unconverged and active flags; the compacted list
  // of the next round's entries (padded to whole tiles), its length and the cub scratch
  DevBuf<int32_t> adCounts, adNum;
  DevBuf<uint8_t> adUnconv, adActive;
  DevBuf<uint32_t> adList;
  DevBuf<unsigned char> adTemp;
  DevBuf<uint2> primMask;         // primary-ray specialisation: [views][tiles] candidate masks (k_primary_prep)
  DevBuf<B2PrimQuad> primQuads;   // ... and [views][B2PT_SMALL_MAX_QUADS] per-quad constants
  int64_t viewCount = 0, viewPixels = 0;
  // -direct G-buffers (b2pt_render_direct*): per-view constants and the device staging of one chunk of views
  DevBuf<b2pt::DirectView> dDirectViews;
  DevBuf<float4> directNormals, directAlbedo;
  DevBuf<float> directDepth;
  DevBuf<int32_t> directPrim;

  // tail-mode depths chosen by the last render with the same scene / canvas / depth / batch shape (reused without
  // a new synchronisation; they are heuristics, any value is correct)
  int64_t tailKey[7] = { -1, -1, -1, -1, -1, -1, -1 };
  int64_t sceneVersion = 0;
  uint64_t sceneHash = 0;
  int tailDepthCached = 0, loopDepthCached = 0;
  int64_t memBudget = 0;  // 0.85 of the memory free at the first render: bounds the default batch size
  int64_t userBudget = 0; // b2pt_set_memory_budget (0 = automatic)

  b2pt_stats stats{};
  bool statsPending = false;
  int64_t pendingCounters = 0;
  int pendingMaxDepth = 0;
  int64_t pendingPathsPerBatch = 0;

  float4* color() { return colorExt ? colorExt : colorOwn.p; }
};

namespace
{

int bind(b2pt_ctx* ctx)
{
  if (!ctx)
    return fail(B2PT_ERR_BAD_VALUE, "null context");
  CU(cudaSetDevice(ctx->device));
  return B2PT_OK;
}

int ensure_color(b2pt_ctx* ctx)
{
  const int64_t n = (int64_t)ctx->cam.W * ctx->cam.H;
  if (ctx->colorExt)
    return B2PT_OK;
  if (ctx->colorPixels != n || !ctx->colorOwn.p)
  {
    CU(ctx->colorOwn.reserve((size_t)n));
    ctx->colorPixels = n;
    CU(cudaMemsetAsync(ctx->colorOwn.p, 0, sizeof(float4) * (size_t)n, ctx->stream));
  }
  return B2PT_OK;
}

// Ray-independent parts of Surface.h:30-104 and :180-181 for one quad (q,r,s,t = v00,v10,v11,v01).
void precompute_quad(B2Quad& Q, H3 q, H3 r, H3 s, H3 t)
{
  hst(Q.v00, q);
  hst(Q.e01, hsub(r, q));
  hst(Q.e03, hsub(t, q));
  hst(Q.v11, s);
  hst(Q.e21, hsub(r, s));
  hst(Q.e23, hsub(t, s));
  hst(Q.nrm, hnormalize(hcross(hsub(r, q), hsub(s, q)))); // vtkm::TriangleNormal(q,r,s), Normalize
  // second-triangle shortcut constants (b2pt_types.h): parallelogram iff q + E01 + E03 reproduces s to 1e-6 of the
  // quad's size
  const double l01 = std::fabs((double)Q.e01[0]) + std::fabs((double)Q.e01[1]) + std::fabs((double)Q.e01[2]);
  const double l03 = std::fabs((double)Q.e03[0]) + std::fabs((double)Q.e03[1]) + std::fabs((double)Q.e03[2]);
  double defect = 0.0;
  for (int c = 0; c < 3; ++c)
    defect = std::fmax(defect, std::fabs((double)Q.v00[c] + (double)Q.e01[c] + (double)Q.e03[c] - (double)Q.v11[c]));
  const bool para = std::isfinite(l01 + l03) && l01 > 0 && l03 > 0 && defect <= 1e-6 * (l01 + l03);
  Q.secC1 = (float)(2.0 * (l01 + l03));
  Q.secC2 = para ? (float)(1e-5 * l03) * 1.0000002f : std::numeric_limits<float>::infinity();
}

// pathtracing/AABBSurface.h:24-78 (FindQuadAABBs): min/max over the four vertices, padded per axis.
void quad_leaf_box(B2GateBox& G, H3 q, H3 r, H3 s, H3 t)
{
  const float v[4][3] = { { q.x, q.y, q.z }, { r.x, r.y, r.z }, { s.x, s.y, s.z }, { t.x, t.y, t.z } };
  for (int c = 0; c < 3; ++c)
  {
    float lo = v[0][c], hi = v[0][c];
    for (int k = 1; k < 4; ++k)
    {
      lo = std::fmin(lo, v[k][c]);
      hi = std::fmax(hi, v[k][c]);
    }
    const float eps = std::fmax(1e-6f, 1.0e-4f * (hi - lo));
    G.bmin[c] = lo - eps;
    G.bmax[c] = hi + eps;
  }
  G.quad = -1;
  G.pad = 0;
}

// A quad needs the leaf-box gate unless it is planar: for planar quads every hit the Lagae-Dutre test accepts
// lies on the quad, hence inside its padded box, and the gate is a no-op.
bool quad_is_planar(H3 q, H3 r, H3 s, H3 t, const float* unitNormal)
{
  const H3 n = { unitNormal[0], unitNormal[1], unitNormal[2] };
  const H3 e[3] = { hsub(r, q), hsub(s, q), hsub(t, q) };
  float scale = 0.f;
  for (const H3& v : e)
    scale = std::fmax(scale, std::sqrt(hdot(v, v)));
  const float dev = std::fmax(std::fabs(hdot(n, e[1])), std::fabs(hdot(n, e[2])));
  return dev <= 1e-5f * scale;
}

// Axis-aligned rectangle detection for the bit-identical specialised test (B2AAQuad, aa_quad_hit): E01 and E23
// must have exactly one non-zero component u, E03 and E21 exactly one non-zero component v != u.
bool classify_axis_aligned(const B2Quad& Q, int slot, B2AAQuad& A)
{
  std::memset(&A, 0, sizeof(A));
  A.cls = -1;
  A.slot = slot;
  A.prim = Q.prim;
  auto single_axis = [](const float* e) -> int {
    int axis = -1;
    for (int c = 0; c < 3; ++c)
      if (e[c] != 0.f)
      {
        if (axis >= 0)
          return -1;
        axis = c;
      }
    return axis;
  };
  const int u = single_axis(Q.e01), v = single_axis(Q.e03);
  if (u < 0 || v < 0 || u == v || single_axis(Q.e23) != u || single_axis(Q.e21) != v)
    return false;
  const int n = 3 - u - v;
  static const int clsOf[3][3] = { { -1, 0, 4 }, { 3, -1, 1 }, { 2, 5, -1 } }; // [u][v]
  A.cls = clsOf[u][v];
  const float eps = (A.cls < 3) ? 1.f : -1.f; // +1 for cyclic (u,v,n)
  const float a = Q.e01[u], b = Q.e03[v], a2 = Q.e23[u], b2 = Q.e21[v];
  A.v00u = Q.v00[u], A.v00v = Q.v00[v], A.v00n = Q.v00[n];
  A.v11u = Q.v11[u], A.v11v = Q.v11[v], A.v11n = Q.v11[n];
  A.a = a, A.b = b, A.a2 = a2;
  A.bPu = -eps * b, A.bPn = eps * b, A.aQv = eps * a, A.aQn = -eps * a;
  A.b2Pu = -eps * b2, A.b2Pn = eps * b2, A.a2Qv = eps * a2, A.a2Qn = -eps * a2;
  // consistent rectangle: the second triangle's frame is the first one's mirrored about the centre
  const bool rect = a2 == -a && b2 == -b && std::fabs((Q.v00[u] + a) - Q.v11[u]) <= 2e-6f * std::fabs(a) &&
    std::fabs((Q.v00[v] + b) - Q.v11[v]) <= 2e-6f * std::fabs(b) && Q.v00[n] == Q.v11[n];
  if (rect)
    A.cls |= 8;
  return true;
}

bool same_vertices(const B2Quad& a, const B2Quad& b)
{
  return std::memcmp(a.v00, b.v00, 12) == 0 && std::memcmp(a.e01, b.e01, 12) == 0 &&
    std::memcmp(a.e03, b.e03, 12) == 0 && std::memcmp(a.v11, b.v11, 12) == 0 && std::memcmp(a.e21, b.e21, 12) == 0 &&
    std::memcmp(a.e23, b.e23, 12) == 0;
}

} // namespace

// 64-bit multiplicative hash over 4-byte words (every hashed table is an array of 4-byte fields without holes)
static uint64_t hash_words(const void* data, size_t bytes, uint64_t h)
{
  const uint32_t* w = static_cast<const uint32_t*>(data);
  for (size_t i = 0; i < bytes / 4; ++i)
  {
    h = (h ^ w[i]) * 0x9E3779B97F4A7C15ull;
    h ^= h >> 29;
  }
  return h;
}

extern "C"
{

int b2pt_version(void) { return 100; }

const char* b2pt_last_error(void) { return g_lastError.c_str(); }

static cudaError_t create_sets(b2pt_ctx* ctx)
{
  for (int k = 0; k < b2pt_ctx::kMaxSets; ++k)
  {
    cudaError_t e;
    if (k > 0 && (e = cudaStreamCreateWithFlags(&ctx->extra[k], cudaStreamNonBlocking)) != cudaSuccess)
      return e;
    if ((e = cudaEventCreateWithFlags(&ctx->evJoin[k], cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->evAcc[k], cudaEventDisableTiming)) != cudaSuccess)
      return e;
  }
  return cudaSuccess;
}

b2pt_ctx* b2pt_create(int device, int* err)
{
  auto bail = [&](int code) -> b2pt_ctx* {
    if (err)
      *err = code;
    return nullptr;
  };
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
  {
    fail(B2PT_ERR_CUDA, "no CUDA device available (%s); libb2pt has no CPU fallback",
         e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return bail(B2PT_ERR_CUDA);
  }
  if (device < 0 || device >= count)
  {
    fail(B2PT_ERR_BAD_VALUE, "device %d out of range [0,%d)", device, count);
    return bail(B2PT_ERR_BAD_VALUE);
  }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
  {
    fail(B2PT_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    return bail(B2PT_ERR_CUDA);
  }
  if (prop.major != 10)
  {
    fail(B2PT_ERR_CUDA, "device %d is sm_%d%d; libb2pt ships sm_100a code only", device, prop.major, prop.minor);
    return bail(B2PT_ERR_CUDA);
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess)
  {
    fail(B2PT_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    return bail(B2PT_ERR_CUDA);
  }
  b2pt_ctx* ctx = new b2pt_ctx();
  ctx->device = device;
  if ((e = cudaStreamCreateWithFlags(&ctx->ownStream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->evStart)) != cudaSuccess || (e = cudaEventCreate(&ctx->evStop)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->evFork, cudaEventDisableTiming)) != cudaSuccess ||
      (e = create_sets(ctx)) != cudaSuccess ||
      (e = b2pt::query_launch_cfg(&ctx->cfg)) != cudaSuccess)
  {
    fail(B2PT_ERR_CUDA, "context set-up failed: %s", cudaGetErrorString(e));
    delete ctx;
    return bail(B2PT_ERR_CUDA);
  }
  ctx->stream = ctx->ownStream;
  if (err)
    *err = B2PT_OK;
  return ctx;
}

void b2pt_destroy(b2pt_ctx* ctx)
{
  if (!ctx)
    return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (cudaStream_t st : ctx->extra)
    if (st)
      cudaStreamSynchronize(st);
  ctx->dNodes.release(), ctx->dWide.release(), ctx->dParent.release(), ctx->dArrived.release(), ctx->dSlots.release(), ctx->dBinSlots.release(), ctx->dLeafSph.release(), ctx->dQuads.release(), ctx->dSph.release(), ctx->dGates.release();
  ctx->colorOwn.release();
  for (auto& b : ctx->bufs)
    b.release_all();
  ctx->counters.release(), ctx->binTotals.release(), ctx->seeds.release(), ctx->nanCounter.release();
  ctx->dViews.release(), ctx->viewColor.release(), ctx->pnm.release(), ctx->primMask.release(), ctx->primQuads.release(); // (DevBuf's destructor would free them too)
  ctx->ckptSnap.release(), ctx->ckptMoment.release(), ctx->featAlbedo.release(), ctx->featNormalDepth.release();
  ctx->dnX[0].release(), ctx->dnX[1].release(), ctx->dnGuideA.release(), ctx->dnGuideNZ.release();
  ctx->dDirectViews.release(), ctx->directNormals.release(), ctx->directAlbedo.release(), ctx->directDepth.release(),
    ctx->directPrim.release();
  if (ctx->evFork)
    cudaEventDestroy(ctx->evFork);
  for (int k = 0; k < b2pt_ctx::kMaxSets; ++k)
  {
    if (ctx->evJoin[k])
      cudaEventDestroy(ctx->evJoin[k]);
    if (ctx->evAcc[k])
      cudaEventDestroy(ctx->evAcc[k]);
    if (ctx->extra[k])
      cudaStreamDestroy(ctx->extra[k]);
  }
  if (ctx->evStart)
    cudaEventDestroy(ctx->evStart);
  if (ctx->evStop)
    cudaEventDestroy(ctx->evStop);
  for (cudaEvent_t ev : ctx->evBounce)
    if (ev)
      cudaEventDestroy(ev);
  for (cudaEvent_t ev : ctx->evMid)
    if (ev)
      cudaEventDestroy(ev);
  if (ctx->ownStream)
    cudaStreamDestroy(ctx->ownStream);
  delete ctx;
}

int b2pt_set_stream(b2pt_ctx* ctx, void* cudaStream)
{
  if (int rc = bind(ctx))
    return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->stream = cudaStream ? static_cast<cudaStream_t>(cudaStream) : ctx->ownStream;
  return B2PT_OK;
}

int b2pt_set_scene(b2pt_ctx* ctx, const float* pts, int64_t nPts, const int64_t* quadIds, int64_t nQuads,
                   const int64_t* spherePt, const float* sphereR, int64_t nSpheres, const int64_t* matIdxQuad,
                   const int64_t* texIdxQuad, const int64_t* matIdxSph, const int64_t* texIdxSph, const int* matType,
                   int nMatType, const int* texType, int nTexType, const float* tex, int nTex,
                   const int64_t* lightQuadIds, int nLightQuads, const int64_t* lightSpherePt,
                   const float* lightSphereR, int nLightSpheres, int lightables, float refIdx)
{
  if (int rc = bind(ctx))
    return rc;
  if (!pts || nPts <= 0 || nQuads < 0 || nSpheres < 0 || (nQuads + nSpheres) == 0)
    return fail(B2PT_ERR_BAD_VALUE, "scene needs points and at least one primitive");
  if ((nQuads && (!quadIds || !matIdxQuad || !texIdxQuad)) ||
      (nSpheres && (!spherePt || !sphereR || !matIdxSph || !texIdxSph)))
    return fail(B2PT_ERR_BAD_VALUE, "null primitive array");
  if (!matType || !texType || !tex || nMatType <= 0 || nTexType <= 0 || nTex <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "null or empty material tables");
  if (nLightQuads < 0 || nLightQuads > B2PT_MAX_LIGHT_QUADS || nLightSpheres < 0 ||
      nLightSpheres > B2PT_MAX_LIGHT_SPH)
    return fail(B2PT_ERR_BAD_VALUE, "at most %d light quads and %d light spheres are supported",
                B2PT_MAX_LIGHT_QUADS, B2PT_MAX_LIGHT_SPH);
  if ((nLightQuads && !lightQuadIds) || (nLightSpheres && (!lightSpherePt || !lightSphereR)))
    return fail(B2PT_ERR_BAD_VALUE, "null light array");
  if (lightables <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "lightables must be positive");
  if (nQuads + nSpheres > 0x7fffff00LL)
    return fail(B2PT_ERR_BAD_VALUE, "too many primitives");

  auto P = [&](int64_t i) -> H3 { return { pts[3 * i], pts[3 * i + 1], pts[3 * i + 2] }; };
  auto material = [&](int64_t m, int64_t t, int32_t& kind, float* alb) -> bool {
    if (m < 0 || m >= nMatType || t < 0 || t >= nTexType)
      return false;
    const int tt = texType[t];
    if (tt < 0 || tt >= nTex)
      return false;
    kind = matType[m];
    alb[0] = tex[3 * tt], alb[1] = tex[3 * tt + 1], alb[2] = tex[3 * tt + 2];
    return true;
  };

  std::vector<B2Quad> quads((size_t)nQuads);
  std::vector<B2GateBox> gates;
  std::vector<B2GateBox> boxes((size_t)nQuads);
  for (int64_t q = 0; q < nQuads; ++q)
  {
    const int64_t* id = quadIds + 5 * q;
    for (int k = 1; k <= 4; ++k)
      if (id[k] < 0 || id[k] >= nPts)
        return fail(B2PT_ERR_BAD_VALUE, "quad %lld references point %lld outside [0,%lld)", (long long)q,
                    (long long)id[k], (long long)nPts);
    B2Quad& Q = quads[(size_t)q];
    precompute_quad(Q, P(id[1]), P(id[2]), P(id[3]), P(id[4]));
    Q.gate = 0;
    Q.pad[0] = 0;
    B2GateBox G;
    quad_leaf_box(G, P(id[1]), P(id[2]), P(id[3]), P(id[4]));
    G.quad = (int32_t)q;
    boxes[(size_t)q] = G;
    if (!quad_is_planar(P(id[1]), P(id[2]), P(id[3]), P(id[4]), Q.nrm))
    {
      gates.push_back(G);
      Q.gate = (int32_t)gates.size();
      Q.pad[0] = 1; // non-planar: the leaf box is part of the acceptance rule
    }
    if (!material(matIdxQuad[q], texIdxQuad[q], Q.kind, Q.alb))
      return fail(B2PT_ERR_BAD_VALUE, "quad %lld has material/texture index out of range", (long long)q);
    Q.prim = (int32_t)q;
    Q.mat = (int32_t)matIdxQuad[q];
    Q.texi = (int32_t)texIdxQuad[q];
  }
  std::vector<B2Sphere> sph((size_t)nSpheres);
  for (int64_t s = 0; s < nSpheres; ++s)
  {
    if (spherePt[s] < 0 || spherePt[s] >= nPts)
      return fail(B2PT_ERR_BAD_VALUE, "sphere %lld references a point out of range", (long long)s);
    B2Sphere& S = sph[(size_t)s];
    hst(S.c, P(spherePt[s]));
    S.r = sphereR[s];
    if (!material(matIdxSph[s], texIdxSph[s], S.kind, S.alb))
      return fail(B2PT_ERR_BAD_VALUE, "sphere %lld has material/texture index out of range", (long long)s);
    S.prim = (int32_t)(nQuads + s);
    S.mat = (int32_t)matIdxSph[s];
    S.texi = (int32_t)texIdxSph[s];
    S.pad = 0;
  }
  B2Lights L{};
  L.nLightQuads = nLightQuads;
  L.nLightSph = nLightSpheres;
  L.weight = (float)(1.0 / (double)(float)lightables); // PdfWorklet.h:294: float weight = 1.0/list_size
  L.refIdx = refIdx;
  for (int l = 0; l < nLightQuads; ++l)
  {
    const int64_t* id = lightQuadIds + 5 * l;
    for (int k = 1; k <= 4; ++k)
      if (id[k] < 0 || id[k] >= nPts)
        return fail(B2PT_ERR_BAD_VALUE, "light quad %d references a point out of range", l);
    B2LightQuad& LQ = L.lq[l];
    std::memset(&LQ, 0, sizeof(LQ));
    H3 q = P(id[1]), r = P(id[2]), s = P(id[3]), t = P(id[4]);
    precompute_quad(LQ.geo, q, r, s, t);
    LQ.geo.prim = -1;
    LQ.geo.gate = 0; // QuadPDFWorklet calls the leaf intersector directly, no BVH (PdfWorklet.h:238)
    classify_axis_aligned(LQ.geo, 0, LQ.aa);
    H3 rq = hsub(r, q), tq = hsub(t, q);
    LQ.area = std::sqrt(hdot(rq, rq)) * std::sqrt(hdot(tq, tq)); // PdfWorklet.h:236-239
    hst(LQ.pt1, q);                                              // PdfWorklet.h:124-125
    hst(LQ.pt2, s);
  }
  for (int l = 0; l < nLightSpheres; ++l)
  {
    if (lightSpherePt[l] < 0 || lightSpherePt[l] >= nPts)
      return fail(B2PT_ERR_BAD_VALUE, "light sphere %d references a point out of range", l);
    hst(L.ls[l].c, P(lightSpherePt[l]));
    L.ls[l].r = lightSphereR[l];
  }
  ctx->sphPointIds.assign(spherePt, spherePt + (nSpheres ? nSpheres : 0));
  ctx->lightSphPointIds.assign(lightSpherePt, lightSpherePt + (nLightSpheres ? nLightSpheres : 0));
  ctx->quads.swap(quads);
  ctx->sph.swap(sph);
  ctx->gates.swap(gates);
  ctx->boxes.swap(boxes);
  ctx->lights = L;
  ctx->nQuads = nQuads;
  ctx->nSph = nSpheres;
  ctx->haveScene = true;
  ctx->haveBvh = false;
  // The tail-mode depths are cached per scene CONTENT: setting the same scene again (a caller that re-uploads its
  // scene for every frame) keeps them, so the render does not pay the one stream synchronisation that measures them.
  uint64_t h = hash_words(ctx->quads.data(), ctx->quads.size() * sizeof(B2Quad), 0x9E3779B97F4A7C15ull);
  h = hash_words(ctx->sph.data(), ctx->sph.size() * sizeof(B2Sphere), h);
  h = hash_words(ctx->gates.data(), ctx->gates.size() * sizeof(B2GateBox), h);
  h = hash_words(&ctx->lights, sizeof(B2Lights), h);
  if (h != ctx->sceneHash || ctx->sceneVersion == 0)
    ++ctx->sceneVersion;
  ctx->sceneHash = h;
  return B2PT_OK;
}

static constexpr uint32_t kBuildFlags = B2PT_BUILD_FLAGS;

// B2PT_VALIDATE_BVH debug self-check of the binary tree on the device, after a build and after a refit: every primitive
// reachable exactly once, its padded box inside the boxes of all its ancestors.
static int validate_binary_tree(b2pt_ctx* ctx, size_t nNodes)
{
  if (!getenv("B2PT_VALIDATE_BVH") || nNodes == 0)
    return B2PT_OK;
  CU(cudaStreamSynchronize(ctx->stream));
  const size_t nSlots = ctx->treeSlots;
  std::vector<B2BvhNode> hn(nNodes);
  std::vector<int32_t> hs(nSlots);
  CU(cudaMemcpy(hn.data(), ctx->dNodes.p, nNodes * sizeof(B2BvhNode), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(hs.data(), ctx->dSlots.p, nSlots * sizeof(int32_t), cudaMemcpyDeviceToHost));
  std::vector<int> seen(nSlots, 0);
  struct W
  {
    int32_t node;
    float lo[3], hi[3];
  };
  std::vector<W> st;
  W r{};
  r.node = 0;
  for (int c = 0; c < 3; ++c)
    r.lo[c] = hn[0].bmin[c], r.hi[c] = hn[0].bmax[c];
  st.push_back(r);
  size_t bad = 0, visited = 0;
  while (!st.empty())
  {
    const W w = st.back();
    st.pop_back();
    const B2BvhNode& nd = hn[(size_t)w.node];
    for (int c = 0; c < 3; ++c)
      if (nd.bmin[c] < w.lo[c] || nd.bmax[c] > w.hi[c])
        ++bad;
    if (nd.count > 0)
    {
      for (int k = 0; k < nd.count; ++k)
      {
        const int32_t enc = hs[(size_t)nd.left + k];
        ++seen[(size_t)nd.left + k];
        ++visited;
        float a[3], b[3];
        if (enc >= 0)
          b2pt::quad_aabb(ctx->quads[(size_t)enc], a, b);
        else
          b2pt::sphere_aabb(ctx->sph[(size_t)(~enc)], a, b);
        for (int c = 0; c < 3; ++c)
          if (a[c] < nd.bmin[c] || b[c] > nd.bmax[c])
            ++bad;
      }
    }
    else
      for (int k = 0; k < 2; ++k)
      {
        W ch{};
        ch.node = nd.left + k;
        for (int c = 0; c < 3; ++c)
          ch.lo[c] = nd.bmin[c], ch.hi[c] = nd.bmax[c];
        st.push_back(ch);
      }
  }
  size_t once = 0;
  for (int v : seen)
    once += v == 1;
  if (bad || once != nSlots || visited != nSlots)
    return fail(B2PT_ERR_STATE, "BVH validation failed: %zu box violations, %zu of %zu slots reached once", bad, once,
                nSlots);
  return B2PT_OK;
}

static int build_trace_structures(b2pt_ctx* ctx, uint32_t flags)
{
  ctx->haveParents = false;
  ctx->treeStale = false;
  ctx->builtFlags = flags & kBuildFlags;
  // Drop bit-identical duplicate quads: a later copy computes the same t and loses the strict t<tmax
  // comparison (Surface.h:178-179), so removing it cannot change any result.
  std::vector<int32_t> keptQuads;
  for (int64_t q = 0; q < ctx->nQuads; ++q)
  {
    bool dup = false;
    if (!(flags & B2PT_FLAG_NO_DEDUP) && ctx->nQuads <= 4096)
      for (int32_t k : keptQuads)
        if (same_vertices(ctx->quads[(size_t)k], ctx->quads[(size_t)q]))
        {
          dup = true;
          break;
        }
    if (!dup)
      keptQuads.push_back((int32_t)q);
  }
  ctx->tracedQuads = (int32_t)keptQuads.size();
  ctx->tracedSph = (int32_t)ctx->nSph;
  // classify: planar quads normal to an axis of one of up to B2PT_MAX_FRAMES frames go through the candidate
  // filter (b2pt_types.h B2FiltQuad); every other quad is traced behind its leaf box
  struct FiltRec
  {
    float c, uc, hu, vc, hv;
  };
  struct FiltEntry
  {
    int frame, axis;
    FiltRec fq;
    int32_t quad;
    bool exact; // world frame and all four vertices share the float plane coordinate (B2Frame::eaCoef)
  };
  std::vector<FiltEntry> filt;
  std::vector<B2Frame> frames;
  std::vector<int32_t> boxedPlanar, boxedNonPlanar;
  float sceneAbs = 0.f;
  for (int32_t k : keptQuads)
  {
    const B2Quad& Q = ctx->quads[(size_t)k];
    for (int c = 0; c < 3; ++c)
    {
      const float vs[4] = { Q.v00[c], Q.v00[c] + Q.e01[c], Q.v11[c], Q.v00[c] + Q.e03[c] };
      for (float v : vs)
        sceneAbs = std::fmax(sceneAbs, std::fabs(v));
    }
  }
  for (const B2Sphere& sp : ctx->sph)
    for (int c = 0; c < 3; ++c)
      sceneAbs = std::fmax(sceneAbs, std::fabs(sp.c[c]) + std::fabs(sp.r));
  {
    B2Frame F0{};
    F0.R[0] = F0.R[4] = F0.R[8] = 1.f;
    F0.identity = 1;
    frames.push_back(F0);
  }
  auto quad_vertices = [&](const B2Quad& Q, double v[4][3]) {
    for (int c = 0; c < 3; ++c)
    {
      v[0][c] = Q.v00[c];
      v[1][c] = (double)Q.v00[c] + (double)Q.e01[c];
      v[2][c] = Q.v11[c];
      v[3][c] = (double)Q.v00[c] + (double)Q.e03[c];
    }
  };
  // frame coordinates of the four vertices; fits if the extent along one frame axis is <= 1e-6 * scale
  auto try_frame = [&](const B2Frame& F, const B2Quad& Q, FiltEntry& E) -> bool {
    double v[4][3], w[4][3];
    quad_vertices(Q, v);
    for (int k = 0; k < 4; ++k)
      for (int a = 0; a < 3; ++a)
        w[k][a] = (double)F.R[3 * a + 0] * (v[k][0] - F.org[0]) + (double)F.R[3 * a + 1] * (v[k][1] - F.org[1]) +
          (double)F.R[3 * a + 2] * (v[k][2] - F.org[2]);
    const double scale = std::max<double>(sceneAbs, 1e-30);
    for (int n = 0; n < 3; ++n)
    {
      double lo[3], hi[3];
      for (int a = 0; a < 3; ++a)
      {
        lo[a] = hi[a] = w[0][a];
        for (int k = 1; k < 4; ++k)
          lo[a] = std::min(lo[a], w[k][a]), hi[a] = std::max(hi[a], w[k][a]);
      }
      if (hi[n] - lo[n] > 1e-6 * scale)
        continue;
      const int u = (n + 1) % 3, vv = (n + 2) % 3;
      // static margin: the exact test's own edge tolerance (1e-5 of the edge length, DESIGN.md) and the
      // plane-offset spread, doubled
      const double mu = 2e-5 * (hi[u] - lo[u]) + 2e-6 * scale, mv = 2e-5 * (hi[vv] - lo[vv]) + 2e-6 * scale;
      E.axis = n;
      E.exact = F.identity != 0 && hi[n] == lo[n];
      E.fq = FiltRec{};
      E.fq.c = (float)(0.5 * (lo[n] + hi[n]));
      E.fq.uc = (float)(0.5 * (lo[u] + hi[u]));
      E.fq.hu = (float)(0.5 * (hi[u] - lo[u]) + mu);
      E.fq.vc = (float)(0.5 * (lo[vv] + hi[vv]));
      E.fq.hv = (float)(0.5 * (hi[vv] - lo[vv]) + mv);
      return true;
    }
    return false;
  };
  for (int32_t k : keptQuads)
  {
    const B2Quad& Q = ctx->quads[(size_t)k];
    bool placed = false;
    const double area2 = (double)hdot({ Q.e01[0], Q.e01[1], Q.e01[2] }, { Q.e01[0], Q.e01[1], Q.e01[2] }) *
      (double)hdot({ Q.e03[0], Q.e03[1], Q.e03[2] }, { Q.e03[0], Q.e03[1], Q.e03[2] });
    const bool sane = area2 > 0.0 && area2 < 1e30 && std::isfinite(area2);
    if (Q.pad[0] == 0 && sane && !(flags & B2PT_FLAG_NO_AA_DEV) && filt.size() < B2PT_MAX_FILT)
    {
      FiltEntry E{};
      E.quad = k;
      for (size_t f = 0; f < frames.size() && !placed; ++f)
        if (try_frame(frames[f], Q, E))
        {
          E.frame = (int)f;
          placed = true;
        }
      if (!placed && frames.size() < B2PT_MAX_FRAMES)
      { // new frame from this quad: n = unit normal, u = E01 direction, v = n x u
        const double n[3] = { Q.nrm[0], Q.nrm[1], Q.nrm[2] };
        double u[3] = { Q.e01[0], Q.e01[1], Q.e01[2] };
        const double un = u[0] * n[0] + u[1] * n[1] + u[2] * n[2];
        for (int c = 0; c < 3; ++c)
          u[c] -= un * n[c];
        const double ul = std::sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        const double nl = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        if (ul > 0 && nl > 0)
        {
          B2Frame Fn{};
          double w[3];
          for (int c = 0; c < 3; ++c)
            u[c] /= ul;
          w[0] = (n[1] * u[2] - n[2] * u[1]) / nl, w[1] = (n[2] * u[0] - n[0] * u[2]) / nl,
          w[2] = (n[0] * u[1] - n[1] * u[0]) / nl;
          for (int c = 0; c < 3; ++c)
          {
            Fn.R[c] = (float)(n[c] / nl);
            Fn.R[3 + c] = (float)u[c];
            Fn.R[6 + c] = (float)w[c];
            Fn.org[c] = Q.v00[c];
          }
          Fn.identity = 0;
          if (try_frame(Fn, Q, E))
          {
            frames.push_back(Fn);
            E.frame = (int)frames.size() - 1;
            placed = true;
          }
        }
      }
      if (placed)
        filt.push_back(E);
    }
    if (!placed)
      (Q.pad[0] ? boxedNonPlanar : boxedPlanar).push_back(k);
  }
  std::stable_sort(filt.begin(), filt.end(), [](const FiltEntry& x, const FiltEntry& y) {
    return x.frame != y.frame ? x.frame < y.frame : x.axis < y.axis;
  });
  { // the filter holds B2PT_MAX_PAIRS pairs; quads that do not fit go behind their leaf box like any other
    int pairs = 0;
    size_t keep = 0, k = 0;
    while (k < filt.size())
    {
      size_t e = k;
      while (e < filt.size() && filt[e].frame == filt[k].frame && filt[e].axis == filt[k].axis)
        ++e;
      const int room = 2 * (B2PT_MAX_PAIRS - pairs);
      const size_t take = std::min<size_t>(e - k, (size_t)std::max(room, 0));
      pairs += (int)((take + 1) / 2);
      keep = k + take;
      if (take < e - k)
        break;
      k = e;
    }
    for (size_t i = keep; i < filt.size(); ++i)
      boxedPlanar.push_back(filt[i].quad);
    filt.resize(keep);
    std::sort(boxedPlanar.begin(), boxedPlanar.end());
  }
  const size_t nBoxed = boxedPlanar.size() + boxedNonPlanar.size();
  const bool fitsSmall = keptQuads.size() <= B2PT_SMALL_MAX_QUADS && ctx->nSph <= B2PT_SMALL_MAX_SPH &&
    nBoxed <= B2PT_SMALL_MAX_GATES;
  ctx->useBvh = !fitsSmall || (flags & B2PT_FLAG_FORCE_BVH);
  ctx->bvhNodes = 0;
  if (!ctx->useBvh)
  {
    B2SmallScene& S = ctx->small;
    std::memset(&S, 0, sizeof(S));
    S.nQuads = (int32_t)keptQuads.size();
    S.nSph = (int32_t)ctx->nSph;
    S.nFilt = (int32_t)filt.size();
    S.firstBoxed = (int32_t)filt.size();
    S.sceneAbs = sceneAbs;
    // frames without quads are dropped (frame 0 may be empty); within a frame quads are grouped by axis and
    // stored two per B2FiltPair, odd groups padded with a never-matching half
    std::vector<int> frameMap(frames.size(), -1);
    S.nFrames = 0;
    int nPairs = 0;
    size_t k = 0;
    while (k < filt.size())
    {
      size_t e = k;
      while (e < filt.size() && filt[e].frame == filt[k].frame && filt[e].axis == filt[k].axis)
        ++e;
      int& fm = frameMap[(size_t)filt[k].frame];
      if (fm < 0)
      {
        fm = S.nFrames++;
        S.frames[fm] = frames[(size_t)filt[k].frame];
        for (int a = 0; a < 3; ++a)
          S.frames[fm].axisEnd[a] = nPairs, S.frames[fm].eaCoef[a] = 4e-6f;
      }
      {
        bool exact = true;
        for (size_t i = k; i < e; ++i)
          exact = exact && filt[i].exact;
        S.frames[fm].eaCoef[filt[k].axis] = exact ? 4e-7f : 4e-6f;
      }
      for (size_t i = k; i < e; i += 2)
      {
        B2FiltPair& P = S.pairs[nPairs];
        for (int h = 0; h < 2; ++h)
        {
          const bool real = i + h < e;
          const FiltRec r = real ? filt[i + h].fq : FiltRec{ std::nanf(""), 0.f, -1.f, 0.f, -1.f };
          P.c[h] = r.c, P.uc[h] = r.uc, P.hu[h] = r.hu, P.vc[h] = r.vc, P.hv[h] = r.hv;
          P.vis[h] = (uint32_t)(2 * nPairs + h);
          S.visitSlot[2 * nPairs + h] = real ? (int32_t)(i + h) : -1;
        }
        ++nPairs;
      }
      for (int a = filt[k].axis; a < 3; ++a)
        S.frames[fm].axisEnd[a] = nPairs;
      k = e;
    }
    S.nVisit = 2 * nPairs;
    { // byte ranges of the axis groups (B2Frame::grpBegin / grpEnd)
      int begin = 0;
      for (int f = 0; f < S.nFrames; ++f)
        for (int a = 0; a < 3; ++a)
        {
          const int end = std::max(begin, S.frames[f].axisEnd[a]);
          S.frames[f].grpBegin[a] = (uint32_t)(begin * (int)sizeof(B2FiltPair));
          S.frames[f].grpEnd[a] = (uint32_t)(end * (int)sizeof(B2FiltPair));
          begin = end;
        }
    }
    for (size_t i = 0; i < filt.size(); ++i)
      S.quads[i] = ctx->quads[(size_t)filt[i].quad]; // slot = position in the (frame, axis)-sorted list
    size_t slot = filt.size();
    for (int pass = 0; pass < 2; ++pass) // planar boxed quads first, non-planar last (DESIGN.md "leaf-box gate")
      for (int32_t k : (pass == 0 ? boxedPlanar : boxedNonPlanar))
      {
        S.quads[slot] = ctx->quads[(size_t)k];
        S.gate[S.nGate] = ctx->boxes[(size_t)k];
        S.gate[S.nGate].quad = (int32_t)slot;
        S.quads[slot].gate = ++S.nGate;
        ++slot;
      }
    for (int64_t s = 0; s < ctx->nSph; ++s)
    {
      const B2Sphere& sp = ctx->sph[(size_t)s];
      ctx->small.sph[s] = sp;
      B2GateBox& G = ctx->small.sphGate[s]; // FindSphereAABBs (AABBSurface.h:82-174): centre +- radius, unpadded
      for (int c = 0; c < 3; ++c)
      {
        G.bmin[c] = std::fmin(sp.c[c] + sp.r, sp.c[c] - sp.r);
        G.bmax[c] = std::fmax(sp.c[c] + sp.r, sp.c[c] - sp.r);
      }
      G.quad = -1;
      G.pad = 0;
    }
    return B2PT_OK;
  }
  for (int c = 0; c < 3; ++c)
    ctx->sortLo[c] = FLT_MAX, ctx->sortHi[c] = -FLT_MAX;
  for (int32_t k : keptQuads)
  {
    float a[3], b[3];
    b2pt::quad_aabb(ctx->quads[(size_t)k], a, b);
    for (int c = 0; c < 3; ++c)
      ctx->sortLo[c] = std::fmin(ctx->sortLo[c], a[c]), ctx->sortHi[c] = std::fmax(ctx->sortHi[c], b[c]);
  }
  for (const B2Sphere& sp : ctx->sph)
    for (int c = 0; c < 3; ++c)
      ctx->sortLo[c] = std::fmin(ctx->sortLo[c], sp.c[c] - sp.r), ctx->sortHi[c] = std::fmax(ctx->sortHi[c], sp.c[c] + sp.r);
  std::vector<B2BvhNode> nodes;
  std::vector<int32_t> slots;
  std::vector<int32_t> treeQuads; // gated quads stay out of the tree (tested after the traversal)
  for (int32_t k : keptQuads)
    if (ctx->quads[(size_t)k].gate == 0)
      treeQuads.push_back(k);
  CU(ctx->dQuads.reserve(std::max<size_t>(ctx->quads.size(), 1)));
  CU(ctx->dSph.reserve(std::max<size_t>(ctx->sph.size(), 1)));
  CU(ctx->dGates.reserve(std::max<size_t>(ctx->gates.size(), 1)));
  if (!ctx->gates.empty())
    CU(cudaMemcpyAsync(ctx->dGates.p, ctx->gates.data(), ctx->gates.size() * sizeof(B2GateBox),
                       cudaMemcpyHostToDevice, ctx->stream));
  if (!ctx->quads.empty())
    CU(cudaMemcpyAsync(ctx->dQuads.p, ctx->quads.data(), ctx->quads.size() * sizeof(B2Quad), cudaMemcpyHostToDevice,
                       ctx->stream));
  if (!ctx->sph.empty())
    CU(cudaMemcpyAsync(ctx->dSph.p, ctx->sph.data(), ctx->sph.size() * sizeof(B2Sphere), cudaMemcpyHostToDevice,
                       ctx->stream));
  size_t nNodes = 0;
  if (flags & B2PT_FLAG_GPU_LBVH)
  { // device builder (b2pt_lbvh.cu): Morton order, radix tree, leaves of <= 4 primitives
    const size_t n = treeQuads.size() + ctx->sph.size();
    if (2 * n >= ((size_t)1 << 24))
      return fail(B2PT_ERR_UNSUPPORTED, "scene too large for the 24-bit BVH index packing");
    float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    for (int32_t k : treeQuads)
    {
      float a[3], b[3];
      b2pt::quad_aabb(ctx->quads[(size_t)k], a, b);
      for (int c = 0; c < 3; ++c)
        lo[c] = std::fmin(lo[c], a[c]), hi[c] = std::fmax(hi[c], b[c]);
    }
    for (const B2Sphere& sp : ctx->sph)
      for (int c = 0; c < 3; ++c)
        lo[c] = std::fmin(lo[c], sp.c[c] - sp.r), hi[c] = std::fmax(hi[c], sp.c[c] + sp.r);
    DevBuf<int32_t> dTreeQuads;
    CU(dTreeQuads.reserve(std::max<size_t>(treeQuads.size(), 1)));
    if (!treeQuads.empty())
      CU(cudaMemcpyAsync(dTreeQuads.p, treeQuads.data(), treeQuads.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                         ctx->stream));
    nNodes = n ? 2 * n : 0;
    CU(ctx->dNodes.reserve(std::max<size_t>(nNodes, 1)));
    CU(ctx->dSlots.reserve(std::max<size_t>(n, 1)));
    CU(ctx->dLeafSph.reserve(std::max<size_t>(n, 1)));
    const cudaError_t le = b2pt::build_lbvh_device(ctx->dQuads.p, ctx->dSph.p, dTreeQuads.p, (int)treeQuads.size(),
                                                   (int)ctx->sph.size(), lo, hi, ctx->dNodes.p, ctx->dSlots.p,
                                                   ctx->dLeafSph.p, ctx->stream);
    dTreeQuads.release();
    CU(le);
  }
  else
  {
    int binDepth = 0;
    if (!b2pt::build_bvh(ctx->quads, treeQuads, ctx->sph, nodes, slots, &binDepth))
      return fail(B2PT_ERR_UNSUPPORTED, "scene too large for the 24-bit BVH index packing");
    if (binDepth > 62) // the traversal stack holds 64 entries (the builder's depth bound keeps real trees far below)
      return fail(B2PT_ERR_UNSUPPORTED, "BVH is %d levels deep; the traversal stack holds 64 entries", binDepth);
    nNodes = nodes.size();
    CU(ctx->dNodes.reserve(std::max<size_t>(nodes.size(), 1)));
    CU(ctx->dSlots.reserve(std::max<size_t>(slots.size(), 1)));
    CU(ctx->dLeafSph.reserve(std::max<size_t>(slots.size(), 1)));
    std::vector<float4> leafSph(slots.size(), make_float4(0.f, 0.f, 0.f, 0.f));
    for (size_t i = 0; i < slots.size(); ++i)
      if (slots[i] < 0)
      {
        const B2Sphere& sp = ctx->sph[(size_t)(~slots[i])];
        leafSph[i] = make_float4(sp.c[0], sp.c[1], sp.c[2], sp.r);
      }
    if (!nodes.empty())
      CU(cudaMemcpyAsync(ctx->dNodes.p, nodes.data(), nodes.size() * sizeof(B2BvhNode), cudaMemcpyHostToDevice,
                         ctx->stream));
    if (!slots.empty())
    {
      CU(cudaMemcpyAsync(ctx->dLeafSph.p, leafSph.data(), leafSph.size() * sizeof(float4), cudaMemcpyHostToDevice,
                         ctx->stream));
      CU(cudaMemcpyAsync(ctx->dSlots.p, slots.data(), slots.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                         ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream)); // host vectors go out of scope
  }
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->treeSlots = treeQuads.size() + ctx->sph.size();
  if (int rc = validate_binary_tree(ctx, nNodes))
    return rc;
  // B2PT_FLAG_WIDE_BVH: the traversal kernels walk the 8-wide compressed tree collapsed from the binary one
  // (b2pt_wide.h); primSlots and leafSph are rewritten in its leaf order.  Opt-in (B2PT_FLAG_WIDE_BVH): the binary tree measured faster.
  ctx->bvh.wide = nullptr;
  ctx->bvh.nWide = 0;
  ctx->bvh.wideDepth = 0;
  if ((flags & B2PT_FLAG_WIDE_BVH) && nNodes > 0)
  {
    const size_t nSlots = treeQuads.size() + ctx->sph.size();
    if (nodes.empty())
    { // device-built tree: bring it to the host for the collapse
      nodes.resize(nNodes);
      slots.resize(nSlots);
      CU(cudaMemcpy(nodes.data(), ctx->dNodes.p, nNodes * sizeof(B2BvhNode), cudaMemcpyDeviceToHost));
      CU(cudaMemcpy(slots.data(), ctx->dSlots.p, nSlots * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    b2pt::WideBuildResult wr;
    if (!b2pt::collapse_to_wide(nodes, slots, ctx->quads, ctx->sph, sceneAbs, wr) || wr.slots.size() != nSlots)
      return fail(B2PT_ERR_STATE, "collapsing the BVH into 8-wide nodes failed");
    if (wr.maxDepth > B2PT_WIDE_STACK)
      return fail(B2PT_ERR_UNSUPPORTED, "8-wide BVH is %d levels deep (limit %d); drop B2PT_FLAG_WIDE_BVH", wr.maxDepth,
                  B2PT_WIDE_STACK);
    if (getenv("B2PT_VALIDATE_BVH"))
    {
      std::string why;
      if (!b2pt::validate_wide(wr, ctx->quads, ctx->sph, why))
        return fail(B2PT_ERR_STATE, "8-wide BVH validation failed: %s", why.c_str());
    }
    static_assert(sizeof(B2WideNode) == 80, "B2WideNode is five 16-byte chunks");
    std::vector<float4> leafSph(nSlots, make_float4(0.f, 0.f, 0.f, 0.f));
    for (size_t i = 0; i < nSlots; ++i)
      if (wr.slots[i] < 0)
      {
        const B2Sphere& sp = ctx->sph[(size_t)(~wr.slots[i])];
        leafSph[i] = make_float4(sp.c[0], sp.c[1], sp.c[2], sp.r);
      }
    CU(ctx->dBinSlots.reserve(nSlots));
    CU(cudaMemcpy(ctx->dBinSlots.p, ctx->dSlots.p, nSlots * sizeof(int32_t), cudaMemcpyDeviceToDevice));
    CU(ctx->dWide.reserve(wr.nodes.size() * 5));
    CU(cudaMemcpy(ctx->dWide.p, wr.nodes.data(), wr.nodes.size() * sizeof(B2WideNode), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->dSlots.p, wr.slots.data(), nSlots * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->dLeafSph.p, leafSph.data(), nSlots * sizeof(float4), cudaMemcpyHostToDevice));
    ctx->bvh.wide = ctx->dWide.p;
    ctx->bvh.nWide = (int32_t)wr.nodes.size();
    ctx->bvh.wideDepth = wr.maxDepth;
  }
  ctx->bvh.nodes = ctx->dNodes.p;
  ctx->bvh.primSlots = ctx->dSlots.p;
  ctx->bvh.leafSph = ctx->dLeafSph.p;
  ctx->bvh.quads = ctx->dQuads.p;
  ctx->bvh.sph = ctx->dSph.p;
  ctx->bvh.gate = ctx->dGates.p;
  ctx->bvh.nGate = (int32_t)ctx->gates.size();
  ctx->bvh.nNodes = (int32_t)nNodes;
  ctx->bvh.nQuads = (int32_t)ctx->quads.size();
  ctx->bvh.nSph = (int32_t)ctx->sph.size();
  ctx->bvhNodes = (int32_t)nNodes;
  return B2PT_OK;
}

int b2pt_build_bvh_ex(b2pt_ctx* ctx, uint32_t flags)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "b2pt_build_bvh before b2pt_set_scene");
  if (int rc = build_trace_structures(
        ctx, flags & (B2PT_FLAG_FORCE_BVH | B2PT_FLAG_NO_DEDUP | B2PT_FLAG_NO_AA | B2PT_FLAG_GPU_LBVH | B2PT_FLAG_WIDE_BVH)))
    return rc;
  ctx->haveBvh = true;
  return B2PT_OK;
}

int b2pt_build_bvh(b2pt_ctx* ctx) { return b2pt_build_bvh_ex(ctx, 0); }

int b2pt_update_spheres(b2pt_ctx* ctx, const float* centers, const float* radii)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "b2pt_update_spheres before b2pt_set_scene");
  if (!centers)
    return fail(B2PT_ERR_BAD_VALUE, "null sphere centres");
  CU(cudaStreamSynchronize(ctx->stream)); // renders in flight still read the old geometry
  for (size_t s = 0; s < ctx->sph.size(); ++s)
  {
    for (int c = 0; c < 3; ++c)
      ctx->sph[s].c[c] = centers[3 * s + c];
    if (radii)
      ctx->sph[s].r = radii[s];
    // a light sphere is a scene sphere referenced by point id (SphereGenerateDir.h / SpherePdf.h): it moves along
    for (size_t l = 0; l < ctx->lightSphPointIds.size(); ++l)
      if (ctx->lightSphPointIds[l] == ctx->sphPointIds[s])
      {
        for (int c = 0; c < 3; ++c)
          ctx->lights.ls[l].c[c] = ctx->sph[s].c[c];
        if (radii)
          ctx->lights.ls[l].r = radii[s];
      }
  }
  ++ctx->sceneVersion;
  if (!ctx->haveBvh)
    return B2PT_OK; // the structures are built from the new geometry anyway
  if (!ctx->useBvh)
  { // kernel-parameter path: the sphere table and the spheres' leaf boxes are the whole "structure"
    for (size_t s = 0; s < ctx->sph.size(); ++s)
    {
      const B2Sphere& sp = ctx->sph[s];
      ctx->small.sph[s] = sp;
      B2GateBox& G = ctx->small.sphGate[s];
      for (int c = 0; c < 3; ++c)
      {
        G.bmin[c] = std::fmin(sp.c[c] + sp.r, sp.c[c] - sp.r);
        G.bmax[c] = std::fmax(sp.c[c] + sp.r, sp.c[c] - sp.r);
      }
    }
    return B2PT_OK;
  }
  if (!ctx->sph.empty())
    CU(cudaMemcpyAsync(ctx->dSph.p, ctx->sph.data(), ctx->sph.size() * sizeof(B2Sphere), cudaMemcpyHostToDevice,
                       ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  // The node boxes and the leaf-ordered sphere copies (leafSph) still hold the old geometry: the next trace refits or
  // rebuilds the tree first (refresh_stale_tree) unless b2pt_refit_bvh does it before.
  ctx->treeStale = true;
  return B2PT_OK;
}

// The binary tree's boxes and leafSph recomputed from the current geometry, topology kept (b2pt_refit_bvh).
static int refit_tree(b2pt_ctx* ctx)
{
  const int nNodes = ctx->bvhNodes;
  if (nNodes <= 0)
  {
    ctx->treeStale = false;
    return B2PT_OK;
  }
  if (!ctx->haveParents)
  { // one-time: parent links of the tree as it sits on the device (either builder's layout)
    std::vector<B2BvhNode> hn((size_t)nNodes);
    CU(cudaMemcpy(hn.data(), ctx->dNodes.p, (size_t)nNodes * sizeof(B2BvhNode), cudaMemcpyDeviceToHost));
    std::vector<int32_t> parent((size_t)nNodes, -2);
    std::vector<int32_t> st(1, 0);
    parent[0] = -1;
    while (!st.empty())
    {
      const int32_t i = st.back();
      st.pop_back();
      if (hn[(size_t)i].count > 0)
        continue;
      for (int k = 0; k < 2; ++k)
      {
        const int32_t c = hn[(size_t)i].left + k;
        if (c <= 0 || c >= nNodes || parent[(size_t)c] != -2)
          return fail(B2PT_ERR_STATE, "b2pt_refit_bvh: malformed tree");
        parent[(size_t)c] = i;
        st.push_back(c);
      }
    }
    CU(ctx->dParent.reserve((size_t)nNodes));
    CU(ctx->dArrived.reserve((size_t)nNodes));
    CU(cudaMemcpy(ctx->dParent.p, parent.data(), (size_t)nNodes * sizeof(int32_t), cudaMemcpyHostToDevice));
    ctx->haveParents = true;
  }
  CU(b2pt::refit_bvh_device(ctx->dNodes.p, ctx->dParent.p, ctx->dArrived.p, nNodes, ctx->dSlots.p, ctx->dQuads.p,
                            ctx->dSph.p, ctx->dLeafSph.p, ctx->stream));
  ctx->treeStale = false;
  return validate_binary_tree(ctx, (size_t)nNodes);
}

int b2pt_refit_bvh(b2pt_ctx* ctx)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveScene || !ctx->haveBvh)
    return fail(B2PT_ERR_STATE, "b2pt_refit_bvh before b2pt_build_bvh");
  if (!ctx->useBvh)
    return B2PT_OK; // no tree on the kernel-parameter path (b2pt_update_spheres refreshed its tables)
  if (ctx->bvh.wide)
    return fail(B2PT_ERR_UNSUPPORTED, "b2pt_refit_bvh refits the binary tree; rebuild when B2PT_FLAG_WIDE_BVH is in use");
  return refit_tree(ctx);
}

// Before a trace: a tree that b2pt_update_spheres left behind the spheres is brought up to date -- the binary tree is
// refitted, the 8-wide tree (which has no refit) rebuilt with the flags it was built with.
static int refresh_stale_tree(b2pt_ctx* ctx)
{
  if (!ctx->treeStale)
    return B2PT_OK;
  return ctx->bvh.wide ? build_trace_structures(ctx, ctx->builtFlags) : refit_tree(ctx);
}

// Camera.cxx:913-914 Look; :803-811 SetUp; RayGen ctor :438-476 with fovX = fovY (:936-938), zoom off.
// Validation messages are the reference's (Camera.cxx:645, 667, 720-724).
static int make_camera(const float pos[3], const float lookAt[3], const float up[3], float fovDeg, int W, int H,
                       B2Camera& c)
{
  if (!pos || !lookAt || !up)
    return fail(B2PT_ERR_BAD_VALUE, "null camera vector");
  if (H <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "Camera height must be greater than zero."); // Camera.cxx:645
  if (W <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "Camera width must be greater than zero."); // Camera.cxx:667
  if (!(fovDeg > 0))
    return fail(B2PT_ERR_BAD_VALUE, "Camera feild of view must be greater than zero."); // Camera.cxx:720
  if (fovDeg > 180)
    return fail(B2PT_ERR_BAD_VALUE, "Camera feild of view must be less than 180."); // Camera.cxx:724
  if ((int64_t)W * H > (int64_t)1 << 26)
    return fail(B2PT_ERR_BAD_VALUE, "canvas larger than 2^26 pixels");
  H3 look = hnormalize(hsub({ lookAt[0], lookAt[1], lookAt[2] }, { pos[0], pos[1], pos[2] }));
  H3 upv = { up[0], up[1], up[2] };
  if (!(upv.x == 0.f && upv.y == 1.f && upv.z == 0.f))
    upv = hnormalize(upv);
  const float pi180 = 0.01745329251994329547f;
  const float thx = std::tan((fovDeg * pi180) * .5f);
  const float thy = std::tan((fovDeg * pi180) * .5f);
  H3 u = hnormalize(hcross(look, upv));
  H3 v = hnormalize(hcross(u, look));
  c = B2Camera{};
  hst(c.dx, hscale(u, 2 * thx / (float)W));
  hst(c.dy, hscale(v, 2 * thy / (float)H));
  hst(c.nlook, hnormalize(look));
  c.pos[0] = pos[0], c.pos[1] = pos[1], c.pos[2] = pos[2];
  c.W = W;
  c.H = H;
  return B2PT_OK;
}

// The up vector as Camera::SetUp (Camera.cxx:803-811) stores it: normalised unless it is exactly (0,1,0).
static void stored_up(const float up[3], float out[3])
{
  H3 upv = { up[0], up[1], up[2] };
  if (!(upv.x == 0.f && upv.y == 1.f && upv.z == 0.f))
    upv = hnormalize(upv);
  hst(out, upv);
}

// Checks of the view-sweep entry points; fn names the entry point in the messages.
static int check_view_list(const char* fn, int nViews, const float* views)
{
  if (nViews < 0 || (nViews > 0 && !views))
    return fail(B2PT_ERR_BAD_VALUE, "%s: bad view list", fn);
  return B2PT_OK;
}

static int check_checkpoints(const char* fn, int nCheckpoints, const int* checkpoints)
{
  if (nCheckpoints < 1 || nCheckpoints > b2pt::kMaxCheckpoints || !checkpoints)
    return fail(B2PT_ERR_BAD_VALUE, "%s: nCheckpoints must be in [1,%d] with a non-NULL list", fn,
                b2pt::kMaxCheckpoints);
  for (int k = 0; k < nCheckpoints; ++k)
    if (checkpoints[k] < 1 || (k > 0 && checkpoints[k] <= checkpoints[k - 1]))
      return fail(B2PT_ERR_BAD_VALUE, "%s: checkpoints must be >= 1 and strictly increasing", fn);
  return B2PT_OK;
}

// The camera of every row (pos[3], lookAt[3], up[3], fovDeg) of a view list, all on a W x H canvas.
static int make_view_cameras(int nViews, const float* views, int W, int H, std::vector<B2Camera>& cams)
{
  cams.resize((size_t)nViews);
  for (int v = 0; v < nViews; ++v)
  {
    const float* p = views + 10 * (size_t)v;
    if (int rc = make_camera(p, p + 3, p + 6, p[9], W, H, cams[(size_t)v]))
      return rc;
  }
  return B2PT_OK;
}

int b2pt_set_camera(b2pt_ctx* ctx, const float pos[3], const float lookAt[3], const float up[3], float fovDeg, int W,
                    int H)
{
  if (int rc = bind(ctx))
    return rc;
  B2Camera c{};
  if (int rc = make_camera(pos, lookAt, up, fovDeg, W, H, c))
    return rc;
  const bool resized = (W != ctx->cam.W || H != ctx->cam.H);
  ctx->cam = c;
  ctx->haveCamera = true;
  stored_up(up, ctx->camUpN);
  for (int k = 0; k < 3; ++k)
    ctx->camLookAt[k] = lookAt[k];
  if (resized && !ctx->colorExt)
    ctx->colorPixels = 0; // force re-allocation + clear
  return B2PT_OK;
}

int b2pt_set_memory_budget(b2pt_ctx* ctx, int64_t bytes)
{
  if (int rc = bind(ctx))
    return rc;
  if (bytes < 0)
    return fail(B2PT_ERR_BAD_VALUE, "negative memory budget");
  ctx->userBudget = bytes;
  return B2PT_OK;
}

int b2pt_seed(b2pt_ctx* ctx, uint32_t seedOffset)
{
  if (int rc = bind(ctx))
    return rc;
  ctx->seedOffset = seedOffset;
  return B2PT_OK;
}

int b2pt_set_color_buffer(b2pt_ctx* ctx, void* deviceFloat4)
{
  if (int rc = bind(ctx))
    return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->colorExt = static_cast<float4*>(deviceFloat4);
  return B2PT_OK;
}

void* b2pt_color_device_ptr(b2pt_ctx* ctx)
{
  if (bind(ctx) != B2PT_OK || !ctx->haveCamera)
    return nullptr;
  if (ensure_color(ctx) != B2PT_OK)
    return nullptr;
  return ctx->color();
}

int b2pt_clear_color(b2pt_ctx* ctx)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_clear_color before b2pt_set_camera");
  if (int rc = ensure_color(ctx))
    return rc;
  CU(cudaMemsetAsync(ctx->color(), 0, sizeof(float4) * (size_t)ctx->cam.W * ctx->cam.H, ctx->stream));
  return B2PT_OK;
}

static int64_t tail_rays_per_warp()
{
  const char* e = getenv("B2PT_TAIL_RAYS_PER_WARP");
  if (e)
  {
    long long v = atoll(e);
    if (v >= 0)
      return v;
  }
  return 512; // below 16 tiles per region the four strategy bins stop filling whole warps (measured flat 256..2048)
}

static int64_t overlap_sets()
{ // B2PT_OVERLAP = number of sample batches in flight (1 = serial), default 4
  const char* e = getenv("B2PT_OVERLAP");
  int64_t v = e ? atoll(e) : 4;
  if (v <= 0)
    v = 1;
  return std::min<int64_t>(v, b2pt_ctx::kMaxSets);
}

static int64_t tail_loop_rays()
{
  const char* e = getenv("B2PT_TAIL_LOOP_RAYS");
  if (e)
  {
    long long v = atoll(e);
    if (v >= 0)
      return v;
  }
  return 24576; // ~break-even between one 8-SM cluster pass and a full-grid launch pair
}

// Bytes of batch buffers per path in flight: one-kernel pipeline = two sets of four bins (52 B records) + radiance
// 16 B; two-kernel pipeline = ray queue 48 B + one set of bins + radiance.
static double bytes_per_path(bool fused) { return fused ? 2 * 4 * 52.0 + 16.0 : 48.0 + 4 * 52.0 + 16.0 + 16.0; } // (+ sort keys, permutation, hits of BVH scenes)

static int64_t batch_target_paths(b2pt_ctx* ctx, bool fused)
{
  const char* e = getenv("B2PT_BATCH_PATHS");
  if (e)
  {
    long long v = atoll(e);
    if (v > 0)
      return v;
  }
  // Up to 128 Mi paths per batch, four batches in flight, inside a memory budget: 0.85 of the memory that is free when
  // the context first renders (before its own buffers exist), or what b2pt_set_memory_budget says.  The card's HBM is
  // there to be used -- larger batches amortise the tail of the bounce loop (measured per 1024-spp step with the
  // two-kernel pipeline: 16 Mi 238.3 ms, 32 Mi 227.2, 64 Mi 220.3, 96 Mi 217.8, 128 Mi 215.1) -- but a co-tenant can
  // cap it.  Folding the four bins of a region into two arrays was measured: each kernel 1.4 % slower.
  if (ctx->memBudget <= 0)
  {
    size_t freeB = 0, totalB = 0;
    ctx->memBudget = cudaMemGetInfo(&freeB, &totalB) == cudaSuccess ? (int64_t)(0.85 * (double)freeB) : ((int64_t)32 << 30);
  }
  const int64_t budget = ctx->userBudget > 0 ? ctx->userBudget : ctx->memBudget;
  int64_t target = (int64_t)((double)budget / (bytes_per_path(fused) * (double)overlap_sets()));
  target = std::min<int64_t>(target, (int64_t)1 << 27);
  target = std::max<int64_t>(target & ~(((int64_t)1 << 20) - 1), (int64_t)1 << 20); // whole Mi paths, at least one
  return target;
}

// Cut `units` (samples of one view, or whole views) of unitPaths paths each into equal batches: as few as
// maxPathsPerBatch allows, but up to one per buffer set while every batch keeps at least 32 Mi paths.
static void plan_batches(int64_t units, int64_t unitPaths, int64_t maxPathsPerBatch, int64_t sets, int64_t& per,
                         int64_t& nBatches)
{
  per = 1;
  nBatches = 0;
  if (units <= 0 || unitPaths <= 0)
    return;
  maxPathsPerBatch = std::min<int64_t>(std::max<int64_t>(maxPathsPerBatch, 1), 0xfffffff0LL);
  const int64_t maxPer = std::max<int64_t>(1, maxPathsPerBatch / unitPaths);
  const int64_t minPer = std::max<int64_t>(1, std::min<int64_t>(maxPer, ((int64_t)1 << 25) / unitPaths));
  int64_t nb = (units + maxPer - 1) / maxPer;
  nb = std::max<int64_t>(nb, std::min<int64_t>(std::max<int64_t>(sets, 1), units / minPer));
  nb = std::max<int64_t>(nb, 1);
  per = (units + nb - 1) / nb;
  nBatches = (units + per - 1) / per;
}

// MapperPathTracer::RenderCellsImpl builds its acceleration structures on every call (:275-276); here
// they are rebuilt only when the scene or the build-affecting flags changed, and brought up to date after
// b2pt_update_spheres (refresh_stale_tree).
static int ensure_built_for(b2pt_ctx* ctx, uint32_t flags)
{
  const uint32_t buildFlags = flags & kBuildFlags;
  if (!ctx->haveBvh || ctx->builtFlags != buildFlags)
  {
    if (int rc = build_trace_structures(ctx, buildFlags))
      return rc;
    ctx->haveBvh = true;
  }
  return refresh_stale_tree(ctx);
}

// A listed round of b2pt_render_views_adaptive: the canvas entries entries[0 .. nReal) (view * viewPixels + pixel,
// padded to nPad by repeating the last one) for the cameras of ctx->dViews; their running sums live in color and
// moment.
struct ListedRound
{
  const uint32_t* entries;
  int64_t nReal, nPad;
  int viewPixels;
  float4 *color, *moment;
};

// One render of the current scene.  nViews == 0: the context's camera, samples [sampleBegin, sampleBegin+sampleCount)
// accumulated into the context's canvas.  nViews > 0 (b2pt_render_views): the same sample range for every camera of
// ctx->dViews, accumulated into ctx->viewColor[view]; a batch holds whole views (viewsPerBatch x sampleCount sample
// slots), so the caller guarantees W*H*sampleCount <= the batch target.  ckpt (b2pt_render_views_checkpoints): the
// batches accumulate through k_accumulate_checkpoints into these snapshot slices as well; entry0 is the first canvas
// entry of the render (its view's slice offset when nViews == 0).  list (nViews == 0): the same sample range for the
// listed entries only, batched as the samples of one view of nPad pixels and accumulated in batch order through
// k_accumulate_list; the per-tile primary masks are off (a tile is no longer 32 neighbouring pixels).
static int render_impl(b2pt_ctx* ctx, int sampleBegin, int sampleCount, int maxDepth, uint32_t flags, int64_t nViews,
                       const b2pt::CheckpointArgs* ckpt = nullptr, const ListedRound* list = nullptr)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "render before b2pt_set_scene");
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "render before b2pt_set_camera");
  if (sampleCount < 0 || sampleBegin < 0)
    return fail(B2PT_ERR_BAD_VALUE, "negative sample range");
  if (maxDepth < 1 || maxDepth > 4096)
    return fail(B2PT_ERR_BAD_VALUE, "maxDepth must be in [1,4096]");
  const bool refStream = (flags & B2PT_FLAG_REFERENCE_STREAM) != 0;
  if (refStream && (flags & B2PT_FLAG_KILL_ZERO_THROUGHPUT))
    return fail(B2PT_ERR_BAD_VALUE, "KILL_ZERO_THROUGHPUT cannot be combined with REFERENCE_STREAM");
  if (refStream && sampleBegin != 0)
    return fail(B2PT_ERR_BAD_VALUE, "REFERENCE_STREAM renders samples from 0 (one persistent stream per pixel)");
  if (int rc = ensure_built_for(ctx, flags))
    return rc;
  const bool viewMode = nViews > 0;
  if (!viewMode && !list)
    if (int rc = ensure_color(ctx))
      return rc;

  const int64_t N = list ? list->nPad : (int64_t)ctx->cam.W * ctx->cam.H;
  // B = sample slots per batch (view mode: whole views, viewsPerBatch x sampleCount slots).  The render is cut into
  // equal batches of `units` (samples, or views of unitPaths paths each): as few as the memory target allows, but up
  // to one per buffer set while every batch keeps at least 32 Mi paths -- four batches in flight beat two larger ones
  // (1024^2, depth 50: 256 spp as 4 x 64 53.8 ms, as 2 x 128 54.3; 64 spp as 2 x 32 14.5 ms, 4 x 16 15.0, 1 x 64 16.3).
  if (viewMode && refStream)
    return fail(B2PT_ERR_BAD_VALUE, "REFERENCE_STREAM cannot be combined with a view-batched render");
  const int64_t unitPaths = viewMode ? N * std::max(sampleCount, 1) : N;
  const int64_t units = viewMode ? nViews : sampleCount;
  // The plan: batch split, per-warp regions and the number of buffer sets in flight.  Results never depend on it.
  struct Plan
  {
    int64_t per = 1, viewsPerBatch = 0, B = 1, nBatches = 0, pathsPerBatch = 0, numWarps = 0, regionCap = 0, queueCap = 0;
    int nSets = 1;
  };
  // Two kernels per bounce (k_trace + k_shade with a ray queue in between) by default; small scenes can run the
  // one-kernel pipeline (k_bounce, B2PT_FLAG_ONE_KERNEL_BOUNCE): half the HBM traffic per survivor, but measured 25 %
  // slower per ray on B200 (DESIGN.md 4), so it is the opt-in.
  const bool fused = !ctx->useBvh && (flags & B2PT_FLAG_ONE_KERNEL_BOUNCE);
  const int blocksPerSM = fused ? std::min(ctx->cfg.traceBlocksPerSM[1][0], ctx->cfg.bounceBlocksPerSM)
                                : std::min(ctx->cfg.traceBlocksPerSM[0][ctx->useBvh ? (ctx->bvh.wide ? 2 : 1) : 0],
                                           ctx->cfg.shadeBlocksPerSM[0][ctx->useBvh ? 1 : 0]);
  // BVH scenes: the ray queue is sorted spatially before every region-mode bounce (B2PT_FLAG_NO_RAY_SORT: queue order)
  const bool raySort = ctx->useBvh && !(flags & B2PT_FLAG_NO_RAY_SORT) && !refStream;
  // ... and, on request, traced by the lean traversal kernel (k_bvh_hits) with the bookkeeping in a second one
  const bool splitTrace = raySort && !ctx->bvh.wide && (flags & B2PT_FLAG_SPLIT_TRACE);
  const int wpb = b2pt::warps_per_block();
  auto make_plan = [&](int64_t target, int64_t setsMax) {
    Plan P;
    int64_t nbPlanned = 0;
    if (!refStream)
      plan_batches(units, unitPaths, target, setsMax, P.per, nbPlanned);
    P.viewsPerBatch = viewMode ? P.per : 0;
    P.B = viewMode ? P.per * sampleCount : P.per;
    P.nBatches = (sampleCount == 0 || units == 0) ? 0 : (units + P.per - 1) / P.per;
    P.pathsPerBatch = N * P.B;
    // Static partition of the queue and the bins into one region per persistent warp (b2pt_types.h).
    P.numWarps = (int64_t)ctx->cfg.numSMs * blocksPerSM * wpb;
    P.numWarps =
      std::max<int64_t>(wpb, std::min<int64_t>(P.numWarps, ((P.pathsPerBatch + 31) / 32 + wpb - 1) / wpb * wpb));
    P.regionCap = (P.pathsPerBatch + P.numWarps - 1) / P.numWarps;
    P.regionCap = std::max<int64_t>(32, (P.regionCap + 31) / 32 * 32);
    P.queueCap = P.numWarps * P.regionCap;
    // Consecutive batches rotate over the context's stream and the extra streams (own buffers each): the tail of one
    // batch (small grids, one cluster) overlaps the head of the next.  Not in reference-stream mode, where sample s+1
    // continues the per-pixel RNG states sample s leaves behind.
    P.nSets = (P.nBatches > 1 && !refStream) ? (int)std::max<int64_t>(1, std::min<int64_t>(setsMax, P.nBatches)) : 1;
    return P;
  };
  auto reserve_sets = [&](const Plan& P) -> cudaError_t {
    for (int set = 0; set < P.nSets; ++set)
    {
      b2pt_ctx::BatchBufs& bb = ctx->bufs[set];
      cudaError_t e = cudaSuccess;
      if (fused) // buffers only the other pipeline needs go back first
        for (auto& q : bb.queue)
          q.release();
      else
      {
        for (auto& p : bb.bins[1])
          p.release();
        bb.binCode[1].release();
      }
      for (int p = 0; p < 3 && e == cudaSuccess; ++p)
      {
        if (!fused)
          e = bb.queue[p].reserve((size_t)P.queueCap);
        for (int h = 0; h < (fused ? 2 : 1) && e == cudaSuccess; ++h)
          e = bb.bins[h][p].reserve((size_t)P.queueCap * 4);
      }
      for (int h = 0; h < (fused ? 2 : 1) && e == cudaSuccess; ++h)
        e = bb.binCode[h].reserve((size_t)P.queueCap * 4);
      if (e == cudaSuccess)
        e = bb.regionCounts.reserve((size_t)P.numWarps * 9);
      if (e == cudaSuccess)
        e = bb.rad.reserve((size_t)P.pathsPerBatch);
      if (e == cudaSuccess && raySort)
      {
        if ((e = bb.sortKeys.reserve((size_t)P.queueCap)) == cudaSuccess &&
            (e = bb.sortPerm.reserve((size_t)P.queueCap)) == cudaSuccess &&
            (e = bb.sortHist.reserve((size_t)b2pt::sort_buckets())) == cudaSuccess)
          e = bb.sortTemp.reserve(b2pt::sort_temp_bytes());
        if (e == cudaSuccess && splitTrace)
          e = bb.hits.reserve((size_t)P.queueCap);
      }
      if (e != cudaSuccess)
        return e;
    }
    return cudaSuccess;
  };
  // The batch target was chosen from the memory that was free when the context rendered first.  If somebody else took
  // it since, the buffers no longer fit: give every set back and plan again with a LOCAL target -- halved while that
  // still shrinks the batches, then with fewer sets in flight -- until the allocation succeeds.  The context's own
  // target is left alone: the next render tries the full plan again.
  int64_t target = batch_target_paths(ctx, fused);
  int64_t setsMax = (flags & B2PT_FLAG_NO_OVERLAP) ? 1 : overlap_sets();
  Plan P = make_plan(target, setsMax);
  for (;;)
  {
    const cudaError_t me = reserve_sets(P);
    if (me == cudaSuccess)
      break;
    if (me != cudaErrorMemoryAllocation)
      return fail(B2PT_ERR_CUDA, "allocating the batch buffers failed: %s", cudaGetErrorString(me));
    cudaGetLastError(); // the allocation error is not sticky; clear it
    CU(cudaStreamSynchronize(ctx->stream));
    for (b2pt_ctx::BatchBufs& bb : ctx->bufs)
      bb.release_all();
    Plan Q = P;
    bool changed = false;
    while (!changed && !getenv("B2PT_BATCH_PATHS") && target > unitPaths && target > ((int64_t)1 << 16))
    { // halve until the plan really gets smaller (a single unit per batch cannot shrink further)
      target >>= 1;
      Q = make_plan(target, setsMax);
      changed = Q.pathsPerBatch < P.pathsPerBatch || Q.nSets < P.nSets;
    }
    while (!changed && setsMax > 1)
    {
      --setsMax;
      Q = make_plan(target, setsMax);
      changed = Q.nSets < P.nSets;
    }
    if (!changed)
      return fail(B2PT_ERR_ALLOC, "allocating the batch buffers failed (%lld paths per batch, %d set(s)): %s",
                  (long long)P.pathsPerBatch, P.nSets, cudaGetErrorString(me));
    P = Q;
  }
  const int64_t viewsPerBatch = P.viewsPerBatch, B = P.B, nBatches = P.nBatches, pathsPerBatch = P.pathsPerBatch;
  const int64_t numWarps = P.numWarps, regionCap = P.regionCap, queueCap = P.queueCap;
  const int nSets = P.nSets;
  const bool overlap = nSets > 1;
  const int64_t nCounters = std::max<int64_t>(1, nBatches * maxDepth); // rays entering bounce d+1, per batch
  CU(ctx->counters.reserve((size_t)nCounters));
  CU(ctx->binTotals.reserve((size_t)nCounters * 4));
  CU(ctx->nanCounter.reserve(1));
  int64_t launches0 = 0;
  CU(cudaEventRecord(ctx->evStart, ctx->stream));
  CU(cudaMemsetAsync(ctx->counters.p, 0, sizeof(uint32_t) * (size_t)nCounters, ctx->stream));
  CU(cudaMemsetAsync(ctx->binTotals.p, 0, sizeof(uint32_t) * (size_t)nCounters * 4, ctx->stream));
  CU(cudaMemsetAsync(ctx->nanCounter.p, 0, sizeof(unsigned long long), ctx->stream));
  if (refStream)
  {
    CU(ctx->seeds.reserve((size_t)N));
    CU(b2pt::launch_fill_seeds(ctx->seeds.p, (int)N, ctx->seedOffset, ctx->stream));
  }
  // Primary-ray specialisation (small scenes whose tiles of 32 path ids are tiles of 32 pixels of one view): candidate
  // masks per tile and quad constants per view, recomputed per render (a few microseconds).
  const bool primMasks =
    !ctx->useBvh && !list && (N % 32) == 0 && nBatches > 0 && !(flags & B2PT_FLAG_NO_PRIMARY_MASKS);
  const int tilesPerView = (int)(N / 32);
  if (primMasks)
  {
    const int nv = viewMode ? (int)nViews : 1;
    CU(ctx->primMask.reserve((size_t)nv * tilesPerView));
    CU(ctx->primQuads.reserve((size_t)nv * B2PT_SMALL_MAX_QUADS));
    CU(b2pt::launch_primary_prep(ctx->small, ctx->cam, viewMode ? ctx->dViews.p : nullptr, nv, tilesPerView,
                                 ctx->primMask.p, ctx->primQuads.p, ctx->stream));
    ++launches0;
  }

  // An error return while batches are in flight on the extra streams must not leave them running behind the caller's
  // back (later work on the context's stream would race with them): the guard drains them on every early exit.
  struct DrainGuard
  {
    b2pt_ctx* c;
    int n;
    bool armed;
    ~DrainGuard()
    {
      if (armed)
        for (int k = 1; k < n; ++k)
          cudaStreamSynchronize(c->extra[k]);
    }
  } drain{ ctx, nSets, overlap };
  if (overlap)
  { // the extra streams start after everything queued so far on the context's stream (clears, seeds, earlier renders)
    CU(cudaEventRecord(ctx->evFork, ctx->stream));
    for (int k = 1; k < nSets; ++k)
      CU(cudaStreamWaitEvent(ctx->extra[k], ctx->evFork, 0));
  }
  int64_t launches = (refStream ? 1 : 0) + launches0;
  // bounces >= tailDepth run in tail mode, bounces >= loopDepth (>= tailDepth) inside one persistent cluster launch;
  // chosen after the first batch.  "Never" is maxDepth for the two-kernel pipeline and maxDepth + 1 for the one-kernel
  // pipeline, whose closing pass is launch number maxDepth.
  const int never = maxDepth + (fused ? 1 : 0);
  int tailDepth = never, loopDepth = never;
  const int64_t tailKey[7] = { ctx->sceneVersion,  N, maxDepth, pathsPerBatch, (int64_t)flags, tail_rays_per_warp(),
                               tail_loop_rays() };
  const bool tailAllowed = nBatches > 1 && !(flags & B2PT_FLAG_NO_TAIL) && maxDepth > 2;
  if (tailAllowed && std::equal(tailKey, tailKey + 7, ctx->tailKey))
  {
    tailDepth = ctx->tailDepthCached;
    loopDepth = ctx->loopDepthCached;
  }
  const int profDepths = std::min(maxDepth - 1, (int)b2pt_ctx::kProfDepths); // events 0..profDepths bracket that many bounces
  ctx->profDepths = nBatches > 0 ? profDepths : 0;
  ctx->profPaths = nBatches > 0 ? N * (viewMode ? B : std::min<int64_t>(B, sampleCount)) : 0;
  for (int64_t batch = 0; batch < nBatches; ++batch)
  {
    // view mode: views [v0, v0+nv) with all their samples; otherwise samples [s0, s0+nb) of the one view
    const int64_t v0 = batch * viewsPerBatch;
    const int64_t nv = viewMode ? std::min<int64_t>(viewsPerBatch, nViews - v0) : 0;
    const int64_t s0 = viewMode ? 0 : batch * B;
    const int64_t nb = viewMode ? nv * sampleCount : std::min<int64_t>(B, sampleCount - s0);
    const int set = (int)(batch % nSets);
    b2pt_ctx::BatchBufs& bb = ctx->bufs[set];
    cudaStream_t bs = set ? ctx->extra[set] : ctx->stream;
    B2RenderArgs A{};
    A.depthTotals = ctx->counters.p + batch * maxDepth;
    A.binTotals = ctx->binTotals.p + batch * maxDepth * 4;
    A.rad = bb.rad.p;
    for (int h = 0; h < 2; ++h)
      A.bins[h] = { bb.bins[h][0].p, bb.bins[h][1].p, bb.bins[h][2].p, bb.binCode[h].p,
                    bb.regionCounts.p + numWarps * (1 + 4 * h) };
    A.binStride = queueCap;
    A.q = { bb.queue[0].p, bb.queue[1].p, bb.queue[2].p };
    A.qCount = bb.regionCounts.p;
    A.numWarps = (int32_t)numWarps;
    A.regionCap = (int32_t)regionCap;
    A.seeds = ctx->seeds.p;
    A.nPaths = N * nb;
    A.nPixels = (int32_t)N;
    A.sampleBase = (int32_t)(sampleBegin + s0);
    A.views = viewMode ? ctx->dViews.p + v0 : (list ? ctx->dViews.p : nullptr);
    A.sppPerView = viewMode ? sampleCount : 0;
    A.primMask = primMasks ? ctx->primMask.p + (viewMode ? v0 * tilesPerView : 0) : nullptr;
    A.primQuads = primMasks ? ctx->primQuads.p + (viewMode ? v0 * B2PT_SMALL_MAX_QUADS : 0) : nullptr;
    A.tilesPerView = tilesPerView;
    A.maxDepth = maxDepth;
    b2pt::make_fastdiv((uint32_t)N, A.divPixelsMagic, A.divPixelsShift);
    b2pt::make_fastdiv((uint32_t)std::max(viewMode ? sampleCount : 1, 1), A.divSppMagic, A.divSppShift);
    A.nLightQuads = ctx->lights.nLightQuads;
    A.nLightSph = ctx->lights.nLightSph;
    A.seedOffset = ctx->seedOffset;
    A.flags = flags;
    if (list)
    { // (bounce 0 reads the list through A.perm, see below)
      A.sppPerView = list->viewPixels;
      b2pt::make_fastdiv((uint32_t)list->viewPixels, A.divSppMagic, A.divSppShift);
    }
    // fused: launches 0 (primary) .. maxDepth (the closing shade pass); split: bounces 0 .. maxDepth-1, two launches each
    for (int depth = 0; depth < maxDepth + (fused ? 1 : 0); ++depth)
    {
      if (batch == 0 && depth <= b2pt_ctx::kProfDepths && depth <= profDepths)
      { // per-launch CUDA events of the first bounces of batch 0 (b2pt_get_bounce_profile)
        if (!ctx->evBounce[depth])
          CU(cudaEventCreate(&ctx->evBounce[depth]));
        CU(cudaEventRecord(ctx->evBounce[depth], bs));
      }
      cudaEvent_t mid = nullptr;
      if (batch == 0 && depth < profDepths)
      {
        if (!ctx->evMid[depth])
          CU(cudaEventCreate(&ctx->evMid[depth]));
        mid = ctx->evMid[depth];
      }
      A.depth = depth;
      const int mode = depth >= tailDepth ? b2pt::B2PT_BOUNCE_TAIL
                                          : (depth == tailDepth - 1 ? b2pt::B2PT_BOUNCE_TO_GLOBAL : b2pt::B2PT_BOUNCE_REGIONS);
      if (fused)
      {
        if (depth == 0)
          CU(b2pt::launch_primary(ctx->cfg, ctx->cam, ctx->small, A, bs));
        else if (depth >= loopDepth)
        { // every remaining bounce and the closing pass in one cluster launch
          CU(b2pt::launch_bounce_tail_loop(ctx->small, ctx->lights, A, bs));
          ++launches;
          break;
        }
        else
          CU(b2pt::launch_bounce_fused(ctx->cfg, mode, ctx->small, ctx->lights, A, bs));
        ++launches;
        if (mid) // one launch per bounce: the whole bounce is reported as the "trace" stage
          CU(cudaEventRecord(mid, bs));
        continue;
      }
      if (depth >= loopDepth)
      { // every remaining bounce in one cluster launch
        CU(b2pt::launch_tail_loop(ctx->cam, ctx->useBvh ? nullptr : &ctx->small, ctx->useBvh ? &ctx->bvh : nullptr,
                                  ctx->lights, A, bs));
        ++launches;
        break;
      }
      A.perm = (list && depth == 0) ? list->entries : nullptr; // listed round: bounce 0 traces the list (k_trace LISTED)
      A.hits = nullptr;
      if (raySort && depth >= 1 && mode != b2pt::B2PT_BOUNCE_TAIL)
      { // queue regions of k_shade(depth - 1) -> permutation by origin cell and direction octant
        CU(b2pt::launch_sort_rays(A, ctx->sortLo, ctx->sortHi, bb.sortHist.p, bb.sortKeys.p, bb.sortPerm.p,
                                  bb.sortTemp.p, bb.sortTemp.cap, bs));
        A.perm = bb.sortPerm.p;
        A.hits = splitTrace ? bb.hits.p : nullptr;
        launches += splitTrace ? 4 : 3;
      }
      CU(b2pt::launch_bounce(ctx->cfg, depth == 0, mode, ctx->cam, ctx->useBvh ? nullptr : &ctx->small,
                             ctx->useBvh ? &ctx->bvh : nullptr, ctx->lights, A, bs, mid));
      launches += 2;
    }
    // the canvas is accumulated in batch order (sample-order sums): wait for the previous batch's accumulate
    // (view batches write disjoint canvases: no order needed)
    if (overlap && batch > 0 && !viewMode)
      CU(cudaStreamWaitEvent(bs, ctx->evAcc[(set + nSets - 1) % nSets], 0));
    // view mode: nv views of sampleCount samples each; otherwise nb samples of the one canvas
    float4* const canvas = viewMode ? ctx->viewColor.p + v0 * N : ctx->color();
    const int accSamples = viewMode ? sampleCount : (int)nb, accViews = viewMode ? (int)nv : 1;
    if (list)
      CU(b2pt::launch_accumulate_list(list->color, list->moment, bb.rad.p, list->entries, (int)list->nReal, (int)N,
                                      (int)nb, ctx->nanCounter.p, bs));
    else if (ckpt)
    {
      b2pt::CheckpointArgs ck = *ckpt;
      ck.sampleBase = A.sampleBase;
      ck.entry0 += v0 * N;
      CU(b2pt::launch_accumulate_checkpoints(canvas, bb.rad.p, (int)N, accSamples, accViews, ctx->nanCounter.p, ck,
                                             bs));
    }
    else
      CU(b2pt::launch_accumulate(canvas, bb.rad.p, (int)N, accSamples, accViews, ctx->nanCounter.p, bs));
    ++launches;
    if (overlap)
      CU(cudaEventRecord(ctx->evAcc[set], bs));
    if (batch == 0 && tailAllowed && tailDepth == never && !std::equal(tailKey, tailKey + 7, ctx->tailKey))
    { // Tail mode for the remaining batches: from the first bounce that less than tailRaysPerWarp rays per region
      // enter, rays live in one flat global queue (k_trace TAIL).  Decided from the first batch's own counters: one
      // stream synchronisation per render.
      CU(cudaStreamSynchronize(ctx->stream));
      std::vector<uint32_t> first((size_t)maxDepth);
      CU(cudaMemcpy(first.data(), ctx->counters.p, sizeof(uint32_t) * (size_t)maxDepth, cudaMemcpyDeviceToHost));
      const int64_t threshold = numWarps * tail_rays_per_warp();
      // (the one-kernel pipeline bins bounce 0 per region, so its first global-bin launch is bounce 1: tailDepth >= 2)
      for (int d = fused ? 2 : 1; d < maxDepth; ++d) // first[d-1] = rays entering bounce d
        if ((int64_t)first[(size_t)d - 1] < threshold)
        {
          tailDepth = d;
          break;
        }
      for (int d = tailDepth; d < maxDepth; ++d)
        if ((int64_t)first[(size_t)d - 1] < tail_loop_rays())
        {
          loopDepth = d;
          break;
        }
      std::copy(tailKey, tailKey + 7, ctx->tailKey);
      ctx->tailDepthCached = tailDepth;
      ctx->loopDepthCached = loopDepth;
    }
  }
  if (overlap)
  { // join: the context's stream continues after everything the extra streams did
    for (int k = 1; k < nSets; ++k)
    {
      CU(cudaEventRecord(ctx->evJoin[k], ctx->extra[k]));
      CU(cudaStreamWaitEvent(ctx->stream, ctx->evJoin[k], 0));
    }
  }
  drain.armed = false;
  CU(cudaEventRecord(ctx->evStop, ctx->stream));

  ctx->stats = b2pt_stats{};
  ctx->stats.paths = N * (int64_t)sampleCount * (viewMode ? nViews : 1);
  ctx->stats.launches = launches;
  ctx->stats.batches = (int32_t)nBatches;
  ctx->stats.samplesPerBatch = (int32_t)B;
  ctx->stats.tracePath = ctx->useBvh ? 1 : 0;
  ctx->stats.tailDepth = std::min(tailDepth, maxDepth);
  ctx->stats.loopDepth = std::min(loopDepth, maxDepth);
  ctx->stats.tracePath = ctx->useBvh ? 1 : 0;
  ctx->stats.bvhNodes = ctx->bvhNodes;
  ctx->stats.tracedQuads = ctx->tracedQuads;
  ctx->stats.tracedSpheres = ctx->tracedSph;
  ctx->statsPending = true;
  ctx->pendingCounters = nBatches * maxDepth;
  ctx->pendingMaxDepth = maxDepth;
  ctx->pendingPathsPerBatch = pathsPerBatch;
  return B2PT_OK;
}

// Host-only self-check of the tree builders on the configs[3]-style scene (no GPU): binary binned-SAH tree, collapse
// into 8-wide compressed nodes, structural validation of both.
int b2pt_bvh_selfcheck(int64_t nSpheres, int64_t* stats4)
{
  if (nSpheres < 1 || nSpheres > 4000000 || !stats4)
    return fail(B2PT_ERR_BAD_VALUE, "b2pt_bvh_selfcheck: bad argument");
  const size_t n = (size_t)nSpheres;
  std::vector<float> pts(3 * (n + 8)), sphR(n), tex(12);
  std::vector<int64_t> quadIds(10), sphPt(n), mq(2), tq(2), ms(n), ts(n);
  std::vector<int> matType(5), texType(5);
  if (int rc = b2pt_scene_spheres(nSpheres, pts.data(), quadIds.data(), sphPt.data(), sphR.data(), mq.data(), tq.data(),
                                  ms.data(), ts.data(), matType.data(), texType.data(), tex.data()))
    return fail(rc, "b2pt_scene_spheres failed");
  std::vector<B2Quad> quads(2);
  std::vector<B2Sphere> sph(n);
  auto P = [&](int64_t i) -> H3 { return { pts[3 * (size_t)i], pts[3 * (size_t)i + 1], pts[3 * (size_t)i + 2] }; };
  float sceneAbs = 0.f;
  for (int q = 0; q < 2; ++q)
  {
    std::memset(&quads[(size_t)q], 0, sizeof(B2Quad));
    const int64_t* id = quadIds.data() + 5 * q;
    precompute_quad(quads[(size_t)q], P(id[1]), P(id[2]), P(id[3]), P(id[4]));
    quads[(size_t)q].prim = q;
  }
  for (size_t k = 0; k < n; ++k)
  {
    std::memset(&sph[k], 0, sizeof(B2Sphere));
    hst(sph[k].c, P((int64_t)k));
    sph[k].r = sphR[k];
    for (int c = 0; c < 3; ++c)
      sceneAbs = std::fmax(sceneAbs, std::fabs(sph[k].c[c]) + sph[k].r);
  }
  std::vector<B2BvhNode> nodes;
  std::vector<int32_t> slots;
  const std::vector<int32_t> treeQuads = { 0, 1 };
  int binDepth = 0;
  if (!b2pt::build_bvh(quads, treeQuads, sph, nodes, slots, &binDepth))
    return fail(B2PT_ERR_UNSUPPORTED, "binary tree does not fit the index packing");
  b2pt::WideBuildResult wr;
  if (!b2pt::collapse_to_wide(nodes, slots, quads, sph, sceneAbs, wr) || wr.slots.size() != n + 2)
    return fail(B2PT_ERR_STATE, "collapse failed");
  std::string why;
  if (!b2pt::validate_wide(wr, quads, sph, why))
    return fail(B2PT_ERR_STATE, "8-wide BVH validation failed: %s", why.c_str());
  stats4[0] = (int64_t)nodes.size();
  stats4[1] = binDepth;
  stats4[2] = (int64_t)wr.nodes.size();
  stats4[3] = wr.maxDepth;
  return B2PT_OK;
}

int b2pt_plan_batches(int64_t units, int64_t unitPaths, int64_t maxPathsPerBatch, int sets, int64_t* unitsPerBatch,
                      int64_t* nBatches)
{
  if (!unitsPerBatch || !nBatches || units < 0 || unitPaths <= 0 || maxPathsPerBatch <= 0 || sets <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "b2pt_plan_batches: bad argument");
  plan_batches(units, unitPaths, maxPathsPerBatch, sets, *unitsPerBatch, *nBatches);
  return B2PT_OK;
}

int b2pt_render_range(b2pt_ctx* ctx, int sampleBegin, int sampleCount, int maxDepth, uint32_t flags)
{
  return render_impl(ctx, sampleBegin, sampleCount, maxDepth, flags, 0);
}

// The view sweep of b2pt_render_views and b2pt_render_views_checkpoints once their arguments are checked: counts[K-1]
// samples of every camera of `cams` (one canvas size) into ctx->viewColor, then for every count k the image its entry
// point returns, converted per the view flags and copied to slice k of rgbaOut (NULL: no copy).  ck == nullptr
// (b2pt_render_views, K == 1, no moments): the batches accumulate through k_accumulate.  Otherwise ck holds the
// checkpoint list (n, count) and they accumulate through k_accumulate_checkpoints, which keeps the running sums at
// every count and, when moment2Out is not NULL or keepMoments is set, the sums of squares (in ctx->ckptMoment).
static int render_view_sweep(b2pt_ctx* ctx, const std::vector<B2Camera>& cams, const int* counts, int K, int maxDepth,
                             uint32_t flags, b2pt::CheckpointArgs* ck, void* rgbaOut, float* moment2Out,
                             bool keepMoments = false)
{
  const int64_t nViews = (int64_t)cams.size();
  if (nViews == 0)
  {
    ctx->viewCount = 0;
    return B2PT_OK;
  }
  const int spp = counts[K - 1];
  const int64_t N = (int64_t)cams[0].W * cams[0].H, NV = N * nViews;
  const bool moments = moment2Out != nullptr || keepMoments;
  CU(ctx->viewColor.reserve((size_t)NV));
  CU(ctx->dViews.reserve((size_t)nViews));
  if (K > 1)
    CU(ctx->ckptSnap.reserve((size_t)(NV * (K - 1))));
  if (moments)
    CU(ctx->ckptMoment.reserve((size_t)(NV * K)));
  ctx->viewCount = nViews;
  ctx->viewPixels = N;
  if (ck)
  {
    ck->snap = ctx->ckptSnap.p;
    ck->moment = moments ? ctx->ckptMoment.p : nullptr;
    ck->sliceStride = NV;
  }
  // the running sums start from zero: the image and the running sum of squares (slice K-1); every other slice is
  // written exactly once
  auto clear = [&]() -> cudaError_t {
    cudaError_t e = cudaMemsetAsync(ctx->viewColor.p, 0, sizeof(float4) * (size_t)NV, ctx->stream);
    if (e == cudaSuccess && moments)
      e = cudaMemsetAsync(ctx->ckptMoment.p + NV * (K - 1), 0, sizeof(float4) * (size_t)NV, ctx->stream);
    return e;
  };
  // the context's own camera gives the canvas shape to the launches; it is restored afterwards
  const B2Camera savedCam = ctx->cam;
  const bool savedHave = ctx->haveCamera;
  float4* const savedExt = ctx->colorExt;
  CU(clear());
  ctx->cam = cams[0];
  ctx->haveCamera = true;
  int rc = B2PT_OK;
  auto restore = [&]() {
    ctx->cam = savedCam;
    ctx->haveCamera = savedHave;
    ctx->colorExt = savedExt;
  };
  bool perView = !(spp > 0 && N * spp <= std::min<int64_t>(batch_target_paths(ctx, true), 0xfffffff0LL));
  if (!perView)
  { // whole views fit a batch: (view, sample, pixel) is one flat index space, one set of launches per batch of views
    // (pageable source: the copy is staged before the call returns, so `cams` may go out of scope)
    cudaError_t e = cudaMemcpyAsync(ctx->dViews.p, cams.data(), sizeof(B2Camera) * (size_t)nViews,
                                    cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess)
    {
      restore();
      return fail(B2PT_ERR_CUDA, "cudaMemcpyAsync(views): %s", cudaGetErrorString(e));
    }
    rc = render_impl(ctx, 0, spp, maxDepth, flags, nViews, ck);
    perView = rc == B2PT_ERR_ALLOC; // the buffers of a whole-view batch could not be allocated: views one by one
  }
  if (perView)
  { // a single view already fills several batches: one ordinary render per view into its slice of every output;
    // sample batches carry the running sums in viewColor and moment slice K-1
    rc = B2PT_OK;
    if (clear() != cudaSuccess)
      rc = fail(B2PT_ERR_CUDA, "clearing the view canvases failed");
    int64_t paths = 0, launches = 0;
    for (int64_t v = 0; v < nViews && rc == B2PT_OK; ++v)
    {
      ctx->cam = cams[(size_t)v];
      ctx->colorExt = ctx->viewColor.p + (size_t)v * N;
      if (ck)
        ck->entry0 = v * N;
      rc = render_impl(ctx, 0, spp, maxDepth, flags, 0, ck);
      paths += ctx->stats.paths;
      launches += ctx->stats.launches;
    }
    ctx->stats.paths = paths;
    ctx->stats.launches = launches;
  }
  restore();
  if (rc != B2PT_OK)
    return rc;
  // per count, the conversion the view flags ask for (the last image is viewColor itself)
  for (int k = 0; k < K; ++k)
  {
    float4* const img = k + 1 < K ? ctx->ckptSnap.p + NV * k : ctx->viewColor.p;
    if (flags & B2PT_FLAG_VIEWS_PNM16)
    { // the integers of the reference's P3 writer instead of the float sums: 6 B instead of 16 B per pixel to the host
      if (!rgbaOut)
        break;
      CU(ctx->pnm.reserve((size_t)NV * 3));
      CU(b2pt::launch_pnm16(img, NV, counts[k], ctx->pnm.p, ctx->stream));
      CU(cudaMemcpyAsync(static_cast<uint16_t*>(rgbaOut) + (size_t)(NV * k) * 3, ctx->pnm.p,
                         sizeof(uint16_t) * 3 * (size_t)NV, cudaMemcpyDeviceToHost, ctx->stream));
      continue;
    }
    if ((flags & B2PT_FLAG_VIEWS_NORMALIZE) && (rgbaOut || k + 1 == K))
      CU(b2pt::launch_normalize(img, NV, counts[k], ctx->stream));
    if (rgbaOut)
      CU(cudaMemcpyAsync(static_cast<float4*>(rgbaOut) + NV * k, img, sizeof(float4) * (size_t)NV,
                         cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (moment2Out)
    CU(cudaMemcpyAsync(moment2Out, ctx->ckptMoment.p, sizeof(float4) * (size_t)(NV * K), cudaMemcpyDeviceToHost,
                       ctx->stream));
  if (rgbaOut || moment2Out)
    CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

int b2pt_render_views(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int spp, int maxDepth,
                      uint32_t flags, void* rgbaOut)
{
  if (int rc = bind(ctx))
    return rc;
  if (int rc = check_view_list("b2pt_render_views", nViews, views))
    return rc;
  if (spp < 0)
    return fail(B2PT_ERR_BAD_VALUE, "negative sample range");
  if (flags & B2PT_FLAG_REFERENCE_STREAM)
    return fail(B2PT_ERR_BAD_VALUE, "REFERENCE_STREAM cannot be combined with a view-batched render");
  if ((flags & B2PT_FLAG_VIEWS_PNM16) && spp <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "spp must be positive"); // the PNM integers divide by spp
  std::vector<B2Camera> cams;
  if (int rc = make_view_cameras(nViews, views, W, H, cams))
    return rc;
  if ((int64_t)W * H * nViews > (int64_t)1 << 30)
    return fail(B2PT_ERR_BAD_VALUE, "b2pt_render_views: more than 2^30 output pixels (16 GiB); split the view list");
  return render_view_sweep(ctx, cams, &spp, 1, maxDepth, flags, nullptr, rgbaOut, nullptr);
}

// b2pt_render_views at spp = checkpoints[K-1] through k_accumulate_checkpoints: sample s of a pixel is the same RNG
// stream and is added in the same order at every spp, so the prefix sum after checkpoints[k] samples is the image
// b2pt_render_views(spp = checkpoints[k]) returns, whatever the batching.
int b2pt_render_views_checkpoints(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                                  const int* checkpoints, int maxDepth, uint32_t flags, void* rgbaOut,
                                  float* moment2Out)
{
  if (int rc = bind(ctx))
    return rc;
  if (int rc = check_view_list("b2pt_render_views_checkpoints", nViews, views))
    return rc;
  if (int rc = check_checkpoints("b2pt_render_views_checkpoints", nCheckpoints, checkpoints))
    return rc;
  if (flags & B2PT_FLAG_REFERENCE_STREAM)
    return fail(B2PT_ERR_BAD_VALUE, "REFERENCE_STREAM cannot be combined with a view-batched render");
  std::vector<B2Camera> cams;
  if (int rc = make_view_cameras(nViews, views, W, H, cams))
    return rc;
  const int K = nCheckpoints;
  const int64_t slices = (K - 1) + (moment2Out ? K : 0) + 1; // snapshots, sums of squares, the last image
  if ((int64_t)W * H * nViews > ((int64_t)1 << 30) / slices)
    return fail(B2PT_ERR_BAD_VALUE,
                "b2pt_render_views_checkpoints: more than 2^30 float4 of device output (16 GiB); split the view list");
  b2pt::CheckpointArgs ck{};
  ck.n = K;
  std::copy(checkpoints, checkpoints + K, ck.count);
  return render_view_sweep(ctx, cams, ck.count, K, maxDepth, flags, &ck, rgbaOut, moment2Out);
}

void b2pt_adaptive_defaults(b2pt_adaptive_params* p)
{
  if (!p)
    return;
  p->threshold = 0.02f;
  p->epsilon = 0.01f;
  p->radius = 1;
}

// Adaptive sampling of a view sweep (DESIGN.md 8f).  Round 0 is render_view_sweep at rounds[0] with the sums of squares
// kept on the device, so it is b2pt_render_views_checkpoints by construction.  After round k, k_adaptive_mark and
// k_adaptive_select choose the canvas entries of round k+1 and cub compacts them into ctx->adList in ascending order;
// the one host read per round is that list's length.  Round k+1 is render_impl over the list (samples
// [rounds[k], rounds[k+1]) of every listed entry), which continues each entry's sums in sample order, so an entry
// that ends with n samples holds the bits of a uniform render of n samples.
int b2pt_render_views_adaptive(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nRounds,
                               const int* rounds, int maxDepth, const b2pt_adaptive_params* params, uint32_t flags,
                               void* rgbaOut, float* moment2Out, int32_t* countOut, int64_t* activeOut)
{
  static const char* const fn = "b2pt_render_views_adaptive";
  if (int rc = bind(ctx))
    return rc;
  if (int rc = check_view_list(fn, nViews, views))
    return rc;
  if (int rc = check_checkpoints(fn, nRounds, rounds))
    return rc;
  if (rounds[0] < 2)
    return fail(B2PT_ERR_BAD_VALUE, "%s: rounds[0] must be >= 2 (a variance needs two samples)", fn);
  if (maxDepth < 1 || maxDepth > 4096)
    return fail(B2PT_ERR_BAD_VALUE, "maxDepth must be in [1,4096]");
  if (flags & (B2PT_FLAG_REFERENCE_STREAM | B2PT_FLAG_ONE_KERNEL_BOUNCE))
    return fail(B2PT_ERR_BAD_VALUE, "%s: REFERENCE_STREAM and ONE_KERNEL_BOUNCE cannot be combined with it", fn);
  b2pt_adaptive_params P;
  if (params)
    P = *params;
  else
    b2pt_adaptive_defaults(&P);
  if (!(P.threshold >= 0.f)) // NaN fails too
    return fail(B2PT_ERR_BAD_VALUE, "%s: threshold must be >= 0 (or +inf), got %g", fn, (double)P.threshold);
  if (!(P.epsilon > 0.f))
    return fail(B2PT_ERR_BAD_VALUE, "%s: epsilon must be > 0, got %g", fn, (double)P.epsilon);
  if (P.radius < 0 || P.radius > 4)
    return fail(B2PT_ERR_BAD_VALUE, "%s: radius must be in [0,4], got %d", fn, P.radius);
  std::vector<B2Camera> cams;
  if (int rc = make_view_cameras(nViews, views, W, H, cams))
    return rc;
  if (2 * (int64_t)W * H * nViews > (int64_t)1 << 30)
    return fail(B2PT_ERR_BAD_VALUE, "%s: more than 2^30 float4 of device state (16 GiB); split the view list", fn);
  if (nViews == 0)
    return B2PT_OK;
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "render before b2pt_set_scene");

  const int K = nRounds;
  const int64_t N = (int64_t)W * H, NV = N * nViews;
  const uint32_t renderFlags = flags & ~(uint32_t)(B2PT_FLAG_VIEWS_NORMALIZE | B2PT_FLAG_VIEWS_PNM16);
  b2pt::CheckpointArgs ck{};
  ck.n = 1;
  ck.count[0] = rounds[0];
  if (int rc = render_view_sweep(ctx, cams, rounds, 1, maxDepth, renderFlags, &ck, nullptr, nullptr, true))
    return rc;
  int64_t paths = ctx->stats.paths, launches = ctx->stats.launches;
  std::vector<int64_t> active((size_t)K, 0);
  active[0] = NV;

  const size_t tempBytes = b2pt::adaptive_select_temp_bytes(NV);
  CU(ctx->adCounts.reserve((size_t)NV));
  CU(ctx->adUnconv.reserve((size_t)NV));
  CU(ctx->adActive.reserve((size_t)NV));
  CU(ctx->adList.reserve((size_t)NV + 32));
  CU(ctx->adNum.reserve(1));
  CU(ctx->adTemp.reserve(std::max<size_t>(tempBytes, 1)));
  // (the whole-view path of round 0 uploads the cameras too, its per-view fallback does not)
  CU(cudaMemcpyAsync(ctx->dViews.p, cams.data(), sizeof(B2Camera) * (size_t)nViews, cudaMemcpyHostToDevice,
                     ctx->stream));
  b2pt::AdaptiveArgs a{};
  a.tau = P.threshold;
  a.eps = P.epsilon;
  a.radius = P.radius;
  a.W = W;
  a.H = H;

  // the listed rounds take the canvas shape from the context's camera, which is restored afterwards
  const B2Camera savedCam = ctx->cam;
  const bool savedHave = ctx->haveCamera;
  ctx->cam = cams[0];
  ctx->haveCamera = true;
  int rc = B2PT_OK;
  for (int k = 0; k + 1 < K && rc == B2PT_OK; ++k)
  {
    a.c = rounds[k];
    a.next = rounds[k + 1];
    a.first = k == 0;
    int32_t n = 0;
    cudaError_t e = b2pt::launch_adaptive_mark(ctx->viewColor.p, ctx->ckptMoment.p, ctx->adCounts.p, ctx->adUnconv.p,
                                               NV, a, ctx->stream);
    if (e == cudaSuccess)
      e = b2pt::launch_adaptive_select(ctx->adUnconv.p, ctx->adCounts.p, ctx->adActive.p, NV, a, ctx->adList.p,
                                       ctx->adNum.p, ctx->adTemp.p, tempBytes, ctx->stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(&n, ctx->adNum.p, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess)
      e = cudaStreamSynchronize(ctx->stream);
    const int64_t nPad = ((int64_t)n + 31) / 32 * 32;
    if (e == cudaSuccess && n > 0)
      e = b2pt::launch_list_pad(ctx->adList.p, n, (int)nPad, ctx->stream);
    if (e != cudaSuccess)
    {
      rc = fail(B2PT_ERR_CUDA, "%s: selecting round %d failed: %s", fn, k + 1, cudaGetErrorString(e));
      break;
    }
    active[(size_t)k + 1] = n;
    if (n == 0)
      break; // nothing has rounds[k+1] samples, so nothing can reach the later rounds either
    const ListedRound L{ ctx->adList.p, n, nPad, (int)N, ctx->viewColor.p, ctx->ckptMoment.p };
    rc = render_impl(ctx, rounds[k], rounds[k + 1] - rounds[k], maxDepth, renderFlags, 0, nullptr, &L);
    paths += (int64_t)n * (rounds[k + 1] - rounds[k]);
    launches += ctx->stats.launches;
  }
  ctx->cam = savedCam;
  ctx->haveCamera = savedHave;
  if (rc != B2PT_OK)
    return rc;
  if (K == 1) // no selection ran: every entry has rounds[0] samples
  {
    a.c = rounds[0];
    a.first = 1;
    CU(b2pt::launch_adaptive_mark(ctx->viewColor.p, ctx->ckptMoment.p, ctx->adCounts.p, ctx->adUnconv.p, NV, a,
                                  ctx->stream));
  }
  if (flags & B2PT_FLAG_VIEWS_PNM16)
  {
    if (rgbaOut)
    {
      CU(ctx->pnm.reserve((size_t)NV * 3));
      CU(b2pt::launch_pnm16_counts(ctx->viewColor.p, NV, ctx->adCounts.p, ctx->pnm.p, ctx->stream));
      CU(cudaMemcpyAsync(rgbaOut, ctx->pnm.p, sizeof(uint16_t) * 3 * (size_t)NV, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  else
  {
    if (flags & B2PT_FLAG_VIEWS_NORMALIZE)
      CU(b2pt::launch_normalize_counts(ctx->viewColor.p, NV, ctx->adCounts.p, ctx->stream));
    if (rgbaOut)
      CU(cudaMemcpyAsync(rgbaOut, ctx->viewColor.p, sizeof(float4) * (size_t)NV, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (moment2Out)
    CU(cudaMemcpyAsync(moment2Out, ctx->ckptMoment.p, sizeof(float4) * (size_t)NV, cudaMemcpyDeviceToHost,
                       ctx->stream));
  if (countOut)
    CU(cudaMemcpyAsync(countOut, ctx->adCounts.p, sizeof(int32_t) * (size_t)NV, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (activeOut)
    std::copy(active.begin(), active.end(), activeOut);
  ctx->stats.paths = paths;
  ctx->stats.launches = launches;
  return B2PT_OK;
}

// Denoiser guides of a view sweep (k_view_features).  Sample s of a pixel is traced from the stream the render gives it
// (pixel + seedOffset + s * B2PT_GOLDEN), through the trace structure a render with these flags would use, so the
// features average the rays the radiance image averages.  Views run in chunks of whole views, each chunk one launch
// into the context's staging buffers (at most max(kFeatureChunkFloat4, K*W*H) float4 per output) and K copies per
// output into the caller's arrays.  The context's camera, canvas, view images and statistics are not touched.
static constexpr int64_t kFeatureChunkFloat4 = (int64_t)1 << 23;
int b2pt_render_views_features(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                               const int* checkpoints, uint32_t flags, float* albedoOut, float* normalDepthOut)
{
  if (int rc = bind(ctx))
    return rc;
  if (int rc = check_view_list("b2pt_render_views_features", nViews, views))
    return rc;
  if (int rc = check_checkpoints("b2pt_render_views_features", nCheckpoints, checkpoints))
    return rc;
  if (checkpoints[nCheckpoints - 1] > (1 << 24))
    return fail(B2PT_ERR_BAD_VALUE,
                "b2pt_render_views_features: more than 2^24 samples (the hit count must stay an exact float)");
  if (flags & ~kBuildFlags)
    return fail(B2PT_ERR_BAD_VALUE,
                "b2pt_render_views_features: flags may only hold FORCE_BVH, NO_DEDUP, NO_AA, GPU_LBVH and WIDE_BVH");
  std::vector<B2Camera> cams;
  if (int rc = make_view_cameras(nViews, views, W, H, cams))
    return rc;
  if (nViews == 0)
    return B2PT_OK;
  const int K = nCheckpoints;
  const int64_t N = (int64_t)W * H, KN = N * K;
  if (KN > ((int64_t)1 << 30))
    return fail(B2PT_ERR_BAD_VALUE, "b2pt_render_views_features: one view's %d slices exceed 2^30 float4", K);
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "b2pt_render_views_features before b2pt_set_scene");
  if (int rc = ensure_built_for(ctx, flags))
    return rc;
  b2pt::FeatureCheckpoints ck{};
  ck.n = K;
  std::copy(checkpoints, checkpoints + K, ck.count);
  const int64_t perChunk = std::max<int64_t>(1, kFeatureChunkFloat4 / KN);
  const size_t cap = (size_t)(std::min<int64_t>(perChunk, nViews) * KN);
  CU(ctx->dViews.reserve((size_t)nViews));
  CU(cudaMemcpyAsync(ctx->dViews.p, cams.data(), sizeof(B2Camera) * (size_t)nViews, cudaMemcpyHostToDevice,
                     ctx->stream));
  if (albedoOut)
    CU(ctx->featAlbedo.reserve(cap));
  if (normalDepthOut)
    CU(ctx->featNormalDepth.reserve(cap));
  for (int64_t v0 = 0; v0 < nViews; v0 += perChunk)
  {
    const int nv = (int)std::min<int64_t>(perChunk, nViews - v0);
    const int64_t n = nv * N; // one slice of the chunk
    CU(b2pt::launch_view_features(ctx->useBvh ? nullptr : &ctx->small, ctx->useBvh ? &ctx->bvh : nullptr,
                                  ctx->dViews.p + v0, nv, (int)N, ctx->seedOffset, ck,
                                  albedoOut ? ctx->featAlbedo.p : nullptr,
                                  normalDepthOut ? ctx->featNormalDepth.p : nullptr, ctx->stream));
    for (int k = 0; k < K; ++k)
    {
      const size_t dst = 4 * (size_t)((k * (int64_t)nViews + v0) * N);
      if (albedoOut)
        CU(cudaMemcpyAsync(albedoOut + dst, ctx->featAlbedo.p + k * n, sizeof(float4) * (size_t)n,
                           cudaMemcpyDeviceToHost, ctx->stream));
      if (normalDepthOut)
        CU(cudaMemcpyAsync(normalDepthOut + dst, ctx->featNormalDepth.p + k * n, sizeof(float4) * (size_t)n,
                           cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

void b2pt_denoise_defaults(b2pt_denoise_params* p)
{
  if (!p)
    return;
  p->levels = 5;
  p->sigmaLum = 4.f;
  p->sigmaAlbedo = 0.1f;
  p->sigmaNormal = 0.3f;
  p->sigmaDepth = 2.f;
}

// Spatial denoiser of a sweep (k_denoise_prep, then one k_atrous per level).  Views run in chunks of whole views: per
// chunk, K host-to-device copies of each input into the context's staging [k][chunk view][pixel] (at most
// max(kDenoiseChunkFloat4, K*W*H) float4 per buffer), the launches, and K copies of the result back.  The colour sums
// land in dnX[0] and the sums of squares in dnX[1]; the prep turns dnX[0] into (m, V0) and the guide sums into the
// guides in place, and the levels ping-pong between dnX[0] and dnX[1].  Every image is filtered on its own, so the
// result does not depend on the chunking.
static constexpr int64_t kDenoiseChunkFloat4 = (int64_t)1 << 23;
int b2pt_denoise_views(b2pt_ctx* ctx, int nViews, int W, int H, int nCheckpoints, const int* checkpoints,
                       const float* color, const float* moment2, const float* albedo, const float* normalDepth,
                       const b2pt_denoise_params* params, uint32_t flags, void* out)
{
  static const char* const fn = "b2pt_denoise_views";
  if (int rc = bind(ctx))
    return rc;
  if (nViews < 0)
    return fail(B2PT_ERR_BAD_VALUE, "%s: negative view count", fn);
  if (int rc = check_checkpoints(fn, nCheckpoints, checkpoints))
    return rc;
  if (!color || !albedo || !normalDepth || !out)
    return fail(B2PT_ERR_BAD_VALUE, "%s: color, albedo, normalDepth and out must not be NULL", fn);
  if (W <= 0 || H <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "%s: W and H must be positive", fn);
  b2pt_denoise_params P;
  if (params)
    P = *params;
  else
    b2pt_denoise_defaults(&P);
  if (P.levels < 0 || P.levels > 10)
    return fail(B2PT_ERR_BAD_VALUE, "%s: levels must be in [0,10], got %d", fn, P.levels);
  const float sigma[4] = { P.sigmaLum, P.sigmaAlbedo, P.sigmaNormal, P.sigmaDepth };
  const char* const sigmaName[4] = { "sigmaLum", "sigmaAlbedo", "sigmaNormal", "sigmaDepth" };
  for (int s = 0; s < 4; ++s)
    if (!(sigma[s] > 0.f)) // NaN fails too
      return fail(B2PT_ERR_BAD_VALUE, "%s: %s must be > 0 (or +inf), got %g", fn, sigmaName[s], (double)sigma[s]);
  if (flags & ~B2PT_FLAG_VIEWS_PNM16)
    return fail(B2PT_ERR_BAD_VALUE, "%s: flags may only hold VIEWS_PNM16", fn);
  const int K = nCheckpoints;
  const int64_t N = (int64_t)W * H, KN = N * K;
  if (KN > ((int64_t)1 << 30))
    return fail(B2PT_ERR_BAD_VALUE, "%s: one view's %d slices exceed 2^30 float4", fn, K);
  if (nViews == 0)
    return B2PT_OK;
  const bool pnm = (flags & B2PT_FLAG_VIEWS_PNM16) != 0;
  b2pt::DenoiseArgs a{};
  a.n = K;
  std::copy(checkpoints, checkpoints + K, a.count);
  a.hasMoments = moment2 != nullptr;
  a.sigmaLum = P.sigmaLum, a.sigmaAlbedo = P.sigmaAlbedo, a.sigmaNormal = P.sigmaNormal, a.sigmaDepth = P.sigmaDepth;
  const int64_t perChunk = std::max<int64_t>(1, kDenoiseChunkFloat4 / KN);
  const size_t cap = (size_t)(std::min<int64_t>(perChunk, nViews) * KN);
  CU(ctx->dnX[0].reserve(cap));
  CU(ctx->dnX[1].reserve(cap));
  CU(ctx->dnGuideA.reserve(cap));
  CU(ctx->dnGuideNZ.reserve(cap));
  if (pnm)
    CU(ctx->pnm.reserve(cap * 3));
  const float* const in[4] = { color, moment2, albedo, normalDepth };
  float4* const stage[4] = { ctx->dnX[0].p, ctx->dnX[1].p, ctx->dnGuideA.p, ctx->dnGuideNZ.p };
  for (int64_t v0 = 0; v0 < nViews; v0 += perChunk)
  {
    const int nv = (int)std::min<int64_t>(perChunk, nViews - v0);
    const int64_t n = nv * N; // one slice of the chunk
    for (int b = 0; b < 4; ++b)
      for (int k = 0; in[b] && k < K; ++k)
        CU(cudaMemcpyAsync(stage[b] + k * n, in[b] + 4 * (size_t)((k * (int64_t)nViews + v0) * N),
                           sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    a.nViews = nv;
    CU(b2pt::launch_denoise_prep(ctx->dnX[0].p, moment2 ? ctx->dnX[1].p : nullptr, ctx->dnGuideA.p, ctx->dnGuideNZ.p,
                                 (int)N, a, ctx->stream));
    int cur = 0;
    for (int level = 0; level < P.levels; ++level, cur ^= 1)
      CU(b2pt::launch_atrous(ctx->dnX[cur].p, ctx->dnX[cur ^ 1].p, ctx->dnGuideA.p, ctx->dnGuideNZ.p, W, H, 1 << level,
                             a, ctx->stream));
    const float4* res = ctx->dnX[cur].p;
    if (pnm)
      CU(b2pt::launch_pnm16(res, n * K, 1, ctx->pnm.p, ctx->stream));
    for (int k = 0; k < K; ++k)
    {
      const size_t dst = (size_t)((k * (int64_t)nViews + v0) * N);
      if (pnm)
        CU(cudaMemcpyAsync(static_cast<uint16_t*>(out) + 3 * dst, ctx->pnm.p + 3 * k * n, sizeof(uint16_t) * 3 * (size_t)n,
                           cudaMemcpyDeviceToHost, ctx->stream));
      else
        CU(cudaMemcpyAsync(static_cast<float4*>(out) + dst, res + k * n, sizeof(float4) * (size_t)n,
                           cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

void* b2pt_views_device_ptr(b2pt_ctx* ctx)
{
  if (bind(ctx) != B2PT_OK || ctx->viewCount == 0)
    return nullptr;
  return ctx->viewColor.p;
}

int b2pt_render(b2pt_ctx* ctx, int spp, int maxDepth, uint32_t flags)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "render before b2pt_set_camera");
  if (int rc = b2pt_clear_color(ctx)) // MapperPathTracer.cxx:222-223
    return rc;
  return b2pt_render_range(ctx, 0, spp, maxDepth, flags);
}

int b2pt_synchronize(b2pt_ctx* ctx)
{
  if (int rc = bind(ctx))
    return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

int b2pt_get_stats(b2pt_ctx* ctx, b2pt_stats* out)
{
  if (int rc = bind(ctx))
    return rc;
  if (!out)
    return fail(B2PT_ERR_BAD_VALUE, "null stats pointer");
  if (ctx->statsPending)
  {
    CU(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ctx->evStart, ctx->evStop));
    ctx->stats.renderMs = ms;
    ctx->hCounters.resize((size_t)std::max<int64_t>(ctx->pendingCounters, 1));
    if (ctx->pendingCounters > 0)
      CU(cudaMemcpy(ctx->hCounters.data(), ctx->counters.p, sizeof(uint32_t) * (size_t)ctx->pendingCounters,
                    cudaMemcpyDeviceToHost));
    int64_t seg = ctx->stats.paths; // every path traces its primary segment
    for (int64_t k = 0; k < ctx->pendingCounters; ++k)
      seg += ctx->hCounters[(size_t)k]; // rays entering bounce d+1 (0 for the last depth)
    ctx->stats.segments = seg;
    // queue traffic: a survivor is written (48 B) and read (48 B) on the ray queue and once more as a binned
    // ray+hit record (52 B written, 52 B read); radiance 16 B written + read per path
    ctx->stats.queueBytes = (seg - ctx->stats.paths) * 96 + seg * 104 + ctx->stats.paths * 32;
    unsigned long long nan = 0;
    CU(cudaMemcpy(&nan, ctx->nanCounter.p, sizeof(nan), cudaMemcpyDeviceToHost));
    ctx->stats.nanSamples = (int64_t)nan;
    ctx->statsPending = false;
  }
  *out = ctx->stats;
  return B2PT_OK;
}

int b2pt_get_bounce_profile(b2pt_ctx* ctx, int maxEntries, float* ms, int64_t* raysIn)
{
  if (int rc = bind(ctx))
    return rc;
  if (maxEntries < 0 || (maxEntries > 0 && (!ms || !raysIn)))
    return fail(B2PT_ERR_BAD_VALUE, "null profile output");
  b2pt_stats st;
  if (int rc = b2pt_get_stats(ctx, &st)) // synchronises and fetches the counters
    return rc;
  const int n = std::min(maxEntries, ctx->profDepths);
  for (int d = 0; d < n; ++d)
  {
    CU(cudaEventElapsedTime(&ms[d], ctx->evBounce[d], ctx->evBounce[d + 1]));
    raysIn[d] = d == 0 ? ctx->profPaths : (int64_t)ctx->hCounters[(size_t)(d - 1)];
  }
  return n;
}

int b2pt_get_stage_profile(b2pt_ctx* ctx, int maxEntries, float* traceMs, float* shadeMs, int64_t* raysIn)
{
  if (int rc = bind(ctx))
    return rc;
  if (maxEntries < 0 || (maxEntries > 0 && (!traceMs || !shadeMs || !raysIn)))
    return fail(B2PT_ERR_BAD_VALUE, "null profile output");
  b2pt_stats st;
  if (int rc = b2pt_get_stats(ctx, &st)) // synchronises and fetches the counters
    return rc;
  const int n = std::min(maxEntries, ctx->profDepths);
  for (int d = 0; d < n; ++d)
  {
    CU(cudaEventElapsedTime(&traceMs[d], ctx->evBounce[d], ctx->evMid[d]));
    CU(cudaEventElapsedTime(&shadeMs[d], ctx->evMid[d], ctx->evBounce[d + 1]));
    raysIn[d] = d == 0 ? ctx->profPaths : (int64_t)ctx->hCounters[(size_t)(d - 1)];
  }
  return n;
}

int b2pt_read_color(b2pt_ctx* ctx, float* rgba)
{
  if (int rc = bind(ctx))
    return rc;
  if (!rgba)
    return fail(B2PT_ERR_BAD_VALUE, "null output");
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_read_color before b2pt_set_camera");
  if (int rc = ensure_color(ctx))
    return rc;
  CU(cudaMemcpyAsync(rgba, ctx->color(), sizeof(float4) * (size_t)ctx->cam.W * ctx->cam.H, cudaMemcpyDeviceToHost,
                     ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

int b2pt_write_color(b2pt_ctx* ctx, const float* rgba)
{
  if (int rc = bind(ctx))
    return rc;
  if (!rgba)
    return fail(B2PT_ERR_BAD_VALUE, "null input");
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_write_color before b2pt_set_camera");
  if (int rc = ensure_color(ctx))
    return rc;
  CU(cudaMemcpyAsync(ctx->color(), rgba, sizeof(float4) * (size_t)ctx->cam.W * ctx->cam.H, cudaMemcpyHostToDevice,
                     ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

int b2pt_normalize(b2pt_ctx* ctx, int spp)
{
  if (int rc = bind(ctx))
    return rc;
  if (spp <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "spp must be positive");
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_normalize before b2pt_set_camera");
  if (int rc = ensure_color(ctx))
    return rc;
  CU(b2pt::launch_normalize(ctx->color(), (int64_t)ctx->cam.W * ctx->cam.H, spp, ctx->stream));
  return B2PT_OK;
}

int b2pt_read_pnm16(b2pt_ctx* ctx, int spp, uint16_t* rgb)
{
  if (int rc = bind(ctx))
    return rc;
  if (spp <= 0)
    return fail(B2PT_ERR_BAD_VALUE, "spp must be positive");
  if (!rgb)
    return fail(B2PT_ERR_BAD_VALUE, "null output");
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_read_pnm16 before b2pt_set_camera");
  if (int rc = ensure_color(ctx))
    return rc;
  const int64_t N = (int64_t)ctx->cam.W * ctx->cam.H;
  CU(ctx->pnm.reserve((size_t)N * 3));
  CU(b2pt::launch_pnm16(ctx->color(), N, spp, ctx->pnm.p, ctx->stream));
  CU(cudaMemcpyAsync(rgb, ctx->pnm.p, sizeof(uint16_t) * 3 * (size_t)N, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

static int ensure_trace(b2pt_ctx* ctx);

// G-buffers of nViews views of N pixels each (views: host array), written to the host arrays at [view][pixel].  Chunks
// of whole views, at most kDirectChunkPixels pixels unless one view alone is larger, run one launch each into the
// context's staging buffers, whose contents are then copied to the chunk's slice of the outputs.
static constexpr int64_t kDirectChunkPixels = (int64_t)1 << 22;
static int render_direct_chunks(b2pt_ctx* ctx, int nViews, const b2pt::DirectView* views, int64_t N, float* normals,
                                float* albedo, float* depth, int32_t* primId)
{
  if (int rc = ensure_trace(ctx))
    return rc;
  B2BvhScene bvh = ctx->bvh;
  if (bvh.wide)
    bvh.primSlots = ctx->dBinSlots.p; // the binary tree's leaf order (the wide tree rewrote dSlots)
  const int64_t perChunk = std::max<int64_t>(1, kDirectChunkPixels / N);
  const size_t cap = (size_t)(std::min<int64_t>(perChunk, nViews) * N);
  CU(ctx->dDirectViews.reserve((size_t)nViews));
  CU(cudaMemcpyAsync(ctx->dDirectViews.p, views, sizeof(b2pt::DirectView) * (size_t)nViews, cudaMemcpyHostToDevice,
                     ctx->stream));
  if (normals)
    CU(ctx->directNormals.reserve(cap));
  if (albedo)
    CU(ctx->directAlbedo.reserve(cap));
  if (depth)
    CU(ctx->directDepth.reserve(cap));
  if (primId)
    CU(ctx->directPrim.reserve(cap));
  for (int64_t v0 = 0; v0 < nViews; v0 += perChunk)
  {
    const int nv = (int)std::min<int64_t>(perChunk, nViews - v0);
    const size_t n = (size_t)(nv * N), off = (size_t)(v0 * N);
    CU(b2pt::launch_direct_views(ctx->useBvh ? nullptr : &ctx->small, ctx->useBvh ? &bvh : nullptr,
                                 ctx->dDirectViews.p + v0, nv, (int)N, normals ? ctx->directNormals.p : nullptr,
                                 albedo ? ctx->directAlbedo.p : nullptr, depth ? ctx->directDepth.p : nullptr,
                                 primId ? ctx->directPrim.p : nullptr, ctx->stream));
    if (normals)
      CU(cudaMemcpyAsync(normals + 4 * off, ctx->directNormals.p, n * sizeof(float4), cudaMemcpyDeviceToHost,
                         ctx->stream));
    if (albedo)
      CU(cudaMemcpyAsync(albedo + 4 * off, ctx->directAlbedo.p, n * sizeof(float4), cudaMemcpyDeviceToHost,
                         ctx->stream));
    if (depth)
      CU(cudaMemcpyAsync(depth + off, ctx->directDepth.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (primId)
      CU(cudaMemcpyAsync(primId + off, ctx->directPrim.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return B2PT_OK;
}

int b2pt_render_direct(b2pt_ctx* ctx, float* normals, float* albedo, float* depth, int32_t* primId)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_render_direct before b2pt_set_camera");
  b2pt::DirectView v;
  v.cam = ctx->cam;
  for (int c = 0; c < 3; ++c)
    v.lookAt[c] = ctx->camLookAt[c], v.upN[c] = ctx->camUpN[c];
  return render_direct_chunks(ctx, 1, &v, (int64_t)ctx->cam.W * ctx->cam.H, normals, albedo, depth, primId);
}

int b2pt_render_direct_views(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, float* normals,
                             float* albedo, float* depth, int32_t* primId)
{
  if (int rc = bind(ctx))
    return rc;
  if (int rc = check_view_list("b2pt_render_direct_views", nViews, views))
    return rc;
  std::vector<B2Camera> cams;
  if (int rc = make_view_cameras(nViews, views, W, H, cams))
    return rc;
  std::vector<b2pt::DirectView> dv((size_t)nViews);
  for (int v = 0; v < nViews; ++v)
  {
    const float* p = views + 10 * (size_t)v;
    b2pt::DirectView& d = dv[(size_t)v];
    d.cam = cams[(size_t)v];
    for (int c = 0; c < 3; ++c)
      d.lookAt[c] = p[3 + c];
    stored_up(p + 6, d.upN);
  }
  if (nViews == 0)
    return B2PT_OK;
  return render_direct_chunks(ctx, nViews, dv.data(), (int64_t)W * H, normals, albedo, depth, primId);
}

// The trace structures for a call without build flags: the ones built last (the default ones if none were), up to
// date with b2pt_update_spheres.
static int ensure_trace(b2pt_ctx* ctx)
{
  if (!ctx->haveScene)
    return fail(B2PT_ERR_STATE, "scene not set");
  if (!ctx->haveBvh)
  {
    if (int rc = build_trace_structures(ctx, 0))
      return rc;
    ctx->haveBvh = true;
  }
  return refresh_stale_tree(ctx);
}

int b2pt_primary_hits(b2pt_ctx* ctx, int32_t* primId, float* t)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_primary_hits before b2pt_set_camera");
  if (int rc = ensure_trace(ctx))
    return rc;
  const size_t N = (size_t)ctx->cam.W * ctx->cam.H;
  DevBuf<int32_t> dPrim;
  DevBuf<float> dT;
  CU(dPrim.reserve(N));
  CU(dT.reserve(N));
  cudaError_t e = b2pt::launch_primary_hits(ctx->cam, ctx->useBvh ? nullptr : &ctx->small,
                                            ctx->useBvh ? &ctx->bvh : nullptr, ctx->seedOffset, dPrim.p, dT.p,
                                            ctx->stream);
  if (e == cudaSuccess && primId)
    e = cudaMemcpyAsync(primId, dPrim.p, N * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && t)
    e = cudaMemcpyAsync(t, dT.p, N * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(ctx->stream);
  dPrim.release();
  dT.release();
  if (e != cudaSuccess)
    return fail(B2PT_ERR_CUDA, "b2pt_primary_hits: %s", cudaGetErrorString(e));
  return B2PT_OK;
}

int b2pt_create_rays(b2pt_ctx* ctx, uint32_t* seedsInOut, float* dirX, float* dirY, float* dirZ, float* originX,
                     float* originY, float* originZ, int64_t* pixelIdx)
{
  if (int rc = bind(ctx))
    return rc;
  if (!ctx->haveCamera)
    return fail(B2PT_ERR_STATE, "b2pt_create_rays before b2pt_set_camera");
  if (!seedsInOut)
    return fail(B2PT_ERR_BAD_VALUE, "null seeds");
  if ((dirX || dirY || dirZ) && !(dirX && dirY && dirZ))
    return fail(B2PT_ERR_BAD_VALUE, "direction outputs must be all set or all null");
  if ((originX || originY || originZ) && !(originX && originY && originZ))
    return fail(B2PT_ERR_BAD_VALUE, "origin outputs must be all set or all null");
  const size_t N = (size_t)ctx->cam.W * ctx->cam.H;
  DevBuf<uint32_t> dSeeds;
  DevBuf<float> dF; // 6 planes
  DevBuf<long long> dPix;
  CU(dSeeds.reserve(N));
  CU(dF.reserve(6 * N));
  CU(dPix.reserve(N));
  cudaError_t e = cudaMemcpyAsync(dSeeds.p, seedsInOut, N * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess)
    e = b2pt::launch_create_rays(ctx->cam, dSeeds.p, dF.p, dF.p + N, dF.p + 2 * N, dF.p + 3 * N, dF.p + 4 * N,
                                 dF.p + 5 * N, dPix.p, ctx->stream);
  auto back = [&](void* dst, const void* src, size_t bytes) {
    if (e == cudaSuccess && dst)
      e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
  };
  back(seedsInOut, dSeeds.p, N * sizeof(uint32_t));
  back(dirX, dF.p, N * 4), back(dirY, dF.p + N, N * 4), back(dirZ, dF.p + 2 * N, N * 4);
  back(originX, dF.p + 3 * N, N * 4), back(originY, dF.p + 4 * N, N * 4), back(originZ, dF.p + 5 * N, N * 4);
  back(pixelIdx, dPix.p, N * sizeof(long long));
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(ctx->stream);
  dSeeds.release(), dF.release(), dPix.release();
  if (e != cudaSuccess)
    return fail(B2PT_ERR_CUDA, "b2pt_create_rays: %s", cudaGetErrorString(e));
  return B2PT_OK;
}

int b2pt_intersect(b2pt_ctx* ctx, int64_t n, const float* ox, const float* oy, const float* oz, const float* dx,
                   const float* dy, const float* dz, float tmin, float tmax, int32_t* primId, float* hrec9,
                   int32_t* matId, int32_t* texId)
{
  if (int rc = bind(ctx))
    return rc;
  if (n < 0)
    return fail(B2PT_ERR_BAD_VALUE, "negative ray count");
  if (n == 0)
    return B2PT_OK;
  if (!ox || !oy || !oz || !dx || !dy || !dz || !primId)
    return fail(B2PT_ERR_BAD_VALUE, "null ray array");
  if (int rc = ensure_trace(ctx))
    return rc;
  const size_t N = (size_t)n;
  DevBuf<float> dIn, dRec;
  DevBuf<int32_t> dIds;
  CU(dIn.reserve(6 * N));
  CU(dRec.reserve(9 * N));
  CU(dIds.reserve(3 * N));
  const float* src[6] = { ox, oy, oz, dx, dy, dz };
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < 6 && e == cudaSuccess; ++k)
    e = cudaMemcpyAsync(dIn.p + k * N, src[k], N * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess)
    e = b2pt::launch_intersect(ctx->useBvh ? nullptr : &ctx->small, ctx->useBvh ? &ctx->bvh : nullptr, n, dIn.p,
                               dIn.p + N, dIn.p + 2 * N, dIn.p + 3 * N, dIn.p + 4 * N, dIn.p + 5 * N, tmin, tmax,
                               dIds.p, dRec.p, dIds.p + N, dIds.p + 2 * N, ctx->stream);
  auto back = [&](void* dst, const void* s, size_t bytes) {
    if (e == cudaSuccess && dst)
      e = cudaMemcpyAsync(dst, s, bytes, cudaMemcpyDeviceToHost, ctx->stream);
  };
  back(primId, dIds.p, N * 4), back(matId, dIds.p + N, N * 4), back(texId, dIds.p + 2 * N, N * 4);
  back(hrec9, dRec.p, 9 * N * 4);
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(ctx->stream);
  dIn.release(), dRec.release(), dIds.release();
  if (e != cudaSuccess)
    return fail(B2PT_ERR_CUDA, "b2pt_intersect: %s", cudaGetErrorString(e));
  return B2PT_OK;
}

int b2pt_allreduce(b2pt_ctx* const* ctxs, int G)
{
  if (!ctxs || G < 1 || G > 8)
    return fail(B2PT_ERR_BAD_VALUE, "b2pt_allreduce needs 1..8 contexts");
  if (G == 1)
    return B2PT_OK;
  const int W = ctxs[0]->cam.W, H = ctxs[0]->cam.H;
  for (int g = 0; g < G; ++g)
  {
    if (!ctxs[g] || !ctxs[g]->haveCamera || ctxs[g]->cam.W != W || ctxs[g]->cam.H != H)
      return fail(B2PT_ERR_BAD_VALUE, "contexts must share one canvas size");
    if (int rc = bind(ctxs[g]))
      return rc;
    if (int rc = ensure_color(ctxs[g]))
      return rc;
    CU(cudaStreamSynchronize(ctxs[g]->stream));
  }
  // peer access over NVLink (idempotent)
  for (int a = 0; a < G; ++a)
    for (int b = 0; b < G; ++b)
      if (a != b && ctxs[a]->device != ctxs[b]->device)
      {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, ctxs[a]->device, ctxs[b]->device));
        if (!can)
          return fail(B2PT_ERR_UNSUPPORTED, "no peer access between devices %d and %d", ctxs[a]->device,
                      ctxs[b]->device);
        CU(cudaSetDevice(ctxs[a]->device));
        cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[b]->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled)
          cudaGetLastError();
        else if (e != cudaSuccess)
          return fail(B2PT_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
      }
  const int64_t n = (int64_t)W * H;
  std::vector<DevBuf<float4>> tmp((size_t)G);
  const float4* srcs[8];
  for (int g = 0; g < G; ++g)
    srcs[g] = ctxs[g]->color();
  // reduce-scatter: GPU g sums slice g of every peer into a private slice buffer (reads cross NVLink) ...
  for (int g = 0; g < G; ++g)
  {
    const int64_t b = n * g / G, e = n * (g + 1) / G;
    CU(cudaSetDevice(ctxs[g]->device));
    CU(tmp[(size_t)g].reserve((size_t)std::max<int64_t>(e - b, 1)));
    CU(b2pt::launch_sum_peers(tmp[(size_t)g].p, srcs, G, b, e, ctxs[g]->stream));
  }
  for (int g = 0; g < G; ++g)
  {
    CU(cudaSetDevice(ctxs[g]->device));
    CU(cudaStreamSynchronize(ctxs[g]->stream));
  }
  // ... all-gather: every GPU's reduced slice is copied to every context's buffer
  for (int g = 0; g < G; ++g)
  {
    const int64_t b = n * g / G, e = n * (g + 1) / G;
    CU(cudaSetDevice(ctxs[g]->device));
    for (int d = 0; d < G; ++d)
      CU(cudaMemcpyPeerAsync(ctxs[d]->color() + b, ctxs[d]->device, tmp[(size_t)g].p, ctxs[g]->device,
                             sizeof(float4) * (size_t)(e - b), ctxs[g]->stream));
  }
  for (int g = 0; g < G; ++g)
  {
    CU(cudaSetDevice(ctxs[g]->device));
    CU(cudaStreamSynchronize(ctxs[g]->stream));
    tmp[(size_t)g].release();
  }
  return B2PT_OK;
}

} // extern "C"
