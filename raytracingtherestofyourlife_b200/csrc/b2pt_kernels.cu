// b2pt_kernels.cu -- hand-written sm_100a kernels of the wavefront path tracer.
//
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (see _build.py).
//
//   k_trace<PRIMARY,Scene,TAIL>   K1+K2: load ray (3x16 B, coalesced; PRIMARY: generate it from (pixel, sample) with
//                                 the wang-hash RNG, primary rays never touch HBM) -> closest hit -> paths that miss
//                                 or land on an emitter finish (radiance written once, 16 B) -> every other hit is
//                                 appended with its ray to one of four bins by shading strategy.
//                                 Small scenes: two-phase candidate filter (b2pt_device.cuh closest_small);
//                                 BVH scenes: persistent lanes with ray replacement (trace_body_bvh).
//   k_shade<Scene,TAIL_IN,GLOBAL_OUT>  K3+K5: fused material / direction sampling / light pdfs / mixture pdf on 32
//                                 records of ONE bin (warp-uniform), survivors compacted into the ray queue.
//   k_tail_loop<Scene>            every remaining bounce of a batch in one launch of one 8-CTA cluster.
//   k_accumulate                  per pixel: sum the batch's samples in registers (sample order) and do a
//                                 single read-modify-write of the canvas float4.
//   k_accumulate_checkpoints      the same loop, also storing the running sum (and sum of squares) at chosen sample
//                                 counts: the images of several sample counts from one render.
//   k_primary_hits                parity hook: production raygen + trace, writes hit primitive id / t.
//   k_view_features<Scene>        per (view, pixel): albedo, normal and depth of the primary hits of its path samples,
//                                 summed in sample order and stored at chosen sample counts (denoiser guides).
//   k_create_rays, k_intersect, k_normalize, k_pnm16, k_fill_seeds, k_sum_peers: stage-level API kernels.
//
// Work distribution: queue and bins are statically partitioned into one region per persistent warp
// (numSMs x occupancy x 8 regions); a warp consumes and refills only its own region with register counters
// (ballot + popcount prefix), no atomics.  TAIL instantiations (deep bounces) use one flat global queue and
// global bins with one warp-aggregated atomicAdd per 32-ray tile.  All counts live in device memory: no host
// round trip sits between bounces.
#include "b2pt_device.cuh"
#include "b2pt_kernels.h"

#include <algorithm>
#include <cooperative_groups.h>
#include <cub/device/device_scan.cuh>
#include <type_traits>

namespace b2pt
{

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
#ifndef B2PT_MIN_BLOCKS
#define B2PT_MIN_BLOCKS 4
#endif
constexpr int kMinBlocksPerSM = B2PT_MIN_BLOCKS; // register cap = 65536 / (256 * blocks)
#ifndef B2PT_TRACE_MIN_BLOCKS
#define B2PT_TRACE_MIN_BLOCKS 4
#endif
constexpr int kTraceMinBlocksPerSM = B2PT_TRACE_MIN_BLOCKS;
// the deep tail of a batch runs inside one launch of a single thread-block cluster (k_tail_loop, k_bounce_tail_loop)
constexpr int kTailCluster = 8;
constexpr int kTailBlock = 512;

struct PeerPtrs
{
  const float4* p[8];
};

// L2 prefetch of the 16-byte element a lane will load in its NEXT iteration (hides part of the HBM latency at the
// head of every tile; the kernels keep only 8 warps per scheduler)
#ifndef B2PT_PREFETCH_AHEAD
#define B2PT_PREFETCH_AHEAD 32
#endif
constexpr int kPrefetchAhead = B2PT_PREFETCH_AHEAD; // records ahead of the one being processed (a warp's next tile = 32)
__device__ __forceinline__ void prefetch_l2(const void* p)
{
#ifndef B2PT_NO_PREFETCH
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}

__device__ __forceinline__ void store_ray(const B2Queue& q, int64_t pos, f3 o, f3 d, f3 T, uint32_t pid, uint32_t rng)
{
  q.p0[pos] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
  q.p1[pos] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
  q.p2[pos] = make_uint4(__float_as_uint(T.z), pid, rng, 0u);
}

// Shared-memory staging of the per-launch tables.  The small scene (about 11 KB) and the light tables are
// copied; a BVH scene is a handful of pointers and stays in the parameter bank.
template <class SceneT>
struct StageArea
{
  B2Lights lights;
};
template <>
struct StageArea<B2SmallScene>
{
  B2SmallScene scene;
  B2Lights lights;
};
template <class T>
__device__ __forceinline__ void stage_copy(T& dst, const T& src)
{
  static_assert(sizeof(T) % 16 == 0, "staged tables are multiples of 16 bytes");
  uint4* d = reinterpret_cast<uint4*>(&dst);
  const uint4* s = reinterpret_cast<const uint4*>(&src);
  for (int i = threadIdx.x; i < (int)(sizeof(T) / 16); i += blockDim.x)
    d[i] = s[i];
}
__device__ __forceinline__ const B2SmallScene& stage_scene(const B2SmallScene& scene, StageArea<B2SmallScene>& a)
{
  stage_copy(a.scene, scene);
  return a.scene;
}
__device__ __forceinline__ const B2BvhScene& stage_scene(const B2BvhScene& scene, StageArea<B2BvhScene>&)
{
  return scene;
}
__device__ __forceinline__ const B2WideScene& stage_scene(const B2WideScene& scene, StageArea<B2WideScene>&)
{
  return scene;
}
template <class SceneT>
__device__ __forceinline__ const B2Lights& stage_lights(const B2Lights& lights, StageArea<SceneT>& a)
{
  stage_copy(a.lights, lights);
  return a.lights;
}

// x[k] for k in 0..3 without a branch tree (the compiler turns the ternary chain over two quadruples into divergent
// branches; three selects per quadruple keep the warp together)
__device__ __forceinline__ uint32_t pick4(int k, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3)
{
  uint32_t r;
  asm("{ .reg .pred p0, p1, p2; setp.eq.s32 p0, %1, 0; setp.eq.s32 p1, %1, 1; setp.eq.s32 p2, %1, 2;\n\t"
      "selp.b32 %0, %4, %5, p2; selp.b32 %0, %3, %0, p1; selp.b32 %0, %2, %0, p0; }"
      : "=&r"(r)
      : "r"(k), "r"(x0), "r"(x1), "r"(x2), "r"(x3));
  return r;
}

// Global tile (32 consecutive path ids) that warp w generates in round j of a PRIMARY launch: slot (w + j) mod numWarps
// of round j.  For a fixed round the slots of the warps are a permutation, so every tile is generated exactly once.
__device__ __forceinline__ int64_t primary_tile(int64_t j, int w, int numWarps)
{
  return j * numWarps + (int64_t)(((int64_t)w + j) % numWarps);
}

// n / d for the divisors the host prepared (B2RenderArgs::div*): Granlund-Montgomery round-up with the 33rd bit of the
// multiplier folded into an add and a shift; exact for every 32-bit n (tests/test_host_logic.py checks the recipe)
__device__ __forceinline__ uint32_t fastdiv(uint32_t n, uint32_t magic, uint32_t shift)
{
  if (shift == 0xffffffffu)
    return n; // divisor 1
  const uint32_t t = __umulhi(n, magic);
  return (t + ((n - t) >> 1)) >> shift;
}

// Ray `idx` of the warp's region.  PRIMARY: generated from (pixel, sample) -- idx is the path id.
template <bool PRIMARY>
__device__ __forceinline__ void load_ray(const B2Camera& cam, const B2RenderArgs& A, int64_t idx, f3& o, f3& d, f3& T,
                                         uint32_t& pid, uint32_t& rng, uint32_t* slotOut = nullptr)
{
  if (PRIMARY)
  {
    pid = (uint32_t)idx; // path id chosen by the caller (tile-interleaved over the warps' regions)
    uint32_t b = fastdiv(pid, A.divPixelsMagic, A.divPixelsShift); // sample slot of the batch
    const uint32_t pixel = pid - b * (uint32_t)A.nPixels;
    if (slotOut)
      *slotOut = b;
    if (A.views)
    { // view-batched render: every view is an independent render with the same per-(pixel, sample) streams
      const uint32_t view = fastdiv(b, A.divSppMagic, A.divSppShift);
      const B2Camera vc = A.views[view];
      b = b - view * (uint32_t)A.sppPerView;
      rng = pixel + A.seedOffset + (uint32_t)(A.sampleBase + (int)b) * B2PT_GOLDEN;
      d = raygen(vc, (int)pixel, rng);
      o = ld3(vc.pos);
    }
    else
    {
      // MapperPathTracer.cxx:265-267: seeds[i] = i.  Production stream: one stream per (pixel, sample).
      rng = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV)
        ? A.seeds[pixel]
        : pixel + A.seedOffset + (uint32_t)(A.sampleBase + (int)b) * B2PT_GOLDEN;
      d = raygen(cam, (int)pixel, rng);
      o = ld3(cam.pos);
    }
    T = mk3(1.f, 1.f, 1.f);
  }
  else
  {
    // .cg loads: queue data is streamed once, and the persistent tail kernel re-reads addresses that other
    // SMs rewrote earlier in the same launch (L1 is not coherent)
    const uint4 a = __ldcg(A.q.p0 + idx);
    const uint4 b = __ldcg(A.q.p1 + idx);
    const uint4 c = __ldcg(A.q.p2 + idx);
    o = mk3(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
    d = mk3(__uint_as_float(a.w), __uint_as_float(b.x), __uint_as_float(b.y));
    T = mk3(__uint_as_float(b.z), __uint_as_float(b.w), __uint_as_float(c.x));
    pid = c.y;
    rng = c.z;
  }
}

// Finished path: radiance written once; in reference-stream mode the pixel's persistent RNG state is advanced
// past the draws the reference still consumes for a dead pixel (SURVEY A.3).
__device__ __forceinline__ void finish_path(const B2RenderArgs& A, uint32_t pid, f3 L, uint32_t rng, bool refStream,
                                            int depthsToBurn)
{
  A.rad[pid] = make_float4(L.x, L.y, L.z, 0.f);
  if (refStream)
  {
    burn_depths(rng, depthsToBurn, A.nLightQuads, A.nLightSph);
    A.seeds[pid % (uint32_t)A.nPixels] = rng;
  }
}

// ---- spatial sorting of the ray queue (BVH scenes).  Incoherent secondary rays make every lane of a warp walk its
// own root-to-leaf path: dependent node fetches that miss L1, lanes that drift apart.  Between k_shade and k_trace the
// queue is therefore bucketed by the ray origin's cell (64^3 Morton cells of the scene box) and direction octant --
// a counting sort: k_sort_keys (keys + histogram), an exclusive scan, k_sort_scatter (permutation) -- and k_trace deals
// each warp a contiguous chunk of the sorted order, so the rays a warp traces together start in one neighbourhood and
// share most of their descent.  The rays themselves stay where k_shade put them (one 4-byte index per ray moves).
// Which rays share a warp never changes a result: every path's arithmetic and its radiance slot are its own.
constexpr int kSortCellBits = 6;                                   // cells per axis = 64
constexpr int kSortBuckets = 1 << (3 * kSortCellBits + 3);         // x octants = 2 Mi buckets
__device__ __forceinline__ int64_t sorted_chunk(const B2RenderArgs& A, int depth)
{
  if (!A.perm || depth < 1)
    return 0;
  const int64_t total = (int64_t)A.depthTotals[depth - 1];
  return (((total + A.numWarps - 1) / A.numWarps) + 31) & ~(int64_t)31;
}
__device__ __forceinline__ uint32_t spread3(uint32_t v)
{ // 6 bits -> every third bit
  v = (v | (v << 8)) & 0x0300F00Fu;
  v = (v | (v << 4)) & 0x030C30C3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}
struct SortBox
{
  float lo[3], cellsPerUnit[3];
};
template <bool SCATTER>
__global__ void __launch_bounds__(kBlock)
  k_sort_rays(const __grid_constant__ B2RenderArgs A, const __grid_constant__ SortBox box, uint32_t* __restrict__ hist,
              uint32_t* __restrict__ keys, uint32_t* __restrict__ perm)
{
  const int w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= A.numWarps)
    return;
  const int64_t base = (int64_t)w * A.regionCap;
  const uint32_t n = A.qCount[w];
  for (uint32_t i = lane; i < n; i += 32)
  {
    if (SCATTER)
    { // hist holds the exclusive scan: bucket start offsets, bumped per ray
      const uint32_t key = keys[base + i];
      perm[atomicAdd(&hist[key], 1u)] = (uint32_t)(base + i);
    }
    else
    {
      const uint4 a = __ldcg(A.q.p0 + base + i), b = __ldcg(A.q.p1 + base + i);
      const float o[3] = { __uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z) };
      const float d[3] = { __uint_as_float(a.w), __uint_as_float(b.x), __uint_as_float(b.y) };
      uint32_t key = 0;
#pragma unroll
      for (int c = 0; c < 3; ++c)
      {
        const float f = (o[c] - box.lo[c]) * box.cellsPerUnit[c];
        const int cell = f > 0.f ? (f < (float)((1 << kSortCellBits) - 1) ? (int)f : (1 << kSortCellBits) - 1) : 0;
        key |= spread3((uint32_t)cell) << c;
      }
      key = (key << 3) | (d[0] < 0.f ? 1u : 0u) | (d[1] < 0.f ? 2u : 0u) | (d[2] < 0.f ? 4u : 0u);
      keys[base + i] = key;
      atomicAdd(&hist[key], 1u);
    }
  }
}

// K1+K2 (+ the sorting half of K5): closest hit of every ray of the warp's queue region (PRIMARY: of freshly
// generated camera rays).  Paths that miss or land on an emitter finish here (their radiance is final); every
// other hit is binned by what the shade stage will do with it -- bin 0: specular (dielectric) hit, bins 1..3:
// lambertian hit whose strategy draw selects the cosine / light-quad / sphere generator -- so that k_shade runs
// warp-uniform work with all 32 lanes alive.  The ray AND its hit (t, primitive) are appended to the warp's
// region of the bin as one dense 52-byte record (coalesced 16-byte stores): ballot + popcount prefix on top of
// a register counter, no atomics.
// TAIL = true (deep bounces, few rays left): the input is ONE flat global queue of A.depthTotals[depth-1] rays
// and the four bins are global too; warps take 32-ray tiles grid-stride and append with one warp-aggregated
// atomicAdd per non-empty bin per tile.  Per-warp regions would leave thousands of warps with a handful of rays
// each (DESIGN.md "tail mode").
// ---- BVH scenes: persistent-lane traversal.  A per-ray traversal loop leaves most lanes idle (measured 7.8 of 32
// active on the 1M-sphere scene: trip counts differ by an order of magnitude between the rays of a warp).  Here a
// lane that finishes its ray hands the hit over and takes the NEXT ray of the warp's own region (a warp-uniform
// cursor, no atomics: the region is private to the warp), and the warp leaves the traversal loop to refill as soon
// as fewer than kRefillLanes lanes are still traversing (Aila & Laine's persistent while-while with replacement).
// The node visits, their order and the leaf tests are those of closest_bvh, so hits are bit-identical.
#ifndef B2PT_BVH_REFILL
#define B2PT_BVH_REFILL 24
#endif
constexpr int kRefillLanes = B2PT_BVH_REFILL;
#ifndef B2PT_BVH_INNER_STEPS
#define B2PT_BVH_INNER_STEPS 8
#endif
constexpr int kInnerSteps = B2PT_BVH_INNER_STEPS;
#ifndef B2PT_BVH_LEAF_CHUNK
#define B2PT_BVH_LEAF_CHUNK 1
#endif
constexpr int kLeafChunk = B2PT_BVH_LEAF_CHUNK;

template <bool PRIMARY, bool TAIL>
__device__ __forceinline__ void trace_body_bvh(const B2Camera& cam, const B2BvhScene& S, const B2RenderArgs& A,
                                               int depth, int w, int lane, int64_t nIn, int64_t tailWarps)
{
  const int64_t base = TAIL ? 0 : (int64_t)w * A.regionCap;
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  const unsigned lt = (1u << lane) - 1u;
  // local ray numbers 0..nLocal-1 of this warp and their queue index (tile-interleaved for PRIMARY and TAIL)
  int64_t nLocal = nIn;
  if (TAIL)
  {
    const int64_t tiles = (nIn + 31) >> 5;
    nLocal = tiles > w ? ((tiles - 1 - w) / tailWarps + 1) * 32 : 0;
  }
  const int64_t stride = TAIL ? tailWarps : (int64_t)A.numWarps;
  const int64_t permBase = sorted_chunk(A, depth) * w; // (sorted input: this warp's chunk of the permutation)
  uint32_t cnt0 = 0, cnt1 = 0, cnt2 = 0, cnt3 = 0;
  int64_t next = 0;
  bool has = false, done = false;
  f3 o = mk3(0.f, 0.f, 0.f), d = o, T = o, inv = o, od = o;
  uint32_t pid = 0, rng = 0, cur = 0;
  float closest = FLT_MAX;
  int best = 0, sp = 0;
  bool found = false;
  // (Keeping the entry distance of every postponed child next to its id, so that a child popped after a closer hit was
  // found is dropped without fetching its pair, was measured 9 % SLOWER -- 862 vs 789 ms on configs[3]: twice the
  // local-memory stack traffic and more spills cost more than the skipped fetches save.  -DB2PT_STACK_T builds it.)
  uint32_t stack[64];
#ifdef B2PT_STACK_T
  float stackT[64];
#endif
  const float4* nodes4 = reinterpret_cast<const float4*>(S.nodes);
  for (;;)
  {
    // ---- refill: lanes without a ray take the next local ray numbers
    const unsigned need = __ballot_sync(0xffffffffu, !has);
    if (need)
    {
      const int64_t r = next + __popc(need & lt);
      if (!has && r < nLocal)
      {
        const int64_t idx = PRIMARY ? (primary_tile(r >> 5, w, A.numWarps) << 5) + (r & 31)
                                    : (TAIL ? ((((r >> 5) * stride + w) << 5) + (r & 31))
                                            : (A.perm ? (int64_t)__ldg(A.perm + permBase + r) : base + r));
        if (PRIMARY ? idx < A.nPaths : (TAIL ? idx < nIn : true))
        {
          load_ray<PRIMARY>(cam, A, idx, o, d, T, pid, rng);
          inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
          od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
          closest = FLT_MAX;
          found = false;
          best = 0;
          sp = 0;
#ifdef B2PT_DEBUG_HIST
          atomicAdd(&g_debugHist[51], 1ull); // binary: rays
#endif
          done = S.nNodes <= 0;
          cur = done ? 0u : bvh_pack(__ldg(nodes4).w, __ldg(nodes4 + 1).w);
          has = true;
        }
      }
      next += __popc(need);
    }
    if (!__any_sync(0xffffffffu, has))
      break;
    // ---- traverse until too few lanes are still busy (or, with nothing left to refill, until all are done)
    for (;;)
    {
      // inner nodes: at most kInnerSteps rounds before the lanes waiting at a leaf get their turn
#pragma unroll 1
      for (int it = 0; it < kInnerSteps; ++it)
      {
        const bool inner = has && !done && !(cur >> 24);
        if (!__any_sync(0xffffffffu, inner))
          break;
        if (!inner)
          continue;
#ifdef B2PT_DEBUG_HIST
        atomicAdd(&g_debugHist[48], 1ull); // binary: inner steps (child pairs)
#endif
        // one 64-byte fetch of the child pair, nearer child first (BVHTraverser.h:189-201)
        const float4* lp = nodes4 + 2 * (size_t)(cur & 0xffffffu);
        const float4 l0 = __ldg(lp), l1 = __ldg(lp + 1), r0 = __ldg(lp + 2), r1 = __ldg(lp + 3);
        // (prefetching both children's next fetch to L1 was measured 1.5x SLOWER: the traversal is bound by L2
        // transaction throughput, ~3.4 TB/s of 64-byte node fetches, not by latency alone)
        float tl, tr;
        const bool hl = slab_hit_fma(l0, l1, inv, od, 0.001f, closest, tl);
        const bool hr = slab_hit_fma(r0, r1, inv, od, 0.001f, closest, tr);
        const uint32_t cl = bvh_pack(l0.w, l1.w), crr = bvh_pack(r0.w, r1.w);
        // (a branch-free form of this update -- selects, speculative read of the stack top, unconditional store above
        // it -- keeps the lanes converged but was measured 4.5 % SLOWER: every lane then touches the local-memory
        // stack every step; profiles/r02_bvh_experiments.md)
#if defined(B2PT_STACK_T) || defined(B2PT_BRANCHY_STEP)
        if (hl && hr)
        {
          const bool rightCloser = tl > tr;
          cur = rightCloser ? crr : cl;
          if (sp < 64)
          {
#ifdef B2PT_STACK_T
            stackT[sp] = rightCloser ? tl : tr;
#endif
            stack[sp++] = rightCloser ? cl : crr;
          }
        }
        else if (hl)
          cur = cl;
        else if (hr)
          cur = crr;
        else
        {
#ifdef B2PT_STACK_T
          while (sp > 0 && stackT[sp - 1] > closest)
            --sp; // entered beyond the closest hit found since it was pushed: nothing in it can win
#endif
          if (sp == 0)
            done = true;
          else
            cur = stack[--sp];
        }
#else
        // One pass for the four outcomes: the next node is a select, only the stack accesses sit under predicates (a
        // lane that neither pushes nor pops does not touch local memory).  The four-way branch this replaces ran each
        // outcome serially: 17 % of the kernel's instructions at 4-6 active lanes (profiles/r02_experiments.md).
        const bool both = hl && hr, none = !(hl || hr);
        const bool rightCloser = tl > tr;
        const uint32_t nearChild = (hl && !(hr && rightCloser)) ? cl : crr;
        if (both && sp < 64)
          stack[sp++] = rightCloser ? cl : crr;
        const bool pop = none && sp > 0;
        const uint32_t top = pop ? stack[sp - 1] : 0u;
        sp -= pop ? 1 : 0;
        done = none && !pop;
        cur = none ? top : nearChild;
#endif
      }
      if (has && !done && (cur >> 24))
      { // leaf: primitives in ascending original index
        const uint32_t count = cur >> 24, left = cur & 0xffffffu;
#ifdef B2PT_DEBUG_HIST
        atomicAdd(&g_debugHist[49], 1ull);                        // binary: leaves visited
        atomicAdd(&g_debugHist[50], (unsigned long long)count);   // binary: primitives offered by them
#endif
        for (uint32_t k0 = 0; k0 < count; k0 += kLeafChunk)
        { // the slots and the leaf-ordered sphere geometry of a chunk are fetched together (independent loads)
          int enc[kLeafChunk];
          float4 geo[kLeafChunk];
#pragma unroll
          for (int j = 0; j < kLeafChunk; ++j)
            if (k0 + j < count)
            {
              enc[j] = __ldg(S.primSlots + left + k0 + j);
              geo[j] = __ldg(S.leafSph + left + k0 + j);
            }
#pragma unroll
          for (int j = 0; j < kLeafChunk; ++j)
            if (k0 + j < count)
            {
              float t;
              if (enc[j] >= 0)
              {
                if (quad_accept(S.quads[enc[j]], o, d, 0.001f, closest, t))
                {
                  closest = t;
                  best = enc[j];
                  found = true;
                }
              }
              else if (sphere_may_hit(mk3(geo[j].x, geo[j].y, geo[j].z), geo[j].w, o, d) &&
                       sphere_gate(mk3(geo[j].x, geo[j].y, geo[j].z), geo[j].w, inv, od, 0.001f, FLT_MAX) &&
                       sphere_accept(mk3(geo[j].x, geo[j].y, geo[j].z), geo[j].w, o, d, 0.001f, closest, t))
              {
                closest = t;
                best = enc[j];
                found = true;
              }
            }
        }
#ifdef B2PT_STACK_T
        while (sp > 0 && stackT[sp - 1] > closest)
          --sp;
#endif
        if (sp == 0)
          done = true;
        else
          cur = stack[--sp];
      }
      const unsigned act = __ballot_sync(0xffffffffu, has && !done);
      if (act == 0u || (next < nLocal && __popc(act) < kRefillLanes))
        break;
    }
    // ---- resolve the finished rays: gated quads, then miss / emitter / bin (as in the generic body)
    const bool resolve = has && done;
    int bin = -1;
    int code = B2PT_MISS;
    if (resolve)
    {
      for (int g = 0; g < S.nGate; ++g)
      {
        float tn, t;
        if (!slab_hit(S.gate[g].bmin, S.gate[g].bmax, inv, od, 0.001f, closest, tn))
          continue;
        const int q = S.gate[g].quad;
        if (quad_accept(S.quads[q], o, d, 0.001f, closest, t))
        {
          closest = t;
          best = q;
          found = true;
        }
      }
      code = found ? best : B2PT_MISS;
      if (code == B2PT_MISS)
        finish_path(A, pid, T * 0.f, rng, refStream, A.maxDepth - depth);
      else
      {
        const int kind = hit_kind(S, code);
        if (kind == 1)
        {
          Hit hit;
          fill_hit(S, code, o, d, closest, hit);
          const f3 em = (dot3(hit.n, d) < 0.0f) ? hit.alb : mk3(0.f, 0.f, 0.f);
          finish_path(A, pid, mul3(T, em), rng, refStream, A.maxDepth - depth);
        }
        else
        {
          uint32_t peek = rng;
          bin = (kind == 2) ? 0 : draw_which(peek);
        }
      }
      has = false;
      done = false;
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, bin == 0), b1 = __ballot_sync(0xffffffffu, bin == 1);
    const unsigned b2 = __ballot_sync(0xffffffffu, bin == 2), b3 = __ballot_sync(0xffffffffu, bin == 3);
    if (TAIL)
    {
      uint32_t got = 0;
      if (lane < 4)
      {
        const unsigned bk = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : b3));
        if (bk)
          got = atomicAdd(&A.binTotals[depth * 4 + lane], (uint32_t)__popc(bk));
      }
      cnt0 = __shfl_sync(0xffffffffu, got, 0), cnt1 = __shfl_sync(0xffffffffu, got, 1);
      cnt2 = __shfl_sync(0xffffffffu, got, 2), cnt3 = __shfl_sync(0xffffffffu, got, 3);
    }
    if (bin >= 0)
    {
      const unsigned mine = pick4(bin, b0, b1, b2, b3);
      const uint32_t cnt = pick4(bin, cnt0, cnt1, cnt2, cnt3);
      const int64_t j = (int64_t)bin * A.binStride + base + cnt + __popc(mine & lt);
      A.bins[0].p0[j] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
      A.bins[0].p1[j] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
      A.bins[0].p2[j] = make_uint4(__float_as_uint(T.z), pid, rng, __float_as_uint(closest));
      A.bins[0].code[j] = (uint32_t)code;
    }
    if (!TAIL)
      cnt0 += __popc(b0), cnt1 += __popc(b1), cnt2 += __popc(b2), cnt3 += __popc(b3);
  }
  if (!TAIL && lane == 0)
  {
    A.bins[0].count[0 * A.numWarps + w] = cnt0;
    A.bins[0].count[1 * A.numWarps + w] = cnt1;
    A.bins[0].count[2 * A.numWarps + w] = cnt2;
    A.bins[0].count[3 * A.numWarps + w] = cnt3;
  }
}

// ---- BVH scenes, binary tree, sorted rays: the traversal on its own.  In trace_body_bvh a lane that finishes a ray
// resolves it (gated quads, emitter / miss bookkeeping, strategy draw, a 52-byte bin record behind four ballots) while
// the other lanes of the warp wait: with ~41 inner steps per ray and a few lanes finishing per round that part ran at
// a quarter of the warp and, with the ray's throughput / path id / RNG state alive through the loop, pinned the kernel
// at 64 registers.  k_bvh_hits keeps only what the descent needs (reciprocal direction, o/d products, closest, stack):
// a finished lane stores 8 bytes (t, primitive) at its queue index and takes the next ray of the warp's chunk of the
// sorted order at once; origin and direction are read again from the queue when a leaf needs the exact tests.
// k_resolve_hits then does the per-ray bookkeeping in queue order with full warps and coalesced accesses.  Node visits,
// their order and the leaf tests are those of closest_bvh, so every hit is bit-identical (tests/test_gpu_spheres.py).
// Measured on configs[3]: 795 ms against 792 ms for the single kernel (4 or 5 CTAs per SM alike; refilling at 32 / 28 /
// 20 busy lanes 857 / 831 / 807 ms; reading the ray again at every leaf instead of keeping it 992 ms): a warp's step
// waits for the slowest of its 32 node fetches (27 % of them leave L1), and neither more warps nor cheaper
// bookkeeping shortens that chain.  Opt-in (B2PT_FLAG_SPLIT_TRACE); profiles/r02_experiments.md.
#ifndef B2PT_LEAN_BLOCKS
#define B2PT_LEAN_BLOCKS 5
#endif
#ifndef B2PT_LEAN_REFILL
#define B2PT_LEAN_REFILL 20 // refill as soon as fewer lanes than this are traversing
#endif
#ifndef B2PT_LEAN_INNER_STEPS
#define B2PT_LEAN_INNER_STEPS 8
#endif
// Staged rays of one warp: the next 32 rays of its chunk, fetched by all 32 lanes at once (one coalesced read of the
// permutation, one gathered read of the rays) so that a lane that needs a new ray takes it from shared memory instead
// of waiting, alone, for three dependent global loads while the rest of the warp idles.
struct LeanStage
{
  uint32_t r[32];
  float o[3][32], d[3][32];
};
__global__ void __launch_bounds__(kBlock, B2PT_LEAN_BLOCKS)
  k_bvh_hits(const __grid_constant__ B2BvhScene S, const __grid_constant__ B2RenderArgs A)
{
  __shared__ LeanStage sStage[kWarps];
  const uint32_t w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  LeanStage& st = sStage[threadIdx.x >> 5];
  const unsigned lt = (1u << lane) - 1u;
  const uint32_t total = A.depthTotals[A.depth - 1];
  const uint32_t nW = gridDim.x * kWarps;
  const uint32_t chunk = (((total + nW - 1) / nW) + 31u) & ~31u;
  if ((uint64_t)chunk * w >= total)
    return; // warp-uniform
  uint32_t next = chunk * w; // first ray of the chunk that is not staged yet
  const uint32_t end = (uint32_t)min((uint64_t)total, (uint64_t)next + chunk);
  uint32_t staged = 0, taken = 0; // rays in the stage / handed out
  bool has = false, done = false;
  f3 o = mk3(0.f, 0.f, 0.f), d = o, inv = o, od = o;
  uint32_t r = 0, cur = 0;
  float closest = FLT_MAX;
  int best = B2PT_MISS, sp = 0;
  uint32_t stack[64];
  const float4* nodes4 = reinterpret_cast<const float4*>(S.nodes);
  const uint32_t rootCur = S.nNodes > 0 ? bvh_pack(__ldg(nodes4).w, __ldg(nodes4 + 1).w) : 0u;
  for (;;)
  {
    // ---- refill: lanes without a ray take staged rays in order; an empty stage is refilled by the whole warp
    unsigned need = __ballot_sync(0xffffffffu, !has);
    while (need)
    {
      if (taken == staged)
      {
        if (next >= end)
          break;
        __syncwarp();
        const uint32_t k = next + lane;
        if (k < end)
        {
          const uint32_t q = __ldg(A.perm + k);
          const uint4 a = __ldcg(A.q.p0 + q), b = __ldcg(A.q.p1 + q);
          st.r[lane] = q;
          st.o[0][lane] = __uint_as_float(a.x), st.o[1][lane] = __uint_as_float(a.y), st.o[2][lane] = __uint_as_float(a.z);
          st.d[0][lane] = __uint_as_float(a.w), st.d[1][lane] = __uint_as_float(b.x), st.d[2][lane] = __uint_as_float(b.y);
        }
        staged = min(32u, end - next);
        taken = 0;
        next += staged;
        __syncwarp();
      }
      const uint32_t slot = taken + __popc(need & lt);
      const bool take = !has && slot < staged;
      if (take)
      {
        r = st.r[slot];
        o = mk3(st.o[0][slot], st.o[1][slot], st.o[2][slot]);
        d = mk3(st.d[0][slot], st.d[1][slot], st.d[2][slot]);
        inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
        od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
        closest = FLT_MAX;
        best = B2PT_MISS;
        sp = 0;
        done = S.nNodes <= 0;
        cur = rootCur;
        has = true;
      }
      taken = min(staged, taken + (uint32_t)__popc(need));
      need = __ballot_sync(0xffffffffu, !has);
    }
    if (!__any_sync(0xffffffffu, has))
      break;
    const bool more = taken < staged || next < end;
    for (;;)
    {
#pragma unroll 1
      for (int it = 0; it < B2PT_LEAN_INNER_STEPS; ++it)
      {
        const bool inner = has && !done && !(cur >> 24);
        if (!__any_sync(0xffffffffu, inner))
          break;
        if (!inner)
          continue;
        const float4* lp = nodes4 + 2 * (size_t)(cur & 0xffffffu);
        const float4 l0 = __ldg(lp), l1 = __ldg(lp + 1), r0 = __ldg(lp + 2), r1 = __ldg(lp + 3);
        float tl, tr;
        const bool hl = slab_hit_fma(l0, l1, inv, od, 0.001f, closest, tl);
        const bool hr = slab_hit_fma(r0, r1, inv, od, 0.001f, closest, tr);
        const uint32_t cl = bvh_pack(l0.w, l1.w), crr = bvh_pack(r0.w, r1.w);
        if (hl && hr)
        {
          const bool rightCloser = tl > tr;
          cur = rightCloser ? crr : cl;
          if (sp < 64)
            stack[sp++] = rightCloser ? cl : crr;
        }
        else if (hl)
          cur = cl;
        else if (hr)
          cur = crr;
        else if (sp == 0)
          done = true;
        else
          cur = stack[--sp];
      }
      if (has && !done && (cur >> 24))
      { // leaf: primitives in ascending original index
        const uint32_t count = cur >> 24, left = cur & 0xffffffu;
        for (uint32_t k0 = 0; k0 < count; ++k0)
        {
          const int enc = __ldg(S.primSlots + left + k0);
          const float4 geo = __ldg(S.leafSph + left + k0);
          float t;
          if (enc >= 0)
          {
            if (quad_accept(S.quads[enc], o, d, 0.001f, closest, t))
            {
              closest = t;
              best = enc;
            }
          }
          else if (sphere_may_hit(mk3(geo.x, geo.y, geo.z), geo.w, o, d) &&
                   sphere_gate(mk3(geo.x, geo.y, geo.z), geo.w, inv, od, 0.001f, FLT_MAX) &&
                   sphere_accept(mk3(geo.x, geo.y, geo.z), geo.w, o, d, 0.001f, closest, t))
          {
            closest = t;
            best = enc;
          }
        }
        if (sp == 0)
          done = true;
        else
          cur = stack[--sp];
      }
      if (has && done)
      { // hand the hit over; the lane is free
        A.hits[r] = make_uint2(__float_as_uint(closest), (uint32_t)best);
        has = false;
        done = false;
      }
      const unsigned act = __ballot_sync(0xffffffffu, has);
      if (act == 0u || (more && __popc(act) < B2PT_LEAN_REFILL))
        break;
    }
  }
}

// The bookkeeping half of a split BVH bounce: queue order, one ray per lane, hits read from A.hits.  Same rules as the
// resolve part of trace_body_bvh (gated quads continue from the tree's closest hit; miss / emitter finish the path;
// every other hit is binned by shading strategy).
__global__ void __launch_bounds__(kBlock, kMinBlocksPerSM)
  k_resolve_hits(const __grid_constant__ B2BvhScene S, const __grid_constant__ B2RenderArgs A)
{
  const int w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= A.numWarps)
    return;
  const int depth = A.depth;
  const int64_t base = (int64_t)w * A.regionCap;
  const int64_t nIn = (int64_t)A.qCount[w];
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  const unsigned lt = (1u << lane) - 1u;
  uint32_t cnt0 = 0, cnt1 = 0, cnt2 = 0, cnt3 = 0;
  for (int64_t i0 = 0; i0 < nIn; i0 += 32)
  {
    const int64_t i = i0 + lane;
    int bin = -1;
    f3 o, d, T;
    uint32_t pid = 0, rng = 0;
    float closest = 0.f;
    int code = B2PT_MISS;
    if (i < nIn)
    {
      const int64_t idx = base + i;
      load_ray<false>(B2Camera{}, A, idx, o, d, T, pid, rng);
      const uint2 h = __ldcg(A.hits + idx);
      closest = __uint_as_float(h.x);
      code = (int)h.y;
      if (S.nGate > 0)
      {
        const f3 inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
        const f3 od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
        for (int g = 0; g < S.nGate; ++g)
        {
          float tn, t;
          if (!slab_hit(S.gate[g].bmin, S.gate[g].bmax, inv, od, 0.001f, closest, tn))
            continue;
          const int q = S.gate[g].quad;
          if (quad_accept(S.quads[q], o, d, 0.001f, closest, t))
          {
            closest = t;
            code = q;
          }
        }
      }
      if (code == B2PT_MISS)
        finish_path(A, pid, T * 0.f, rng, refStream, A.maxDepth - depth);
      else
      {
        const int kind = hit_kind(S, code);
        if (kind == 1)
        {
          Hit hit;
          fill_hit(S, code, o, d, closest, hit);
          const f3 em = (dot3(hit.n, d) < 0.0f) ? hit.alb : mk3(0.f, 0.f, 0.f);
          finish_path(A, pid, mul3(T, em), rng, refStream, A.maxDepth - depth);
        }
        else
        {
          uint32_t peek = rng;
          bin = (kind == 2) ? 0 : draw_which(peek);
        }
      }
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, bin == 0), b1 = __ballot_sync(0xffffffffu, bin == 1);
    const unsigned b2 = __ballot_sync(0xffffffffu, bin == 2), b3 = __ballot_sync(0xffffffffu, bin == 3);
    if (bin >= 0)
    {
      const unsigned mine = pick4(bin, b0, b1, b2, b3);
      const uint32_t cnt = pick4(bin, cnt0, cnt1, cnt2, cnt3);
      const int64_t j = (int64_t)bin * A.binStride + base + cnt + __popc(mine & lt);
      A.bins[0].p0[j] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
      A.bins[0].p1[j] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
      A.bins[0].p2[j] = make_uint4(__float_as_uint(T.z), pid, rng, __float_as_uint(closest));
      A.bins[0].code[j] = (uint32_t)code;
    }
    cnt0 += __popc(b0), cnt1 += __popc(b1), cnt2 += __popc(b2), cnt3 += __popc(b3);
  }
  if (lane == 0)
  {
    A.bins[0].count[0 * A.numWarps + w] = cnt0;
    A.bins[0].count[1 * A.numWarps + w] = cnt1;
    A.bins[0].count[2 * A.numWarps + w] = cnt2;
    A.bins[0].count[3 * A.numWarps + w] = cnt3;
  }
}

// ---- BVH scenes, 8-wide compressed tree (B2WideScene; b2pt_wide.h, b2pt_device.cuh "8-wide compressed BVH").
// The same persistent-lane scheme: a lane that finishes its ray takes the next ray of the warp's own region.  Every
// iteration a lane with a node group visits ONE child node (eight quantised boxes in one 80-byte fetch: identical
// straight-line work for every lane, whether the children are subtrees or primitives), then the lanes whose node had
// primitive children that passed their box run ONE exact primitive test.  The ray's throughput, path id and RNG state
// are not carried through the traversal: the finished lane reads them back from its queue entry (primary rays keep the
// RNG state, the rest is implied).
#ifndef B2PT_WIDE_REFILL
#define B2PT_WIDE_REFILL 22
#endif
constexpr int kWideRefillLanes = B2PT_WIDE_REFILL;

template <bool PRIMARY, bool TAIL>
__device__ __forceinline__ void trace_body_wide(const B2Camera& cam, const B2BvhScene& S, const B2RenderArgs& A, int depth,
                                                int w, int lane, int64_t nIn, int64_t tailWarps)
{
  const int64_t base = TAIL ? 0 : (int64_t)w * A.regionCap;
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  const unsigned lt = (1u << lane) - 1u;
  int64_t nLocal = nIn;
  if (TAIL)
  {
    const int64_t tiles = (nIn + 31) >> 5;
    nLocal = tiles > w ? ((tiles - 1 - w) / tailWarps + 1) * 32 : 0;
  }
  const int64_t stride = TAIL ? tailWarps : (int64_t)A.numWarps;
  const int64_t permBase = sorted_chunk(A, depth) * w; // (sorted input: this warp's chunk of the permutation)
  auto ray_index = [&](int64_t r) -> int64_t {
    return PRIMARY ? (primary_tile(r >> 5, w, A.numWarps) << 5) + (r & 31)
                   : (TAIL ? ((((r >> 5) * stride + w) << 5) + (r & 31))
                           : (A.perm ? (int64_t)__ldg(A.perm + permBase + r) : base + r));
  };
  uint32_t cnt0 = 0, cnt1 = 0, cnt2 = 0, cnt3 = 0;
  int64_t next = 0;
  bool has = false, live = false;
  f3 o = mk3(0.f, 0.f, 0.f), d = o, inv = o, od = o;
  uint32_t rngP = 0, oct = 0, myRay = 0;
  float closest = FLT_MAX;
  int best = 0, bestId = 0x7fffffff;
  WideTrav R;
  R.nx = R.ny = R.px = R.py = 0u;
  R.sp = 0;
  uint32_t stackX[kWideStack], stackY[kWideStack];
  for (;;)
  {
    // ---- refill: lanes without a ray take the next local ray numbers
    const unsigned need = __ballot_sync(0xffffffffu, !has);
    if (need)
    {
      const int64_t r = next + __popc(need & lt);
      if (!has && r < nLocal)
      {
        const int64_t idx = ray_index(r);
        if (PRIMARY ? idx < A.nPaths : (TAIL ? idx < nIn : true))
        {
          f3 T;
          uint32_t pid;
          load_ray<PRIMARY>(cam, A, idx, o, d, T, pid, rngP);
          inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
          od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
          oct = wide_octant(inv);
          closest = FLT_MAX;
          best = 0;
          bestId = 0x7fffffff;
          myRay = (uint32_t)r;
#ifdef B2PT_DEBUG_HIST
          atomicAdd(&g_debugHist[42], 1ull); // wide: rays
#endif
          wide_start(R, oct, S.nWide > 0);
          has = true;
          live = wide_next(R, stackX, stackY);
        }
      }
      next += __popc(need);
    }
    if (!__any_sync(0xffffffffu, has))
      break;
    // ---- traverse until too few lanes are still busy (or, with nothing left to refill, until all are done)
    for (;;)
    {
      const bool doA = live && !(R.py & 0xffu);
      if (__any_sync(0xffffffffu, doA))
      {
        if (doA)
        {
          wide_step_node(S, R, stackX, stackY, inv, od, oct, 0.001f, closest);
#ifdef B2PT_DEBUG_HIST
          atomicAdd(&g_debugHist[40], 1ull); // wide: node visits
          atomicAdd(&g_debugHist[43], (unsigned long long)__popc(R.ny & 0xffu)); // inner children hit
          atomicAdd(&g_debugHist[44], (unsigned long long)__popc(R.py & 0xffu)); // primitive children hit (boxes)
#endif
        }
      }
      const bool doB = live && (R.py & 0xffu);
      if (__any_sync(0xffffffffu, doB))
      {
        if (doB)
        {
          wide_step_prim(S, R, o, d, inv, od, oct, 0.001f, FLT_MAX, closest, best, bestId);
#ifdef B2PT_DEBUG_HIST
          atomicAdd(&g_debugHist[41], 1ull); // wide: exact primitive tests
#endif
        }
      }
      if (live)
        live = wide_next(R, stackX, stackY);
      const unsigned act = __ballot_sync(0xffffffffu, live);
      if (act == 0u || (next < nLocal && __popc(act) < kWideRefillLanes))
        break;
    }
    // ---- resolve the finished rays: gated quads, then miss / emitter / bin (as in the generic body)
    const bool resolve = has && !live;
    int bin = -1;
    int code = B2PT_MISS;
    f3 T = mk3(1.f, 1.f, 1.f);
    uint32_t pid = 0, rng = rngP;
    if (resolve)
    {
      const int64_t idx = ray_index((int64_t)myRay);
      if (PRIMARY)
        pid = (uint32_t)idx;
      else
      {
        const uint4 b = __ldcg(A.q.p1 + idx), c = __ldcg(A.q.p2 + idx);
        T = mk3(__uint_as_float(b.z), __uint_as_float(b.w), __uint_as_float(c.x));
        pid = c.y;
        rng = c.z;
      }
      bool found = bestId != 0x7fffffff;
      for (int g = 0; g < S.nGate; ++g)
      {
        float tn, t;
        if (!slab_hit(S.gate[g].bmin, S.gate[g].bmax, inv, od, 0.001f, closest, tn))
          continue;
        const int q = S.gate[g].quad;
        if (quad_accept(S.quads[q], o, d, 0.001f, closest, t))
        {
          closest = t;
          best = q;
          found = true;
        }
      }
      code = found ? best : B2PT_MISS;
      if (code == B2PT_MISS)
        finish_path(A, pid, T * 0.f, rng, refStream, A.maxDepth - depth);
      else
      {
        const int kind = hit_kind(S, code);
        if (kind == 1)
        {
          Hit hit;
          fill_hit(S, code, o, d, closest, hit);
          const f3 em = (dot3(hit.n, d) < 0.0f) ? hit.alb : mk3(0.f, 0.f, 0.f);
          finish_path(A, pid, mul3(T, em), rng, refStream, A.maxDepth - depth);
        }
        else
        {
          uint32_t peek = rng;
          bin = (kind == 2) ? 0 : draw_which(peek);
        }
      }
      has = false;
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, bin == 0), b1 = __ballot_sync(0xffffffffu, bin == 1);
    const unsigned b2 = __ballot_sync(0xffffffffu, bin == 2), b3 = __ballot_sync(0xffffffffu, bin == 3);
    if (TAIL)
    {
      uint32_t got = 0;
      if (lane < 4)
      {
        const unsigned bk = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : b3));
        if (bk)
          got = atomicAdd(&A.binTotals[depth * 4 + lane], (uint32_t)__popc(bk));
      }
      cnt0 = __shfl_sync(0xffffffffu, got, 0), cnt1 = __shfl_sync(0xffffffffu, got, 1);
      cnt2 = __shfl_sync(0xffffffffu, got, 2), cnt3 = __shfl_sync(0xffffffffu, got, 3);
    }
    if (bin >= 0)
    {
      const unsigned mine = pick4(bin, b0, b1, b2, b3);
      const uint32_t cnt = pick4(bin, cnt0, cnt1, cnt2, cnt3);
      const int64_t j = (int64_t)bin * A.binStride + base + cnt + __popc(mine & lt);
      A.bins[0].p0[j] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
      A.bins[0].p1[j] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
      A.bins[0].p2[j] = make_uint4(__float_as_uint(T.z), pid, rng, __float_as_uint(closest));
      A.bins[0].code[j] = (uint32_t)code;
    }
    if (!TAIL)
      cnt0 += __popc(b0), cnt1 += __popc(b1), cnt2 += __popc(b2), cnt3 += __popc(b3);
  }
  if (!TAIL && lane == 0)
  {
    A.bins[0].count[0 * A.numWarps + w] = cnt0;
    A.bins[0].count[1 * A.numWarps + w] = cnt1;
    A.bins[0].count[2 * A.numWarps + w] = cnt2;
    A.bins[0].count[3 * A.numWarps + w] = cnt3;
  }
}

// Work of one warp in k_trace: rays [.., nIn) of its region (TAIL: tiles w, w+tailWarps, ... of the flat queue).
template <bool PRIMARY, class SceneT, bool TAIL>
__device__ __forceinline__ void trace_body(const B2Camera& cam, const SceneT& S, const B2RenderArgs& A, int depth,
                                           int w, int lane, int64_t nIn, int64_t tailWarps)
{
  if constexpr (std::is_same<SceneT, B2WideScene>::value)
  {
    trace_body_wide<PRIMARY, TAIL>(cam, S, A, depth, w, lane, nIn, tailWarps);
    return;
  }
  if constexpr (std::is_same<SceneT, B2BvhScene>::value)
  {
    trace_body_bvh<PRIMARY, TAIL>(cam, S, A, depth, w, lane, nIn, tailWarps);
    return;
  }
  const int64_t base = TAIL ? 0 : (int64_t)w * A.regionCap;
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  uint32_t cnt0 = 0, cnt1 = 0, cnt2 = 0, cnt3 = 0;
  int slot = w; // PRIMARY: this warp's tile slot within the current round (primary_tile)
  for (int64_t i0 = TAIL ? (int64_t)w * 32 : 0; i0 < nIn; i0 += TAIL ? tailWarps * 32 : 32)
  {
    const int64_t i = i0 + lane;
    int bin = -1;
    f3 o, d, T;
    uint32_t pid = 0, rng = 0;
    float t = 0.f;
    int code = B2PT_MISS;
    const int64_t idx = PRIMARY ? ((int64_t)((uint32_t)(i0 >> 5) * (uint32_t)A.numWarps + (uint32_t)slot) << 5) + lane : base + i;
    if (PRIMARY)
      slot = slot + 1 == A.numWarps ? 0 : slot + 1;
    if (!PRIMARY && !TAIL && i + kPrefetchAhead < nIn)
    {
      prefetch_l2(A.q.p0 + idx + kPrefetchAhead);
      prefetch_l2(A.q.p1 + idx + kPrefetchAhead);
      prefetch_l2(A.q.p2 + idx + kPrefetchAhead);
    }
    if (PRIMARY ? idx < A.nPaths : i < nIn)
    {
      uint32_t slotB = 0; // PRIMARY: sample slot of the path; the same for the 32 paths of a tile (nPixels % 32 == 0)
      load_ray<PRIMARY>(cam, A, idx, o, d, T, pid, rng, &slotB);
      bool masked = false;
      if constexpr (PRIMARY && std::is_same<SceneT, B2SmallScene>::value)
        masked = A.primMask != nullptr;
      if constexpr (PRIMARY && std::is_same<SceneT, B2SmallScene>::value)
        if (masked)
      { // the tile's candidate mask and the view's per-quad constants (warp-uniform; nPixels % 32 == 0)
        const uint32_t tileBase = (uint32_t)idx - (uint32_t)lane;
        const uint32_t view = A.views ? fastdiv(slotB, A.divSppMagic, A.divSppShift) : 0u;
        const uint32_t tileInView = (tileBase - slotB * (uint32_t)A.nPixels) >> 5;
        const uint2 mask = __ldg(A.primMask + (size_t)view * A.tilesPerView + tileInView);
#ifdef B2PT_DEBUG_HIST
        if (lane == 0)
        { // [40..]: tiles, filter candidates, gate/sphere bits, tiles with any gate bit
          atomicAdd(&g_debugHist[40], 1ull);
          atomicAdd(&g_debugHist[41], (unsigned long long)__popc(mask.x));
          atomicAdd(&g_debugHist[42], (unsigned long long)__popc(mask.y));
          atomicAdd(&g_debugHist[43], mask.y ? 1ull : 0ull);
          atomicAdd(&g_debugHist[44 + min(__popc(mask.x), 3)], 1ull); // tiles with 0 / 1 / 2 / >= 3 candidates
        }
#endif
        code = closest_small_masked(S, A.primQuads + (size_t)view * B2PT_SMALL_MAX_QUADS, mask, o, d, 0.001f, FLT_MAX, t);
      }
      if (!masked)
        code = closest_hit(S, o, d, 0.001f, FLT_MAX, t);
      if (code == B2PT_MISS)
        finish_path(A, pid, T * 0.f, rng, refStream, A.maxDepth - depth); // a[d]=1, e[d]=0
      else
      {
        const int kind = hit_kind(S, code);
        if (kind == 1)
        { // DiffuseLightWorklet::emit: front face only, but the normal was already flipped -> two-sided
          Hit hit;
          fill_hit(S, code, o, d, t, hit);
          const f3 em = (dot3(hit.n, d) < 0.0f) ? hit.alb : mk3(0.f, 0.f, 0.f);
          finish_path(A, pid, mul3(T, em), rng, refStream, A.maxDepth - depth);
        }
        else
        {
          uint32_t peek = rng;
          bin = (kind == 2) ? 0 : draw_which(peek);
        }
      }
    }
    // destination of this lane's record: rank among the lanes of its bin on top of the bin's counter (a
    // register per warp region; tail mode: one atomicAdd per non-empty bin per tile); the four ballots are
    // warp-uniform work, the stores happen once (no per-bin divergent blocks)
    const unsigned lt = (1u << lane) - 1u;
    const unsigned b0 = __ballot_sync(0xffffffffu, bin == 0), b1 = __ballot_sync(0xffffffffu, bin == 1);
    const unsigned b2 = __ballot_sync(0xffffffffu, bin == 2), b3 = __ballot_sync(0xffffffffu, bin == 3);
    if (TAIL)
    {
      uint32_t got = 0;
      if (lane < 4)
      {
        const unsigned bk = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : b3));
        if (bk)
          got = atomicAdd(&A.binTotals[depth * 4 + lane], (uint32_t)__popc(bk));
      }
      cnt0 = __shfl_sync(0xffffffffu, got, 0), cnt1 = __shfl_sync(0xffffffffu, got, 1);
      cnt2 = __shfl_sync(0xffffffffu, got, 2), cnt3 = __shfl_sync(0xffffffffu, got, 3);
    }
    if (bin >= 0)
    {
      const unsigned mine = pick4(bin, b0, b1, b2, b3);
      const uint32_t cnt = pick4(bin, cnt0, cnt1, cnt2, cnt3);
      const int64_t j = (int64_t)bin * A.binStride + base + cnt + __popc(mine & lt);
      A.bins[0].p0[j] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
      A.bins[0].p1[j] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
      A.bins[0].p2[j] = make_uint4(__float_as_uint(T.z), pid, rng, __float_as_uint(t));
      A.bins[0].code[j] = (uint32_t)code;
    }
    if (!TAIL)
      cnt0 += __popc(b0), cnt1 += __popc(b1), cnt2 += __popc(b2), cnt3 += __popc(b3);
  }
  if (!TAIL && lane == 0)
  {
    A.bins[0].count[0 * A.numWarps + w] = cnt0;
    A.bins[0].count[1 * A.numWarps + w] = cnt1;
    A.bins[0].count[2 * A.numWarps + w] = cnt2;
    A.bins[0].count[3 * A.numWarps + w] = cnt3;
  }
}

template <bool PRIMARY, class SceneT, bool TAIL>
__global__ void __launch_bounds__(kBlock, kTraceMinBlocksPerSM)
  k_trace(const __grid_constant__ B2Camera cam, const __grid_constant__ SceneT scene,
          const __grid_constant__ B2RenderArgs A)
{
  static_assert(!(PRIMARY && TAIL), "primary rays are never traced in tail mode");
  const int w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  // PRIMARY: the batch's 32-path tiles are dealt round by round to the warps, skewed by one slot per round
  // (primary_tile), so every region samples the whole image and the regions shrink at the same rate; contiguous
  // pixel ranges would leave the regions that cover the image border (rays that miss) empty, and so would a plain
  // round-robin whenever numWarps and the tiles per image row share a factor (4736 warps, 32 tiles per 1024-pixel row:
  // warp w would only ever see column strip w % 32).
  const int64_t tilesTotal = (A.nPaths + 31) >> 5;
  const int64_t tailWarps = (int64_t)gridDim.x * kWarps;
  int64_t nIn;
  if (TAIL)
  {
    const int64_t nAll = (int64_t)A.depthTotals[A.depth - 1];
    // rays of this warp: tiles w, w + tailWarps, ... of the flat queue (the last tile may be partial)
    nIn = nAll;
    if ((int64_t)blockIdx.x * kWarps * 32 >= nAll)
      return; // no tile for any warp of this CTA
  }
  else if (PRIMARY)
    nIn = w < A.numWarps ? ((tilesTotal + A.numWarps - 1) / A.numWarps) * 32 : 0; // rounds; the last may be partial
  else if (A.perm)
  { // sorted input: chunk w of the permutation (the last chunks may be short or empty)
    const int64_t total = (int64_t)A.depthTotals[A.depth - 1], chunk = sorted_chunk(A, A.depth);
    nIn = w < A.numWarps ? max((int64_t)0, min(chunk, total - chunk * w)) : 0;
  }
  else
    nIn = w < A.numWarps ? (int64_t)A.qCount[w] : 0;
  // CTAs whose eight regions are all empty (deep bounces) leave before staging the scene.
  if (!TAIL && !__syncthreads_or(nIn > 0))
  {
    if (w < A.numWarps && lane == 0)
      for (int k = 0; k < 4; ++k)
        A.bins[0].count[k * A.numWarps + w] = 0;
    return;
  }
  __shared__ StageArea<SceneT> sStage;
  const SceneT& S = stage_scene(scene, sStage);
  __syncthreads();
  if (!TAIL && w >= A.numWarps)
    return;
  trace_body<PRIMARY, SceneT, TAIL>(cam, S, A, A.depth, w, lane, nIn, tailWarps);
}

// K3+K5: material response, direction generator, light pdfs, mixture pdf and the next ray for every binned hit
// of the warp's regions; survivors are compacted into the warp's region of the ray queue.  A warp works on 32
// consecutive records of ONE bin, so the strategy branch is warp-uniform.
// TAIL_IN: the bins are global (binTotals[depth*4+k] records, tiles taken grid-stride).  GLOBAL_OUT: survivors are
// appended to ONE flat global queue (warp-aggregated atomicAdd on A.depthTotals[depth]) instead of the warp's region;
// used by the last regular bounce before the tail and by every tail bounce.
// Work of one warp in k_shade: the four bins of its region (TAIL_IN: tiles of the global bins, dealt so that the
// bins of a nearly empty queue land on different warps).
template <class SceneT, bool TAIL_IN, bool GLOBAL_OUT>
__device__ __forceinline__ void shade_body(const SceneT& S, const B2Lights& LT, const B2RenderArgs& A, int depth, int w,
                                           int lane, int64_t tailWarps)
{
  const int64_t base = TAIL_IN ? 0 : (int64_t)w * A.regionCap;
  const bool lastDepth = (depth == A.maxDepth - 1);
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  uint32_t qcnt = 0;
  for (int k = 0; k < 4; ++k)
  {
    const int64_t nk =
      TAIL_IN ? (int64_t)__ldcg(&A.binTotals[depth * 4 + k]) : (int64_t)A.bins[0].count[k * A.numWarps + w];
    const int64_t binBase = (int64_t)k * A.binStride + base;
    // TAIL_IN: tile t of bin k goes to warp (t + k*tailWarps/4) mod tailWarps
    const int64_t wk = TAIL_IN ? (w + tailWarps - (k * tailWarps) / 4) % tailWarps : 0;
    for (int64_t i0 = TAIL_IN ? wk * 32 : 0; i0 < nk; i0 += TAIL_IN ? tailWarps * 32 : 32)
    {
      const int64_t i = i0 + lane;
      bool survive = false;
      f3 o, d, T;
      uint32_t pid = 0, rng = 0;
      if (!TAIL_IN && i + kPrefetchAhead < nk)
      {
        prefetch_l2(A.bins[0].p0 + binBase + i + kPrefetchAhead);
        prefetch_l2(A.bins[0].p1 + binBase + i + kPrefetchAhead);
        prefetch_l2(A.bins[0].p2 + binBase + i + kPrefetchAhead);
        prefetch_l2(A.bins[0].code + binBase + i + kPrefetchAhead);
      }
      if (i < nk)
      {
        const int64_t j = binBase + i;
        const uint4 a = __ldcg(A.bins[0].p0 + j), b = __ldcg(A.bins[0].p1 + j), c = __ldcg(A.bins[0].p2 + j);
        o = mk3(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
        d = mk3(__uint_as_float(a.w), __uint_as_float(b.x), __uint_as_float(b.y));
        T = mk3(__uint_as_float(b.z), __uint_as_float(b.w), __uint_as_float(c.x));
        pid = c.y;
        rng = c.z;
        Hit hit;
        fill_hit(S, (int)__ldcg(A.bins[0].code + j), o, d, __uint_as_float(c.w), hit);
        f3 L;
        BounceResult r = (k == 0) ? shade_specular(LT, hit, o, d, rng) : shade_lambert(LT, hit, o, d, T, rng, A.flags, L);
        if (r == BOUNCE_CONTINUE && lastDepth)
        { // still alive after maxDepth bounces: e[D-1] = 0 (MapperPathTracer.cxx:328-331); no draws left to burn
          finish_path(A, pid, T * 0.f, rng, refStream, 0);
        }
        else if (r == BOUNCE_DONE) // zero-throughput kill (never in reference-stream mode)
          finish_path(A, pid, L, rng, false, 0);
        else
          survive = true;
      }
      // ---- K5: compaction of survivors: ballot + popcount prefix on top of the warp region's register counter
      // (GLOBAL_OUT: on top of one atomicAdd per tile on the global queue's counter)
      const unsigned ballot = __ballot_sync(0xffffffffu, survive);
      if (GLOBAL_OUT)
      {
        uint32_t got = 0;
        if (lane == 0 && ballot)
          got = atomicAdd(&A.depthTotals[depth], (uint32_t)__popc(ballot));
        qcnt = __shfl_sync(0xffffffffu, got, 0);
      }
      if (survive)
        store_ray(A.q, (GLOBAL_OUT ? 0 : base) + qcnt + __popc(ballot & ((1u << lane) - 1u)), o, d, T, pid, rng);
      if (!GLOBAL_OUT)
        qcnt += __popc(ballot);
    }
  }
  if (!GLOBAL_OUT && lane == 0)
  {
    A.qCount[w] = qcnt;
    if (qcnt)
      atomicAdd(&A.depthTotals[depth], qcnt); // statistics only: one add per warp per launch
  }
}

template <class SceneT, bool TAIL_IN, bool GLOBAL_OUT>
__global__ void __launch_bounds__(kBlock, kMinBlocksPerSM)
  k_shade(const __grid_constant__ SceneT scene, const __grid_constant__ B2Lights lights,
          const __grid_constant__ B2RenderArgs A)
{
  static_assert(GLOBAL_OUT || !TAIL_IN, "tail bounces always write the global queue");
  const int w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int64_t tailWarps = (int64_t)gridDim.x * kWarps;
  if (TAIL_IN)
  {
    // (no early exit: the bins' tiles are dealt to warps all over the grid; the grid is small)
  }
  else
  {
    uint32_t nAny = 0;
    if (w < A.numWarps)
      nAny =
        A.bins[0].count[w] | A.bins[0].count[A.numWarps + w] | A.bins[0].count[2 * A.numWarps + w] | A.bins[0].count[3 * A.numWarps + w];
    if (!__syncthreads_or(nAny != 0))
    { // nothing binned for any warp of this CTA: its queue regions become empty, no staging needed
      if (!GLOBAL_OUT && w < A.numWarps && lane == 0)
        A.qCount[w] = 0;
      return;
    }
  }
  __shared__ StageArea<SceneT> sStage;
  const SceneT& S = stage_scene(scene, sStage);
  const B2Lights& LT = stage_lights(lights, sStage);
  __syncthreads();
  if (!TAIL_IN && w >= A.numWarps)
    return;
  shade_body<SceneT, TAIL_IN, GLOBAL_OUT>(S, LT, A, A.depth, w, lane, tailWarps);
}

// ------------------------------------------------------------------------------------------------------------------
// Small scenes: ONE kernel per bounce.  k_bounce at depth d shades the hits the trace of bounce d-1 binned (bin set
// (d-1)&1: K3, warp-uniform per bin), traces the scattered ray at once (K2, the ray never leaves the registers) and
// bins the new hit into set d&1 (the sorting half of K5).  Nothing dies in the shade stage (every binned hit scatters),
// so there is no compaction and no ray queue between the stages: a survivor costs one 52-byte record read and one
// written per bounce where the two-kernel pipeline moved four (bin + queue, 200 B).  d == maxDepth is the closing
// launch: the hits of the last bounce are shaded (their attenuation can still poison the sum, their draws still
// advance a reference-stream state) and finish with e[D-1] = 0.
// IN_GLOBAL / OUT_GLOBAL: the tail of the bounce loop keeps its records in flat global bins (counters in binTotals,
// one warp-aggregated atomicAdd per bin and tile), see k_trace.
template <class SceneT, bool IN_GLOBAL, bool OUT_GLOBAL>
__device__ __forceinline__ void bounce_body(const SceneT& S, const B2Lights& LT, const B2RenderArgs& A, int depth, int w,
                                            int lane, int64_t tailWarps)
{
  const B2Bins& Bi = A.bins[(depth - 1) & 1];
  const B2Bins& Bo = A.bins[depth & 1];
  const int64_t baseIn = IN_GLOBAL ? 0 : (int64_t)w * A.regionCap;
  const int64_t baseOut = OUT_GLOBAL ? 0 : (int64_t)w * A.regionCap;
  const bool closing = depth >= A.maxDepth;
  const bool refStream = (A.flags & B2PT_FLAG_REFERENCE_STREAM_DEV) != 0;
  const unsigned lt = (1u << lane) - 1u;
  uint32_t cnt0 = 0, cnt1 = 0, cnt2 = 0, cnt3 = 0;
  uint32_t processed = 0;
  for (int k = 0; k < 4; ++k)
  {
    const int64_t nk =
      IN_GLOBAL ? (int64_t)__ldcg(&A.binTotals[(depth - 1) * 4 + k]) : (int64_t)Bi.count[k * A.numWarps + w];
    const int64_t binBase = (int64_t)k * A.binStride + baseIn;
    // IN_GLOBAL: tile t of bin k goes to warp (t + k*tailWarps/4) mod tailWarps (the bins of a nearly empty tail land
    // on different warps)
    const int64_t wk = IN_GLOBAL ? (w + tailWarps - (k * tailWarps) / 4) % tailWarps : 0;
    for (int64_t i0 = IN_GLOBAL ? wk * 32 : 0; i0 < nk; i0 += IN_GLOBAL ? tailWarps * 32 : 32)
    {
      const int64_t i = i0 + lane;
      int bin = -1;
      f3 o, d, T;
      uint32_t pid = 0, rng = 0;
      float t = 0.f;
      int code = B2PT_MISS;
      bool traced = false; // this lane's path entered bounce `depth` (statistics)
      if (!IN_GLOBAL && i + 32 < nk)
      {
        prefetch_l2(Bi.p0 + binBase + i + 32);
        prefetch_l2(Bi.p1 + binBase + i + 32);
        prefetch_l2(Bi.p2 + binBase + i + 32);
        prefetch_l2(Bi.code + binBase + i + 32);
      }
      if (i < nk)
      {
        const int64_t j = binBase + i;
        const uint4 a = __ldcg(Bi.p0 + j), b = __ldcg(Bi.p1 + j), c = __ldcg(Bi.p2 + j);
        o = mk3(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
        d = mk3(__uint_as_float(a.w), __uint_as_float(b.x), __uint_as_float(b.y));
        T = mk3(__uint_as_float(b.z), __uint_as_float(b.w), __uint_as_float(c.x));
        pid = c.y;
        rng = c.z;
        Hit hit;
        fill_hit(S, (int)__ldcg(Bi.code + j), o, d, __uint_as_float(c.w), hit);
        f3 L;
        const BounceResult r =
          (k == 0) ? shade_specular(LT, hit, o, d, rng) : shade_lambert(LT, hit, o, d, T, rng, A.flags, L);
        if (r == BOUNCE_DONE) // zero-throughput kill (never in reference-stream mode)
          finish_path(A, pid, L, rng, false, 0);
        else if (closing) // still alive after maxDepth bounces: e[D-1] = 0 (MapperPathTracer.cxx:328-331)
          finish_path(A, pid, T * 0.f, rng, refStream, 0);
        else
        {
          traced = true;
          code = closest_hit(S, o, d, 0.001f, FLT_MAX, t);
          if (code == B2PT_MISS)
            finish_path(A, pid, T * 0.f, rng, refStream, A.maxDepth - depth); // a[d]=1, e[d]=0
          else
          {
            const int kind = hit_kind(S, code);
            if (kind == 1)
            { // DiffuseLightWorklet::emit: front face only, but the normal was already flipped -> two-sided
              Hit h2;
              fill_hit(S, code, o, d, t, h2);
              const f3 em = (dot3(h2.n, d) < 0.0f) ? h2.alb : mk3(0.f, 0.f, 0.f);
              finish_path(A, pid, mul3(T, em), rng, refStream, A.maxDepth - depth);
            }
            else
            {
              uint32_t peek = rng;
              bin = (kind == 2) ? 0 : draw_which(peek);
            }
          }
        }
      }
      if (closing)
        continue; // (warp-uniform) nothing is binned by the closing launch
      processed += (uint32_t)__popc(__ballot_sync(0xffffffffu, traced));
      const unsigned b0 = __ballot_sync(0xffffffffu, bin == 0), b1 = __ballot_sync(0xffffffffu, bin == 1);
      const unsigned b2 = __ballot_sync(0xffffffffu, bin == 2), b3 = __ballot_sync(0xffffffffu, bin == 3);
      if (OUT_GLOBAL)
      {
        uint32_t got = 0;
        if (lane < 4)
        {
          const unsigned bk = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : b3));
          if (bk)
            got = atomicAdd(&A.binTotals[depth * 4 + lane], (uint32_t)__popc(bk));
        }
        cnt0 = __shfl_sync(0xffffffffu, got, 0), cnt1 = __shfl_sync(0xffffffffu, got, 1);
        cnt2 = __shfl_sync(0xffffffffu, got, 2), cnt3 = __shfl_sync(0xffffffffu, got, 3);
      }
      if (bin >= 0)
      {
        const unsigned mine = bin == 0 ? b0 : (bin == 1 ? b1 : (bin == 2 ? b2 : b3));
        const uint32_t cnt = bin == 0 ? cnt0 : (bin == 1 ? cnt1 : (bin == 2 ? cnt2 : cnt3));
        const int64_t j = (int64_t)bin * A.binStride + baseOut + cnt + __popc(mine & lt);
        Bo.p0[j] = make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(d.x));
        Bo.p1[j] = make_uint4(__float_as_uint(d.y), __float_as_uint(d.z), __float_as_uint(T.x), __float_as_uint(T.y));
        Bo.p2[j] = make_uint4(__float_as_uint(T.z), pid, rng, __float_as_uint(t));
        Bo.code[j] = (uint32_t)code;
      }
      if (!OUT_GLOBAL)
        cnt0 += __popc(b0), cnt1 += __popc(b1), cnt2 += __popc(b2), cnt3 += __popc(b3);
    }
  }
  if (lane == 0)
  {
    if (!OUT_GLOBAL && !closing)
    {
      Bo.count[0 * A.numWarps + w] = cnt0;
      Bo.count[1 * A.numWarps + w] = cnt1;
      Bo.count[2 * A.numWarps + w] = cnt2;
      Bo.count[3 * A.numWarps + w] = cnt3;
    }
    // statistics: rays entering bounce `depth` (b2pt_get_stats: segments; the host's tail-mode decision)
    if (processed && !closing)
      atomicAdd(&A.depthTotals[depth - 1], processed);
  }
}

template <class SceneT, bool IN_GLOBAL, bool OUT_GLOBAL>
__global__ void __launch_bounds__(kBlock, kTraceMinBlocksPerSM)
  k_bounce(const __grid_constant__ SceneT scene, const __grid_constant__ B2Lights lights,
           const __grid_constant__ B2RenderArgs A)
{
  static_assert(OUT_GLOBAL || !IN_GLOBAL, "tail bounces keep their records in the global bins");
  const int w = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int64_t tailWarps = (int64_t)gridDim.x * kWarps;
  if (!IN_GLOBAL)
  {
    const B2Bins& Bi = A.bins[(A.depth - 1) & 1];
    uint32_t nAny = 0;
    if (w < A.numWarps)
      nAny = Bi.count[w] | Bi.count[A.numWarps + w] | Bi.count[2 * A.numWarps + w] | Bi.count[3 * A.numWarps + w];
    if (!__syncthreads_or(nAny != 0))
    { // nothing binned for any warp of this CTA: its regions stay empty, no staging needed
      if (!OUT_GLOBAL && w < A.numWarps && lane == 0)
        for (int k = 0; k < 4; ++k)
          A.bins[A.depth & 1].count[k * A.numWarps + w] = 0;
      return;
    }
  }
  __shared__ StageArea<SceneT> sStage;
  const SceneT& S = stage_scene(scene, sStage);
  const B2Lights& LT = stage_lights(lights, sStage);
  __syncthreads();
  if (!IN_GLOBAL && w >= A.numWarps)
    return;
  bounce_body<SceneT, IN_GLOBAL, OUT_GLOBAL>(S, LT, A, A.depth, w, lane, tailWarps);
}

// The deep tail of the one-kernel pipeline in ONE launch (see k_tail_loop): every remaining bounce and the closing
// shade pass inside a single thread-block cluster, one hardware barrier per bounce.
template <class SceneT>
__global__ void __cluster_dims__(kTailCluster, 1, 1) __launch_bounds__(kTailBlock, 1)
  k_bounce_tail_loop(const __grid_constant__ SceneT scene, const __grid_constant__ B2Lights lights,
                     const __grid_constant__ B2RenderArgs A)
{
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int w = blockIdx.x * (kTailBlock / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int64_t tailWarps = (int64_t)gridDim.x * (kTailBlock / 32);
  __shared__ StageArea<SceneT> sStage;
  const SceneT& S = stage_scene(scene, sStage);
  const B2Lights& LT = stage_lights(lights, sStage);
  __syncthreads();
  for (int depth = A.depth; depth <= A.maxDepth; ++depth)
  {
    const uint32_t* tot = A.binTotals + (depth - 1) * 4;
    const uint32_t nIn = __ldcg(tot) | __ldcg(tot + 1) | __ldcg(tot + 2) | __ldcg(tot + 3);
    if (nIn == 0)
      break; // uniform over the cluster: nobody writes these counters any more
    bounce_body<SceneT, true, true>(S, LT, A, depth, w, lane, tailWarps);
    __threadfence();
    cluster.sync();
  }
}

// The deep tail in ONE launch: a single thread-block cluster (kTailCluster CTAs = SMs) runs every remaining bounce
// of the batch, trace and shade phases separated by the cluster's hardware barrier, and stops as soon as the queue
// is empty.  Used from the first bounce that fewer than ~24 K rays enter: there a full-grid launch pair costs
// more in launch latency and per-CTA set-up than the work itself.  Queue/bin data and the counters are read with
// .cg loads (they were written by other SMs earlier in this launch).
template <class SceneT>
__global__ void __cluster_dims__(kTailCluster, 1, 1) __launch_bounds__(kTailBlock, 1)
  k_tail_loop(const __grid_constant__ B2Camera cam, const __grid_constant__ SceneT scene,
              const __grid_constant__ B2Lights lights, const __grid_constant__ B2RenderArgs A)
{
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int w = blockIdx.x * (kTailBlock / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int64_t tailWarps = (int64_t)gridDim.x * (kTailBlock / 32);
  __shared__ StageArea<SceneT> sStage;
  const SceneT& S = stage_scene(scene, sStage);
  const B2Lights& LT = stage_lights(lights, sStage);
  __syncthreads();
  for (int depth = A.depth; depth < A.maxDepth; ++depth)
  {
    const int64_t nIn = (int64_t)__ldcg(&A.depthTotals[depth - 1]);
    if (nIn == 0)
      break; // uniform over the cluster: nobody writes this counter any more
    trace_body<false, SceneT, true>(cam, S, A, depth, w, lane, nIn, tailWarps);
    __threadfence();
    cluster.sync();
    shade_body<SceneT, true, true>(S, LT, A, depth, w, lane, tailWarps);
    __threadfence();
    cluster.sync();
  }
}

// Per view and per tile of 32 consecutive pixels: which primitives of a small scene can any primary ray of the tile
// hit (B2RenderArgs::primMask), plus the per-view constants of quad_hit_primary (B2PrimQuad).  One thread per
// (view, tile); double precision, a few hundred operations per quad.  The rule is a rigorous superset of what the
// per-ray candidate filter of closest_small keeps (DESIGN.md "primary tiles"):
//  * The float direction of a primary ray (Camera.cxx:483-524 in float, then normalised) is parallel, to within
//    2e-6 rad, to  nlook + dx*sx + dy*sy  for some (sx, sy) in the tile's jitter rectangle; widening the rectangle by
//    `grow` pixels (>= 4x that angle) makes it exactly parallel to a direction of the widened frustum, and the hit
//    point on a plane does not depend on the direction's length.
//  * For a plane  x_n = c  of a filter frame the hit coordinates  o_u + (c - o_n) d_u/d_n  are linear-fractional in
//    (sx, sy) while d_n keeps its sign, so their range over the frustum is attained at its four corner directions.
//  * The per-ray filter passes a quad iff its (float) hit point lies in the quad's rectangle widened by
//    marg = S (2e-5 + 2e-5 D), D = |d|_1/|d_n|, which bounds its own evaluation error too; the tile keeps the quad iff
//    the corner range meets the rectangle widened by 2.02 marg(D_max).  d_n changing sign (or nearly grazing) keeps
//    every quad of that axis.  A plane wholly behind the tile (t < 0 everywhere, by more than 1e-3 S, D < 50) is
//    dropped: the exact test rejects t < 0.
//  * Gate boxes (boxed quads, spheres): interval slab test of the frustum against the box widened by 1e-5 S, far
//    beyond the rounding of the per-ray float slab test that remains the acceptance rule.
__global__ void __launch_bounds__(128)
  k_primary_prep(const __grid_constant__ B2SmallScene S, const __grid_constant__ B2Camera cam0, const B2Camera* views,
                 int nViews, int tilesPerView, uint2* masks, B2PrimQuad* pq)
{
  const int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (int64_t)nViews * tilesPerView)
    return;
  const int view = (int)(id / tilesPerView), tile = (int)(id - (int64_t)view * tilesPerView);
  const B2Camera cam = views ? views[view] : cam0;
  for (int q = tile; q < S.nQuads; q += tilesPerView)
  { // per-view quad constants, dealt over the view's threads; the float arithmetic of quad_hit (this file is compiled
    // without FMA contraction)
    const B2Quad& Q = S.quads[q];
    const f3 o = ld3(cam.pos);
    const f3 T = o - ld3(Q.v00);
    const f3 Qv = cross3(T, ld3(Q.e01));
    B2PrimQuad C;
    C.T[0] = T.x, C.T[1] = T.y, C.T[2] = T.z;
    C.tnum = dot3(ld3(Q.e03), Qv);
    C.Qv[0] = Qv.x, C.Qv[1] = Qv.y, C.Qv[2] = Qv.z;
    C.tn1 = (fabsf(T.x) + fabsf(T.y)) + fabsf(T.z) + Q.secC1;
    pq[(size_t)view * B2PT_SMALL_MAX_QUADS + q] = C;
  }
  // pixel rectangle of the tile (a tile that wraps to the next row covers whole rows)
  const int W = cam.W, H = cam.H;
  const int64_t p0 = (int64_t)tile * 32, p1 = min(p0 + 31, (int64_t)W * H - 1);
  int i0 = (int)(p0 % W), i1 = (int)(p1 % W);
  const int j0 = (int)(p0 / W), j1 = (int)(p1 / W);
  if (j1 != j0)
    i0 = 0, i1 = W - 1;
  const double dxl = sqrt((double)cam.dx[0] * cam.dx[0] + (double)cam.dx[1] * cam.dx[1] + (double)cam.dx[2] * cam.dx[2]);
  const double dyl = sqrt((double)cam.dy[0] * cam.dy[0] + (double)cam.dy[1] * cam.dy[1] + (double)cam.dy[2] * cam.dy[2]);
  const double growx = fmax(0.01, 1.6e-5 / fmax(dxl, 1e-300)), growy = fmax(0.01, 1.6e-5 / fmax(dyl, 1e-300));
  // sx = i + (1 - ru) - W/2 in [i - W/2, i + 1 - W/2], sy = j + rv - H/2 (Camera.cxx:508-509)
  const double sx[2] = { (double)i0 - 0.5 * W - growx, (double)i1 + 1.0 - 0.5 * W + growx };
  const double sy[2] = { (double)j0 - 0.5 * H - growy, (double)j1 + 1.0 - 0.5 * H + growy };
  double dw[4][3]; // corner directions, world frame
  for (int k = 0; k < 4; ++k)
    for (int c = 0; c < 3; ++c)
      dw[k][c] = (double)cam.nlook[c] + (double)cam.dx[c] * sx[k & 1] + (double)cam.dy[c] * sy[k >> 1];
  const double ow[3] = { cam.pos[0], cam.pos[1], cam.pos[2] };
  const double Sr = fmax((double)S.sceneAbs, fmax(fabs(ow[0]), fmax(fabs(ow[1]), fabs(ow[2]))));
  uint32_t mx = 0u, my = 0u;
  int pBegin = 0;
  for (int f = 0; f < S.nFrames; ++f)
  {
    const B2Frame& Fr = S.frames[f];
    double ol[3], dl[4][3];
    double Sf = Sr;
    if (Fr.identity)
    {
      for (int c = 0; c < 3; ++c)
      {
        ol[c] = ow[c];
        for (int k = 0; k < 4; ++k)
          dl[k][c] = dw[k][c];
      }
    }
    else
    {
      for (int a = 0; a < 3; ++a)
      {
        ol[a] = (double)Fr.R[3 * a] * (ow[0] - Fr.org[0]) + (double)Fr.R[3 * a + 1] * (ow[1] - Fr.org[1]) +
          (double)Fr.R[3 * a + 2] * (ow[2] - Fr.org[2]);
        for (int k = 0; k < 4; ++k)
          dl[k][a] = (double)Fr.R[3 * a] * dw[k][0] + (double)Fr.R[3 * a + 1] * dw[k][1] + (double)Fr.R[3 * a + 2] * dw[k][2];
      }
      Sf = 4.0 * Sr;
    }
    double dabsMax = 0.0;
    for (int k = 0; k < 4; ++k)
      dabsMax = fmax(dabsMax, fabs(dl[k][0]) + fabs(dl[k][1]) + fabs(dl[k][2]));
    for (int n = 0; n < 3; ++n)
    {
      const int pEnd = Fr.axisEnd[n];
      if (pEnd <= pBegin)
        continue;
      const int u = (n + 1) % 3, v = (n + 2) % 3;
      double dnMin = 1e300;
      bool pos = true, neg = true;
      for (int k = 0; k < 4; ++k)
      {
        dnMin = fmin(dnMin, fabs(dl[k][n]));
        pos = pos && dl[k][n] > 0.0;
        neg = neg && dl[k][n] < 0.0;
      }
      const bool oneSign = (pos || neg) && dnMin > 1e-9 * dabsMax;
      const double D = oneSign ? dabsMax / dnMin : 1e300;
      const double M = 2.02 * Sf * (2e-5 * D + 2e-5);
      for (int p = pBegin; p < pEnd; ++p)
        for (int h = 0; h < 2; ++h)
        {
          const int vis = 2 * p + h;
          if (S.visitSlot[vis] < 0)
            continue;
          bool keep = true;
          if (oneSign && D < 1e6)
          {
            const double kk = (double)S.pairs[p].c[h] - ol[n];
            double umin = 1e300, umax = -1e300, vmin = 1e300, vmax = -1e300;
            for (int k = 0; k < 4; ++k)
            {
              const double tt = kk / dl[k][n];
              const double hu = ol[u] + tt * dl[k][u], hv = ol[v] + tt * dl[k][v];
              umin = fmin(umin, hu), umax = fmax(umax, hu), vmin = fmin(vmin, hv), vmax = fmax(vmax, hv);
            }
            const double uc = S.pairs[p].uc[h], hu = (double)S.pairs[p].hu[h] + M;
            const double vc = S.pairs[p].vc[h], hv = (double)S.pairs[p].hv[h] + M;
            keep = umax >= uc - hu && umin <= uc + hu && vmax >= vc - hv && vmin <= vc + hv;
            const bool behind = (kk > 0.0) != pos; // c - o_n and d_n of opposite sign at every corner: t < 0
            if (behind && fabs(kk) > 1e-3 * Sf && D < 50.0)
              keep = false;
          }
          if (keep)
            mx |= 1u << vis;
        }
      pBegin = pEnd;
    }
    pBegin = max(pBegin, Fr.axisEnd[2]);
  }
  // gate boxes of the boxed quads and of the spheres: conservative interval slab test in world coordinates
  double dlo[3], dhi[3];
  for (int c = 0; c < 3; ++c)
  {
    dlo[c] = fmin(fmin(dw[0][c], dw[1][c]), fmin(dw[2][c], dw[3][c]));
    dhi[c] = fmax(fmax(dw[0][c], dw[1][c]), fmax(dw[2][c], dw[3][c]));
  }
  auto box_may_hit = [&](const float* bmin, const float* bmax) -> bool {
    double enter = 0.0, leave = 1e300; // lowest possible entry, highest possible exit over the direction box
    for (int c = 0; c < 3; ++c)
    {
      const double pad = 1e-5 * Sr + 1e-5 * ((double)bmax[c] - (double)bmin[c]);
      const double lo = (double)bmin[c] - pad - ow[c], hi = (double)bmax[c] + pad - ow[c];
      if (dlo[c] > 0.0 || dhi[c] < 0.0)
      { // the component keeps its sign: t = (plane - o)/d over d in [dlo, dhi]
        const double a[4] = { lo / dlo[c], lo / dhi[c], hi / dlo[c], hi / dhi[c] };
        const double tnearLo = fmin(fmin(a[0], a[1]), fmin(a[2], a[3]));
        const double tfarHi = fmax(fmax(a[0], a[1]), fmax(a[2], a[3]));
        // (entry and exit of one direction are the smaller / larger of its two plane distances; the extremes over
        // the interval bound them from below / above)
        enter = fmax(enter, tnearLo);
        leave = fmin(leave, tfarHi);
      }
      // a component that may vanish puts no constraint (conservative)
    }
    return enter <= leave;
  };
  for (int g = 0; g < S.nGate; ++g)
    if (box_may_hit(S.gate[g].bmin, S.gate[g].bmax))
      my |= 1u << g;
  for (int s = 0; s < S.nSph; ++s)
    if (box_may_hit(S.sphGate[s].bmin, S.sphGate[s].bmax))
      my |= 1u << (B2PT_PRIM_SPH_SHIFT + s);
  masks[id] = make_uint2(mx, my);
}

__global__ void __launch_bounds__(256)
  k_accumulate(float4* __restrict__ color, const float4* __restrict__ rad, int nPixels, int samplesPerView, int nViews,
               unsigned long long* nanCounter)
{
  // canvas entry P = view * nPixels + pixel (one view unless the render is view-batched); the view's samples are
  // the slots [view * samplesPerView, (view + 1) * samplesPerView) of the batch
  const int64_t P = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= (int64_t)nPixels * nViews)
    return;
  const int64_t view = P / nPixels;
  const float4* r0 = rad + view * samplesPerView * (int64_t)nPixels + (P - view * nPixels);
  float4 c = color[P];
  int nan = 0;
  for (int b = 0; b < samplesPerView; ++b)
  {
    const float4 r = r0[(size_t)b * nPixels];
    nan += (r.x != r.x || r.y != r.y || r.z != r.z) ? 1 : 0;
    c.x += r.x; // cols += sumtotl, MapperPathTracer.cxx:350, in sample order
    c.y += r.y;
    c.z += r.z;
  }
  color[P] = c;
  if (nan)
    atomicAdd(nanCounter, (unsigned long long)nan);
}

// k_accumulate's loop (same sums, same order, same NaN count) that also keeps the prefix sums at sample counts
// ck.count[0..n-2]: when sample sampleBase + b is the count[k]-th of the pixel, the running sum goes to snapshot
// slice k.  The last checkpoint is `color` itself.  With ck.moment, the running sum of squares r*r (alpha lane 0)
// lives in moment slice n-1 across sample batches and is snapshotted at the same counts.
__global__ void __launch_bounds__(256)
  k_accumulate_checkpoints(float4* __restrict__ color, const float4* __restrict__ rad, int nPixels, int samplesPerView,
                           int nViews, unsigned long long* nanCounter, const __grid_constant__ CheckpointArgs ck)
{
  const int64_t P = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= (int64_t)nPixels * nViews)
    return;
  const int64_t view = P / nPixels;
  const float4* r0 = rad + view * samplesPerView * (int64_t)nPixels + (P - view * nPixels);
  const int64_t e = ck.entry0 + P; // entry of every slice
  float4 c = color[P];
  float4 m = ck.moment ? ck.moment[(ck.n - 1) * ck.sliceStride + e] : make_float4(0.f, 0.f, 0.f, 0.f);
  int k = 0; // next checkpoint this batch can reach
  while (k < ck.n - 1 && ck.count[k] <= ck.sampleBase)
    ++k;
  int nan = 0;
  for (int b = 0; b < samplesPerView; ++b)
  {
    const float4 r = r0[(size_t)b * nPixels];
    nan += (r.x != r.x || r.y != r.y || r.z != r.z) ? 1 : 0;
    c.x += r.x;
    c.y += r.y;
    c.z += r.z;
    if (ck.moment)
    {
      m.x += r.x * r.x;
      m.y += r.y * r.y;
      m.z += r.z * r.z;
    }
    if (k < ck.n - 1 && ck.sampleBase + b + 1 == ck.count[k])
    {
      ck.snap[k * ck.sliceStride + e] = c;
      if (ck.moment)
        ck.moment[k * ck.sliceStride + e] = m;
      ++k;
    }
  }
  color[P] = c;
  if (ck.moment)
    ck.moment[(ck.n - 1) * ck.sliceStride + e] = m;
  if (nan)
    atomicAdd(nanCounter, (unsigned long long)nan);
}

template <class SceneT>
__global__ void __launch_bounds__(256)
  k_primary_hits(const __grid_constant__ B2Camera cam, const __grid_constant__ SceneT scene, uint32_t seedOffset,
                 int32_t* primOut, float* tOut)
{
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= cam.W * cam.H)
    return;
  uint32_t rng = (uint32_t)p + seedOffset;
  f3 d = raygen(cam, p, rng);
  Hit hit;
  bool h = trace(scene, ld3(cam.pos), d, 0.001f, FLT_MAX, hit);
  if (primOut)
    primOut[p] = h ? hit.prim : -1;
  if (tOut)
    tOut[p] = h ? hit.t : FLT_MAX;
}

// -direct G-buffers (main.cc:402-422: runNorms / runAlbedo + the depth buffer): one un-jittered ray per pixel
// (Camera::PerspectiveRayGen), closest QUAD hit (MapperQuad.cxx:103-113 extracts quads only) beyond t = 0, the two
// Shade rules.  Misses leave (0,0,0,0) / depth 0.  The Phong colour image of the stock VTK-m shader is out of scope.
// Closest quad of a direct ray beyond t = 0; on both paths an exact-t tie goes to the lowest quad index (the oracle's
// brute-force order), so the G-buffers do not depend on the trace structure or on the tree a builder made.
__device__ __forceinline__ int closest_direct(const B2SmallScene& S, f3 o, f3 d, float& t)
{
  return closest_small(S, o, d, 0.f, FLT_MAX, t, /*withSpheres*/ false);
}
__device__ __forceinline__ int closest_direct(const B2BvhScene& S, f3 o, f3 d, float& t)
{
  return closest_bvh(S, o, d, 0.f, FLT_MAX, t, /*withSpheres*/ false, /*tiesToLowestIndex*/ true);
}
// One thread per (view, pixel) of a chunk of whole views: idx = view * nPixels + pixel, outputs [view][pixel].  The
// chunk holds fewer than 2^32 pixels, so fastdiv's 32-bit numerator takes idx.
template <class SceneT>
__global__ void __launch_bounds__(256)
  k_direct_views(const __grid_constant__ SceneT scene, const DirectView* __restrict__ views, int64_t n,
                 uint32_t nPixels, uint32_t divMagic, uint32_t divShift, float4* normals, float4* albedo, float* depth,
                 int32_t* primOut)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n)
    return;
  const uint32_t view = fastdiv((uint32_t)idx, divMagic, divShift);
  const int p = (int)((uint32_t)idx - view * nPixels);
  const DirectView& V = views[view];
  const B2Camera cam = V.cam;
  const f3 o = ld3(cam.pos);
  const f3 d = raygen_corner(cam, p);
  float t;
  const int code = closest_direct(scene, o, d, t);
  float4 nrm = make_float4(0.f, 0.f, 0.f, 0.f), alb = nrm;
  float dep = 0.f;
  int prim = -1;
  if (code != B2PT_MISS)
  {
    Hit hit;
    fill_hit(scene, code, o, d, t, hit);
    direct_shade(hit.n, hit.p, o, ld3(V.lookAt), ld3(V.upN), nrm, alb);
    dep = t;
    prim = hit.prim;
  }
  if (normals)
    normals[idx] = nrm;
  if (albedo)
    albedo[idx] = alb;
  if (depth)
    depth[idx] = dep;
  if (primOut)
    primOut[idx] = prim;
}

// Denoiser guides of a chunk of whole views: one thread per (view, pixel), idx = view * nPixels + pixel as in
// k_direct_views.  Sample s is the render's path sample s: its stream, raygen and closest hit (trace) are k_trace's, so
// the features describe the same rays the radiance image averages.  Per sample: albedo = the reflectance the path's
// first bounce applies (lambertian: the texture colour; dielectric: 1, shade_specular's attenuation; emitter: its
// colour clamped to [0,1]), a hit flag, the shading normal and t; all zero on a miss.  The sums run in registers in
// sample order (plain adds under -fmad=false) and slice k receives them after count[k] samples.
template <class SceneT>
__global__ void __launch_bounds__(256)
  k_view_features(const __grid_constant__ SceneT scene, const B2Camera* __restrict__ cams, int64_t n,
                  uint32_t nPixels, uint32_t divMagic, uint32_t divShift, uint32_t seedOffset,
                  const __grid_constant__ FeatureCheckpoints ck, float4* albedoOut, float4* normalDepthOut)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n)
    return;
  const uint32_t view = fastdiv((uint32_t)idx, divMagic, divShift);
  const int p = (int)((uint32_t)idx - view * nPixels);
  const B2Camera cam = cams[view];
  const f3 o = ld3(cam.pos);
  float4 alb = make_float4(0.f, 0.f, 0.f, 0.f), nd = alb;
  const int last = ck.count[ck.n - 1];
  int k = 0, next = ck.count[0];
  for (int s = 0; s < last; ++s)
  {
    uint32_t rng = (uint32_t)p + seedOffset + (uint32_t)s * B2PT_GOLDEN;
    const f3 d = raygen(cam, p, rng);
    Hit hit;
    f3 a = mk3(0.f, 0.f, 0.f), nrm = a;
    float h = 0.f, t = 0.f;
    if (trace(scene, o, d, 0.001f, FLT_MAX, hit))
    {
      a = hit.kind == 2 ? mk3(1.f, 1.f, 1.f)
        : hit.kind == 1 ? mk3(fminf(fmaxf(hit.alb.x, 0.f), 1.f), fminf(fmaxf(hit.alb.y, 0.f), 1.f),
                              fminf(fmaxf(hit.alb.z, 0.f), 1.f))
                        : hit.alb;
      nrm = hit.n;
      h = 1.f;
      t = hit.t;
    }
    alb.x += a.x, alb.y += a.y, alb.z += a.z, alb.w += h;
    nd.x += nrm.x, nd.y += nrm.y, nd.z += nrm.z, nd.w += t;
    if (s + 1 == next)
    {
      const int64_t e = (int64_t)k * n + idx;
      if (albedoOut)
        albedoOut[e] = alb;
      if (normalDepthOut)
        normalDepthOut[e] = nd;
      ++k;
      next = k < ck.n ? ck.count[k] : 0;
    }
  }
}

// pathtracing/Camera.cxx:894-953: fills + RayGen + origin broadcast, fused.
__global__ void __launch_bounds__(256)
  k_create_rays(const __grid_constant__ B2Camera cam, uint32_t* seeds, float* dx, float* dy, float* dz, float* ox,
                float* oy, float* oz, long long* pixelIdx)
{
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= cam.W * cam.H)
    return;
  uint32_t rng = seeds[p];
  f3 d = raygen(cam, p, rng);
  seeds[p] = rng;
  if (dx)
    dx[p] = d.x, dy[p] = d.y, dz[p] = d.z;
  if (ox)
    ox[p] = cam.pos[0], oy[p] = cam.pos[1], oz[p] = cam.pos[2];
  if (pixelIdx)
    pixelIdx[p] = p;
}

template <class SceneT>
__global__ void __launch_bounds__(256)
  k_intersect(const __grid_constant__ SceneT scene, long long n, const float* ox, const float* oy, const float* oz,
              const float* dx, const float* dy, const float* dz, float tmin, float tmax, int32_t* primId, float* hrec9,
              int32_t* matId, int32_t* texId)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  Hit hit;
  bool h = trace(scene, mk3(ox[i], oy[i], oz[i]), mk3(dx[i], dy[i], dz[i]), tmin, tmax, hit);
  primId[i] = h ? hit.prim : -1;
  if (matId)
    matId[i] = h ? hit.mat : -1;
  if (texId)
    texId[i] = h ? hit.texi : -1;
  if (hrec9)
  {
    // Record.h:4 order U,V,T,Nx,Ny,Nz,Px,Py,Pz; u,v are never consumed by the path tracer: written as 0
    hrec9[0 * n + i] = 0.f;
    hrec9[1 * n + i] = 0.f;
    hrec9[2 * n + i] = h ? hit.t : tmax;
    hrec9[3 * n + i] = h ? hit.n.x : 0.f;
    hrec9[4 * n + i] = h ? hit.n.y : 0.f;
    hrec9[5 * n + i] = h ? hit.n.z : 0.f;
    hrec9[6 * n + i] = h ? hit.p.x : 0.f;
    hrec9[7 * n + i] = h ? hit.p.y : 0.f;
    hrec9[8 * n + i] = h ? hit.p.z : 0.f;
  }
}

// main.cc:253-287 NormalizeFunctor: sqrt(de_nan(sum)/spp); the alpha lane goes through the same sqrt.
__global__ void __launch_bounds__(256) k_normalize(float4* color, long long n, float spp)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  float4 c = color[i];
  if (!(c.x == c.x))
    c.x = 0.f;
  if (!(c.y == c.y))
    c.y = 0.f;
  if (!(c.z == c.z))
    c.z = 0.f;
  color[i] = make_float4(sqrtf(c.x / spp), sqrtf(c.y / spp), sqrtf(c.z / spp), sqrtf(c.w / spp));
}

// main.cc:325-384 save(): the three integers the reference prints per pixel of a P3 file, int(255.99 * col[k]) with
// col = NormalizeFunctor(sum) (de_nan, /spp, sqrt); the product is Float64 as in the reference (255.99 is a double
// literal), truncated toward zero; values past 65535 (radiance sums beyond 6.5e4 x spp) saturate.
__global__ void __launch_bounds__(256)
  k_pnm16(const float4* __restrict__ color, long long n, float spp, uint16_t* __restrict__ rgb)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const float4 c = color[i];
  const float v[3] = { c.x, c.y, c.z };
#pragma unroll
  for (int k = 0; k < 3; ++k)
  {
    const float x = (v[k] == v[k]) ? v[k] : 0.f;
    const double p = 255.99 * (double)sqrtf(x / spp);
    rgb[3 * i + k] = (uint16_t)(p >= 65535.0 ? 65535 : __double2int_rz(p));
  }
}

__global__ void __launch_bounds__(256) k_fill_seeds(uint32_t* seeds, int n, uint32_t seedOffset)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    seeds[i] = (uint32_t)i + seedOffset; // MapperPathTracer.cxx:265-267
}

__global__ void __launch_bounds__(256)
  k_sum_peers(float4* dst, const __grid_constant__ PeerPtrs srcs, int G, long long begin, long long end)
{
  for (long long i = begin + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < end;
       i += (long long)gridDim.x * blockDim.x)
  {
    float4 acc = srcs.p[0][i];
    for (int g = 1; g < G; ++g)
    {
      const float4 v = srcs.p[g][i];
      acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
    }
    dst[i - begin] = acc;
  }
}

// --------------------------------------------------------------------------------------- launchers
cudaError_t query_launch_cfg(LaunchCfg* cfg)
{
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return e;
  e = cudaDeviceGetAttribute(&cfg->numSMs, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess)
    return e;
  auto occ = [&](const void* fn, int& out) -> cudaError_t {
    int n = 0;
    cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fn, kBlock, 0);
    out = n > 0 ? n : 1;
    return err;
  };
  if ((e = occ((const void*)k_trace<true, B2SmallScene, false>, cfg->traceBlocksPerSM[1][0])) != cudaSuccess ||
      (e = occ((const void*)k_trace<false, B2SmallScene, false>, cfg->traceBlocksPerSM[0][0])) != cudaSuccess ||
      (e = occ((const void*)k_trace<true, B2BvhScene, false>, cfg->traceBlocksPerSM[1][1])) != cudaSuccess ||
      (e = occ((const void*)k_trace<false, B2BvhScene, false>, cfg->traceBlocksPerSM[0][1])) != cudaSuccess ||
      (e = occ((const void*)k_trace<true, B2WideScene, false>, cfg->traceBlocksPerSM[1][2])) != cudaSuccess ||
      (e = occ((const void*)k_trace<false, B2WideScene, false>, cfg->traceBlocksPerSM[0][2])) != cudaSuccess ||
      (e = occ((const void*)k_shade<B2SmallScene, false, false>, cfg->shadeBlocksPerSM[0][0])) != cudaSuccess ||
      (e = occ((const void*)k_shade<B2BvhScene, false, false>, cfg->shadeBlocksPerSM[0][1])) != cudaSuccess ||
      (e = occ((const void*)k_bounce<B2SmallScene, false, false>, cfg->bounceBlocksPerSM)) != cudaSuccess ||
      (e = occ((const void*)k_bvh_hits, cfg->leanBlocksPerSM)) != cudaSuccess)
    return e;
  return cudaSuccess;
}

// One bounce = k_trace then k_shade on the same stream.  mode B2PT_BOUNCE_REGIONS: both on the fixed persistent
// grid that owns the args.numWarps regions; B2PT_BOUNCE_TO_GLOBAL: the same, but k_shade appends the survivors to
// the flat global queue; B2PT_BOUNCE_TAIL: global queue and bins, a small persistent grid (2 CTAs per SM).
template <class SceneT>
static cudaError_t launch_bounce_t(const LaunchCfg& cfg, bool primary, int mode, const B2Camera& cam, const SceneT& S,
                                   const B2Lights& lights, const B2RenderArgs& args, cudaStream_t stream,
                                   cudaEvent_t betweenStages)
{
  const int grid = (args.numWarps + kWarps - 1) / kWarps;
  const int tailGrid = std::max(1, std::min(grid, cfg.numSMs * 2));
  if (mode == B2PT_BOUNCE_TAIL)
  {
    if (primary)
      return cudaErrorInvalidValue;
    k_trace<false, SceneT, true><<<tailGrid, kBlock, 0, stream>>>(cam, S, args);
  }
  else if (primary)
    k_trace<true, SceneT, false><<<grid, kBlock, 0, stream>>>(cam, S, args);
  else if (std::is_same<SceneT, B2BvhScene>::value && args.perm && args.hits)
  { // split bounce: lean traversal over the sorted order, then the bookkeeping in queue order
    const B2BvhScene& BS = reinterpret_cast<const B2BvhScene&>(S);
    k_bvh_hits<<<cfg.numSMs * cfg.leanBlocksPerSM, kBlock, 0, stream>>>(BS, args);
    k_resolve_hits<<<grid, kBlock, 0, stream>>>(BS, args);
  }
  else
    k_trace<false, SceneT, false><<<grid, kBlock, 0, stream>>>(cam, S, args);
  if (betweenStages)
    cudaEventRecord(betweenStages, stream);
  // (the shade stage never traverses: the wide scene shades through the kernels of its base type)
  using ShadeT = typename std::conditional<std::is_same<SceneT, B2WideScene>::value, B2BvhScene, SceneT>::type;
  const ShadeT& SS = S;
  if (mode == B2PT_BOUNCE_TAIL)
    k_shade<ShadeT, true, true><<<tailGrid, kBlock, 0, stream>>>(SS, lights, args);
  else if (mode == B2PT_BOUNCE_TO_GLOBAL)
    k_shade<ShadeT, false, true><<<grid, kBlock, 0, stream>>>(SS, lights, args);
  else
    k_shade<ShadeT, false, false><<<grid, kBlock, 0, stream>>>(SS, lights, args);
  return cudaGetLastError();
}

// One-kernel pipeline of small scenes.  Bounce 0 = k_trace<PRIMARY> (raygen + closest hit, bins into set 0); bounce
// d >= 1 = k_bounce (shade the hits of bounce d-1, trace, bin into set d&1); d == maxDepth = the closing shade pass.
cudaError_t launch_primary(const LaunchCfg& cfg, const B2Camera& cam, const B2SmallScene& S, const B2RenderArgs& args,
                           cudaStream_t stream)
{
  const int grid = (args.numWarps + kWarps - 1) / kWarps;
  k_trace<true, B2SmallScene, false><<<grid, kBlock, 0, stream>>>(cam, S, args);
  return cudaGetLastError();
}

cudaError_t launch_bounce_fused(const LaunchCfg& cfg, int mode, const B2SmallScene& S, const B2Lights& lights,
                                const B2RenderArgs& args, cudaStream_t stream)
{
  if (args.depth < 1)
    return cudaErrorInvalidValue;
  const int grid = (args.numWarps + kWarps - 1) / kWarps;
  const int tailGrid = std::max(1, std::min(grid, cfg.numSMs * 2));
  if (mode == B2PT_BOUNCE_TAIL)
    k_bounce<B2SmallScene, true, true><<<tailGrid, kBlock, 0, stream>>>(S, lights, args);
  else if (mode == B2PT_BOUNCE_TO_GLOBAL)
    k_bounce<B2SmallScene, false, true><<<grid, kBlock, 0, stream>>>(S, lights, args);
  else
    k_bounce<B2SmallScene, false, false><<<grid, kBlock, 0, stream>>>(S, lights, args);
  return cudaGetLastError();
}

cudaError_t launch_bounce_tail_loop(const B2SmallScene& S, const B2Lights& lights, const B2RenderArgs& args,
                                    cudaStream_t stream)
{
  if (args.depth < 2)
    return cudaErrorInvalidValue;
  k_bounce_tail_loop<B2SmallScene><<<kTailCluster, kTailBlock, 0, stream>>>(S, lights, args);
  return cudaGetLastError();
}

size_t sort_temp_bytes()
{
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, (uint32_t*)nullptr, (uint32_t*)nullptr, kSortBuckets);
  return bytes;
}
int sort_buckets() { return kSortBuckets; }

cudaError_t launch_sort_rays(const B2RenderArgs& args, const float lo[3], const float hi[3], uint32_t* hist,
                             uint32_t* keys, uint32_t* perm, void* temp, size_t tempBytes, cudaStream_t stream)
{
  SortBox box;
  for (int c = 0; c < 3; ++c)
  {
    box.lo[c] = lo[c];
    const float ext = hi[c] - lo[c];
    box.cellsPerUnit[c] = ext > 0.f ? (float)(1 << kSortCellBits) / ext : 0.f;
  }
  const int grid = (args.numWarps + kWarps - 1) / kWarps;
  cudaError_t e = cudaMemsetAsync(hist, 0, sizeof(uint32_t) * kSortBuckets, stream);
  if (e != cudaSuccess)
    return e;
  k_sort_rays<false><<<grid, kBlock, 0, stream>>>(args, box, hist, keys, perm);
  e = cub::DeviceScan::ExclusiveSum(temp, tempBytes, hist, hist, kSortBuckets, stream);
  if (e != cudaSuccess)
    return e;
  k_sort_rays<true><<<grid, kBlock, 0, stream>>>(args, box, hist, keys, perm);
  return cudaGetLastError();
}

// Calls f with the scene a launch traverses: the 8-wide tree when bvh->wide (a B2WideScene built from *bvh), else the
// binary tree *bvh, else the small scene *small.  Returns what f returns.
template <class F>
static auto with_trace_scene(const B2SmallScene* small, const B2BvhScene* bvh, F&& f)
{
  if (bvh && bvh->wide)
  {
    B2WideScene ws;
    static_cast<B2BvhScene&>(ws) = *bvh;
    return f(static_cast<const B2WideScene&>(ws));
  }
  if (bvh)
    return f(*bvh);
  return f(*small);
}

cudaError_t launch_tail_loop(const B2Camera& cam, const B2SmallScene* small, const B2BvhScene* bvh,
                             const B2Lights& lights, const B2RenderArgs& args, cudaStream_t stream)
{
  if (args.depth < 1)
    return cudaErrorInvalidValue;
  with_trace_scene(small, bvh, [&](const auto& S) {
    k_tail_loop<std::decay_t<decltype(S)>><<<kTailCluster, kTailBlock, 0, stream>>>(cam, S, lights, args);
  });
  return cudaGetLastError();
}

cudaError_t launch_bounce(const LaunchCfg& cfg, bool primary, int mode, const B2Camera& cam, const B2SmallScene* small,
                          const B2BvhScene* bvh, const B2Lights& lights, const B2RenderArgs& args,
                          cudaStream_t stream, cudaEvent_t betweenStages)
{
  return with_trace_scene(small, bvh, [&](const auto& S) {
    return launch_bounce_t(cfg, primary, mode, cam, S, lights, args, stream, betweenStages);
  });
}

int warps_per_block() { return kWarps; }

#ifdef B2PT_DEBUG_HIST
extern "C" int b2pt_debug_hist(unsigned long long* out, int reset)
{
  if (out && cudaMemcpyFromSymbol(out, g_debugHist, sizeof(g_debugHist)) != cudaSuccess)
    return -1;
  if (reset)
  {
    unsigned long long z[256] = {};
    if (cudaMemcpyToSymbol(g_debugHist, z, sizeof(z)) != cudaSuccess)
      return -1;
  }
  return 0;
}
#endif

cudaError_t launch_primary_prep(const B2SmallScene& S, const B2Camera& cam, const B2Camera* views, int nViews,
                                int tilesPerView, uint2* masks, B2PrimQuad* pq, cudaStream_t stream)
{
  const int64_t n = (int64_t)nViews * tilesPerView;
  if (n <= 0)
    return cudaSuccess;
  k_primary_prep<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(S, cam, views, nViews, tilesPerView, masks, pq);
  return cudaGetLastError();
}

cudaError_t launch_accumulate(float4* color, const float4* rad, int nPixels, int samplesPerView, int nViews,
                              unsigned long long* nanCounter, cudaStream_t stream)
{
  const int64_t n = (int64_t)nPixels * nViews;
  k_accumulate<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(color, rad, nPixels, samplesPerView, nViews,
                                                                nanCounter);
  return cudaGetLastError();
}

cudaError_t launch_accumulate_checkpoints(float4* color, const float4* rad, int nPixels, int samplesPerView, int nViews,
                                          unsigned long long* nanCounter, const CheckpointArgs& ck, cudaStream_t stream)
{
  const int64_t n = (int64_t)nPixels * nViews;
  k_accumulate_checkpoints<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(color, rad, nPixels, samplesPerView,
                                                                            nViews, nanCounter, ck);
  return cudaGetLastError();
}

cudaError_t launch_primary_hits(const B2Camera& cam, const B2SmallScene* small, const B2BvhScene* bvh,
                                uint32_t seedOffset, int32_t* primOut, float* tOut, cudaStream_t stream)
{
  const int n = cam.W * cam.H;
  with_trace_scene(small, bvh, [&](const auto& S) {
    k_primary_hits<std::decay_t<decltype(S)>><<<(n + 255) / 256, 256, 0, stream>>>(cam, S, seedOffset, primOut, tOut);
  });
  return cudaGetLastError();
}

cudaError_t launch_direct_views(const B2SmallScene* small, const B2BvhScene* bvh, const DirectView* views, int nViews,
                                int nPixels, float4* normals, float4* albedo, float* depth, int32_t* primOut,
                                cudaStream_t stream)
{
  const int64_t n = (int64_t)nViews * nPixels;
  if (n <= 0)
    return cudaSuccess;
  if (n > 0xffffffffLL)
    return cudaErrorInvalidValue;
  uint32_t magic, shift;
  make_fastdiv((uint32_t)nPixels, magic, shift);
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (bvh)
    k_direct_views<B2BvhScene><<<grid, 256, 0, stream>>>(*bvh, views, n, (uint32_t)nPixels, magic, shift, normals,
                                                         albedo, depth, primOut);
  else
    k_direct_views<B2SmallScene><<<grid, 256, 0, stream>>>(*small, views, n, (uint32_t)nPixels, magic, shift, normals,
                                                           albedo, depth, primOut);
  return cudaGetLastError();
}

cudaError_t launch_view_features(const B2SmallScene* small, const B2BvhScene* bvh, const B2Camera* cams, int nViews,
                                 int nPixels, uint32_t seedOffset, const FeatureCheckpoints& ck, float4* albedo,
                                 float4* normalDepth, cudaStream_t stream)
{
  const int64_t n = (int64_t)nViews * nPixels;
  if (n <= 0)
    return cudaSuccess;
  if (n > 0xffffffffLL || ck.n < 1 || ck.n > kMaxCheckpoints)
    return cudaErrorInvalidValue;
  uint32_t magic, shift;
  make_fastdiv((uint32_t)nPixels, magic, shift);
  const unsigned grid = (unsigned)((n + 255) / 256);
  with_trace_scene(small, bvh, [&](const auto& S) {
    k_view_features<std::decay_t<decltype(S)>><<<grid, 256, 0, stream>>>(S, cams, n, (uint32_t)nPixels, magic, shift,
                                                                         seedOffset, ck, albedo, normalDepth);
  });
  return cudaGetLastError();
}

cudaError_t launch_create_rays(const B2Camera& cam, uint32_t* seeds, float* dx, float* dy, float* dz, float* ox,
                               float* oy, float* oz, long long* pixelIdx, cudaStream_t stream)
{
  const int n = cam.W * cam.H;
  k_create_rays<<<(n + 255) / 256, 256, 0, stream>>>(cam, seeds, dx, dy, dz, ox, oy, oz, pixelIdx);
  return cudaGetLastError();
}

cudaError_t launch_intersect(const B2SmallScene* small, const B2BvhScene* bvh, int64_t n, const float* ox,
                             const float* oy, const float* oz, const float* dx, const float* dy, const float* dz,
                             float tmin, float tmax, int32_t* primId, float* hrec9, int32_t* matId, int32_t* texId,
                             cudaStream_t stream)
{
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (grid == 0)
    return cudaSuccess;
  with_trace_scene(small, bvh, [&](const auto& S) {
    k_intersect<std::decay_t<decltype(S)>>
      <<<grid, 256, 0, stream>>>(S, n, ox, oy, oz, dx, dy, dz, tmin, tmax, primId, hrec9, matId, texId);
  });
  return cudaGetLastError();
}

cudaError_t launch_normalize(float4* color, int64_t n, int spp, cudaStream_t stream)
{
  if (n <= 0)
    return cudaSuccess;
  k_normalize<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(color, n, (float)spp);
  return cudaGetLastError();
}

cudaError_t launch_pnm16(const float4* color, int64_t n, int spp, uint16_t* rgb, cudaStream_t stream)
{
  if (n <= 0)
    return cudaSuccess;
  k_pnm16<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(color, n, (float)spp, rgb);
  return cudaGetLastError();
}

cudaError_t launch_fill_seeds(uint32_t* seeds, int n, uint32_t seedOffset, cudaStream_t stream)
{
  if (n <= 0)
    return cudaSuccess;
  k_fill_seeds<<<(n + 255) / 256, 256, 0, stream>>>(seeds, n, seedOffset);
  return cudaGetLastError();
}

cudaError_t launch_sum_peers(float4* dst, const float4* const* srcs, int G, int64_t begin, int64_t end,
                             cudaStream_t stream)
{
  if (G < 1 || G > 8)
    return cudaErrorInvalidValue;
  if (end <= begin)
    return cudaSuccess;
  PeerPtrs pp;
  for (int g = 0; g < 8; ++g)
    pp.p[g] = g < G ? srcs[g] : nullptr;
  int64_t n = end - begin;
  int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  k_sum_peers<<<grid, 256, 0, stream>>>(dst, pp, G, begin, end);
  return cudaGetLastError();
}

} // namespace b2pt
