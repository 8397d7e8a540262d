// b2pt_types.h -- plain data shared by host set-up code and the sm_100a kernels.
//
// Layout notes (DESIGN.md "Data layout in HBM"):
//  * Small scenes (<= B2PT_SMALL_MAX_QUADS quads, <= B2PT_SMALL_MAX_SPH spheres) travel to the kernels as a
//    __grid_constant__ kernel parameter: every lane reads the same primitive at the same time, so the
//    constant bank (uniform loads) serves them with no vector-register or LSU traffic.
//  * Ray-independent pieces of the reference's Lagae-Dutre quad test (edge vectors, the geometric
//    normal) are precomputed on the host with the same float operations the reference performs per ray
//    (Surface.h:56-58, 79-80, 180-181), so per-ray results stay bit-identical.
//  * Ray queues are SoA-of-16-byte-chunks: three uint4 planes per queue (48 B per ray, 44 B used).
#ifndef B2PT_TYPES_H
#define B2PT_TYPES_H

#include <stdint.h>

#define B2PT_SMALL_MAX_QUADS 48
#define B2PT_SMALL_MAX_SPH 8
#define B2PT_MAX_LIGHT_QUADS 2
#define B2PT_MAX_LIGHT_SPH 2
#define B2PT_GOLDEN 0x9E3779B9u
// device-side copies of the public render flags (include/b2pt.h)
#define B2PT_FLAG_REFERENCE_STREAM_DEV 0x1u
#define B2PT_FLAG_KILL_ZERO_THROUGHPUT_DEV 0x2u
#define B2PT_FLAG_NO_AA_DEV 0x10u // build-time: trace every quad with the general Lagae-Dutre test

struct alignas(16) B2Quad // 32 words = 128 B, 16-byte aligned
{
  float v00[3]; // q
  float e01[3]; // r - q   (Surface.h:58  E01 = v10 - v00)
  float e03[3]; // t - q   (Surface.h:56  E03 = v01 - v00)
  float v11[3]; // s
  float e21[3]; // r - s   (Surface.h:80  E21 = v10 - v11)
  float e23[3]; // t - s   (Surface.h:79  E23 = v01 - v11)
  float nrm[3]; // normalize((r-q)x(s-q)) (Surface.h:180-181), not yet flipped
  float alb[3]; // tex[texType[texIdx]]
  int32_t kind; // matType[matIdx]: 0 lambertian, 1 light, 2 dielectric
  int32_t prim; // original quad index
  int32_t mat;  // matIdx (HitId M)
  int32_t texi; // texIdx (HitId T)
  int32_t gate; // 0: planar quad, no leaf-box gate needed; k>0: must pass slab test of gate box k-1 first
  int32_t pad[1]; // pad[0] != 0: non-planar quad (the leaf box is part of its acceptance rule)
  // Second-triangle shortcut of quad_hit (b2pt_device.cuh): for a parallelogram the second triangle's barycentrics
  // are 1 - alpha, 1 - beta, so its reject tests cannot fire while  (1 - max(alpha, beta)) * |det|  exceeds
  // (|T|_1 + secC1) * |d|_1 * secC2, a bound (>= 8x) on the rounding error of both evaluations.
  // secC1 = 2 (|E01|_1 + |E03|_1), secC2 = 1e-5 |E03|_1; secC2 = +inf for quads that are not parallelograms.
  float secC1, secC2;
};

// Leaf AABB of a primitive as the reference's BVH sees it (pathtracing/AABBSurface.h:24-78).  The reference
// reaches a primitive only if the ray passes this box (one primitive per LinearBVH leaf), which matters for
// non-planar quads: Lagae-Dutre returns spurious far hits on them that the box culls.
struct alignas(16) B2GateBox
{
  float bmin[3];
  float bmax[3];
  int32_t quad; // index of the gated quad in the scene's quad array (BVH path: tested after the traversal)
  int32_t pad;
};
#define B2PT_SMALL_MAX_GATES 24

// Axis-aligned rectangle (E01 = a*e_u, E03 = b*e_v, E23 = a2*e_u, E21 = b2*e_v with exact zeros elsewhere),
// stored in the permuted frame (u,v,n).  Every product of the Lagae-Dutre test that multiplies by one of those
// exact zeros contributes +-0 to its sum, so the test below performs only the remaining operations and is
// bit-identical to the general form for finite inputs (DESIGN.md "axis-aligned specialisation").  The
// permutation sign eps is folded into the constants:
//   P_u = d_n*bPu, P_n = d_u*bPn, det = a*P_u, Q_v = T_n*aQv, Q_n = T_v*aQn, E03.Q = b*Q_v   (first triangle)
//   P'_u = d_n*b2Pu, P'_n = d_u*b2Pn, det' = a2*P'_u, Q'_v = T'_n*a2Qv, Q'_n = T'_v*a2Qn      (second triangle)
struct alignas(16) B2AAQuad // 20 words = 80 B, read as five 16-byte chunks
{
  float v00u, v00v, v00n, bPu;
  float v11u, v11v, v11n, bPn;
  float a, aQv, aQn, b;
  float a2, b2Pu, b2Pn, a2Qv;
  float a2Qn;
  int32_t cls;  // bits 0-2: 0..5 = (u,v,n) = xyz, yzx, zxy, yxz, xzy, zyx; bit 3: consistent rectangle
                // (second-triangle shortcut allowed); -1: not axis-aligned
  int32_t slot; // index into the quad array holding normal / material / ids
  int32_t prim; // original quad index (tie-break: lowest index wins an exact-t tie)
};

struct alignas(16) B2Sphere // 12 words = 48 B
{
  float c[3];
  float r;
  float alb[3];
  int32_t kind;
  int32_t prim; // nQuads + sphere index
  int32_t mat;
  int32_t texi;
  int32_t pad;
};

struct alignas(16) B2LightQuad // light quad used by QuadWorkletGenerateDir / QuadPDFWorklet
{
  B2Quad geo;  // same precomputation as a scene quad
  float area;  // |r-q| * |t-q| (PdfWorklet.h:236-239)
  float pt1[3]; // pts[id[1]]
  float pt2[3]; // pts[id[3]]
  float pad;
  B2AAQuad aa; // aa.cls >= 0: the light quad is an axis-aligned rectangle (fast pdf test)
};

struct B2LightSphere
{
  float c[3];
  float r;
};

struct B2Camera // RayGen members, pathtracing/Camera.cxx:431-438
{
  float nlook[3];
  float dx[3];
  float dy[3];
  float pos[3];
  int32_t W, H;
};

// Thin lens of one camera (b2pt_set_lens, DESIGN.md 8h), built on the host in float32: u = dx/|dx|, v = dy/|dy|,
// r = aperture/2, f = the focus distance along nlook.  Kept apart from B2Camera so that no existing kernel parameter
// block changes; the lens launches take one extra pointer to these records, one per camera.
struct alignas(16) B2Lens
{
  float u[3], v[3];
  float r, f;
};

struct alignas(16) B2Lights
{
  int32_t nLightQuads, nLightSph;
  float weight; // 1/lightables (PdfWorklet.h:294)
  float refIdx;
  B2LightQuad lq[B2PT_MAX_LIGHT_QUADS];
  B2LightSphere ls[B2PT_MAX_LIGHT_SPH];
};

// Candidate filter of the small-scene trace (closest_small, phase 1; records: B2FiltPair).  A planar quad whose plane is normal to one
// axis of a FRAME (frame 0 = world axes; further frames are rotated boxes such as the Cornell tall box) is
// described by that plane's coordinate and the bounding rectangle of its vertices on the other two axes
// (u = axis n+1, v = axis n+2, cyclic).  The filter intersects the ray with the plane in fast arithmetic (FMA,
// MUFU.RCP) and keeps the quad as a CANDIDATE when the hit point lies inside the rectangle widened by a rigorous
// error margin; only candidates run the reference's Lagae-Dutre test (quad_hit), so accepted hits and their t
// stay bit-identical.  Margins: DESIGN.md "candidate filter".
// Filter records are stored two quads at a time so that phase 1 runs on packed FP32 pairs (FFMA2 / FADD2 on
// sm_100): a pair holds two quads of the same frame axis; an odd group is padded with a dummy half (c = NaN, never
// a candidate).  The visit index of a half is 2*pair + half; visitSlot[] maps it to the quad's slot.
struct alignas(16) B2FiltPair // 48 B: three 16-byte chunks
{
  float c[2];  // plane coordinate on the frame axis n
  float uc[2]; // rectangle centre on axis u
  float hu[2]; // half width (static margin included) on axis u
  float vc[2];
  float hv[2];
  uint32_t vis[2]; // visit indices of the two halves (2*pair, 2*pair + 1): the low bits of the filter's keys (FiltState)
};
struct alignas(16) B2Frame // 112 B
{
  float R[9];         // rows = frame axes in world coordinates (world -> frame rotation)
  float org[3];       // frame origin (subtracted before the rotation)
  int32_t axisEnd[3]; // end index in pairs[] of the quads normal to frame axis 0,1,2 (cumulative over frames)
  int32_t identity;   // 1: world axes, no transform
  // absolute error bound of the filter's plane distance, per axis group, in units of (coordinate scale) / |d_n|:
  // 4e-6 in general (rotation into the frame, plane offsets within 1e-6 of the scale); 4e-7 for a group of the world
  // frame whose quads are exactly planar (all four vertices share the float coordinate): there the filter's
  // t' = c rcp(d_n) - o_n rcp(d_n) is off by at most 6e-8 |o_n| / |d_n| and the exact test's t by a relative 6e-7 only
  // (filt_axis).  A tight bound matters for rays that graze their own plane -- every light-sampled ray that leaves the
  // ceiling one unit above the light quad --: with the general bound the own plane passes the distance threshold.
  float eaCoef[3];
  float padf;
  // byte offsets, from the scene's first pair, of the pairs of axis group 0,1,2: [begin, end) -- what filt_axis walks
  // (axisEnd stays the index form k_primary_prep uses)
  uint32_t grpBegin[3], padb;
  uint32_t grpEnd[3], pade;
};
#define B2PT_MAX_FRAMES 4
#define B2PT_MAX_PAIRS 16
#define B2PT_MAX_FILT (2 * B2PT_MAX_PAIRS) // visit indices fit one 32-bit candidate mask

struct alignas(16) B2SmallScene
{
  int32_t nQuads, nSph;
  int32_t nGate, nFilt;
  // Trace order: filtered quads quads[0..nFilt) through the two-phase candidate filter; then the remaining
  // quads, quads[firstBoxed..nQuads), each behind the slab test of its own leaf box gate[quad.gate-1] --
  // planar ones first (the box is a conservative filter there), non-planar ones last (the box is part of the
  // acceptance rule); then the spheres.  quads[] holds every traced quad (attributes by slot).
  int32_t firstBoxed, nFrames;
  float sceneAbs; // max |coordinate| of the traced primitives (scale of the filter margins)
  int32_t pad1;
  B2Frame frames[B2PT_MAX_FRAMES];
  B2FiltPair pairs[B2PT_MAX_PAIRS];
  int32_t visitSlot[B2PT_MAX_FILT]; // visit index -> slot in quads[], -1 for a padding half
  int32_t nVisit, padv[3];          // 2 * number of pairs
  B2GateBox gate[B2PT_SMALL_MAX_GATES];
  B2Quad quads[B2PT_SMALL_MAX_QUADS];
  B2Sphere sph[B2PT_SMALL_MAX_SPH];
  B2GateBox sphGate[B2PT_SMALL_MAX_SPH]; // the spheres' own leaf boxes (centre +- radius, unpadded; sphere_gate)
};

// Primary-ray specialisation of the small-scene trace (k_primary_prep -> k_trace<PRIMARY>).  Every primary ray of a
// view leaves the camera position, so the origin-dependent part of the Lagae-Dutre test is a per-quad constant:
// T = o - v00, Qv = T x E01, tnum = E03 . Qv (Surface.h:62-66, 100-101), evaluated once per view with the same float
// operations quad_hit performs per ray (bit-identical), plus tn1 = (|T|_1 + secC1) of the second-triangle shortcut.
struct alignas(16) B2PrimQuad // 32 B, by slot of B2SmallScene::quads
{
  float T[3];
  float tnum;
  float Qv[3];
  float tn1;
};
// ... and the 32 rays of a tile (32 consecutive pixels) span a narrow frustum, so the set of quads any of them can hit
// is a per-tile constant: a bit mask computed once per view by k_primary_prep with a rigorous superset rule
// (DESIGN.md "primary tiles").  x: bit v = filter visit index v (B2SmallScene::visitSlot); y: bit g = gate box g of a
// boxed quad (g < B2PT_SMALL_MAX_GATES), bit 24+s = sphere s.
#define B2PT_PRIM_SPH_SHIFT 24

// BVH scene: global-memory primitive arrays + 32-byte nodes (see b2pt_bvh.h)
struct B2BvhNode // 32 B, two 16-byte loads
{
  float bmin[3];
  int32_t left;  // inner: index of left child (right = left+1); leaf: first primitive slot
  float bmax[3];
  int32_t count; // 0 = inner node, >0 = leaf with `count` primitive slots
};

#define B2PT_WIDE_STACK 32 // traversal stack entries per ray (groups); the tree may be at most this deep
// 8-wide compressed BVH node (b2pt_wide.h builds it, wide_node_hits in b2pt_device.cuh tests it): 80 B = five 16-byte
// loads.  Child s has the box  org + 2^(e-127) * [qlo[.][s], qhi[.][s]]  per axis; an empty slot has qlo > qhi.
// Inner children are nodes childBase + rank of s in innerMask; primitive children are the leaf-order slots
// primBase + rank of s in primMask.
struct alignas(16) B2WideNode
{
  float org[3];
  uint8_t ex, ey, ez, innerMask;
  uint32_t childBase, primBase;
  uint8_t primMask, pad8[7];
  uint8_t qlo[3][8];
  uint8_t qhi[3][8];
};

struct B2BvhScene
{
  const B2BvhNode* nodes;
  const int32_t* primSlots; // slot -> encoded primitive: >=0 quad index into quads[], <0 sphere ~index
  const float4* leafSph;    // slot -> (cx,cy,cz,r) of the sphere in that slot (zeros for quads): a leaf's spheres are
                            // contiguous, fetched without going through primSlots -> sph[] (one latency, not two)
  const B2Quad* quads;
  const B2Sphere* sph;
  const B2GateBox* gate;
  int32_t nNodes, nQuads, nSph, nGate;
  // the 8-wide tree the traversal walks (nodes / the binary tree above are what it was collapsed from; primSlots and
  // leafSph are in the wide tree's leaf order)
  const uint4* wide; // B2WideNode[nWide] as 5 x uint4 each
  int32_t nWide, wideDepth;
};

// Same scene, traversed through the 8-wide tree (a distinct type selects the wide traversal kernels at compile time;
// B2PT_FLAG_WIDE_BVH; the binary tree is the default).
struct B2WideScene : B2BvhScene
{
};

// One ray queue = three planes of uint4.
struct B2Queue
{
  uint4* p0; // ox oy oz dx
  uint4* p1; // dy dz tr tg
  uint4* p2; // tb pathId rng aux
};

// One set of the four sorted hit bins: bin k (0 specular hits, 1..3 lambertian hits by sampling strategy), entry
// [k*binStride + w*regionCap + i], i < count[k*numWarps + w] (tail mode: flat [k*binStride + i], counts in
// binTotals); a record is three 16-byte planes (ox oy oz dx) (dy dz Tr Tg) (Tb pathId rng t) plus the primitive code.
struct B2Bins
{
  uint4* p0;
  uint4* p1;
  uint4* p2;
  uint32_t* code;
  uint32_t* count; // [4*numWarps]
};

// Launch arguments of the bounce kernels.  The ray queue and the four sorted hit bins are statically
// partitioned into one REGION per persistent warp (numWarps regions of regionCap entries, regionCap a multiple
// of 32): warp w consumes and refills only region w, with register counters -- no atomics on the data path.
// Two pipelines share them:
//  * small scenes, ONE kernel per bounce (k_bounce): the records binned by the trace of bounce d-1 sit in bin set
//    (d-1)&1, are shaded and traced again, and the new hits go to bin set d&1 -- no ray queue at all;
//  * BVH scenes, two kernels per bounce (k_trace, k_shade): k_trace bins into set 0, k_shade reads set 0 and compacts
//    the survivors into the ray queue q.
struct B2RenderArgs
{
  B2Queue q;            // BVH pipeline: compact ray queue, entry [w*regionCap + i], i < qCount[w]
  B2Bins bins[2];
  uint32_t* qCount;     // [numWarps]
  uint32_t* depthTotals; // [maxDepth] of this batch: rays entering bounce d+1 (statistics; in tail mode also the
                         // append counter of the global ray queue)
  uint32_t* binTotals;   // [maxDepth*4] of this batch: tail mode, records appended to global bin k at bounce d
  float4* rad;          // per-path radiance, [b*N + pixel]
  uint32_t* seeds;      // per-pixel persistent RNG state (reference-stream mode)
  // view-batched render (b2pt_render_views): sample slot b of the batch belongs to view b / sppPerView of this
  // array and is that view's sample b % sppPerView; nullptr = single view, the camera kernel parameter
  const B2Camera* views;
  // primary-ray specialisation (small scenes, nPixels % 32 == 0; nullptr = generic path): per view, tilesPerView
  // candidate masks and B2PT_SMALL_MAX_QUADS per-quad constants
  const uint2* primMask;
  const B2PrimQuad* primQuads;
  // BVH pipeline, bounces >= 1 in region mode: the rays of the queue in spatially sorted order (k_sort_keys /
  // k_sort_scatter: perm[j] = queue entry of the j-th ray by origin cell and direction octant); warp w traces the
  // chunk [w*chunk, (w+1)*chunk) of it, chunk = total / numWarps rounded up to whole tiles.  nullptr = queue order.
  // Bounce 0 of a listed round (k_trace LISTED, b2pt_render_views_adaptive): the list instead -- path id b * nPixels
  // + e traces sample sampleBase + b of canvas entry perm[e] = view * sppPerView + pixel with camera views[view];
  // nPixels is the padded list length, and sppPerView / divSpp* hold the pixels per view.
  const uint32_t* perm;
  // BVH pipeline with a binary tree and sorted rays: the closest hit of queue entry r, written by k_bvh_hits
  // (x = bits of t, y = primitive code or B2PT_MISS) and consumed by k_resolve_hits.  nullptr = k_trace does both.
  uint2* hits;
  int64_t binStride;    // numWarps * regionCap
  int64_t nPaths;       // paths in this batch (N * samplesInBatch)
  int32_t numWarps;
  int32_t regionCap;
  int32_t nPixels;
  int32_t sampleBase;   // global index of the batch's first sample
  int32_t depth;        // this bounce
  int32_t maxDepth;
  int32_t sppPerView;
  int32_t tilesPerView; // nPixels / 32
  // n / nPixels and n / sppPerView for 32-bit n without the division sequence (host: make_fastdiv; device: fastdiv):
  // q = (t + ((n - t) >> 1)) >> shift with t = umulhi(n, magic); a divisor of 1 has magic = 0, shift = 0xffffffff
  uint32_t divPixelsMagic, divPixelsShift, divSppMagic, divSppShift;
  int32_t nLightQuads, nLightSph; // light counts (reference-stream mode: draws a dead pixel still burns per depth)
  uint32_t seedOffset;
  uint32_t flags;
};

#endif
