// b2pt_kernels.h -- host-callable launchers of the sm_100a kernels (implemented in b2pt_kernels.cu).
#ifndef B2PT_KERNELS_H
#define B2PT_KERNELS_H

#include <cuda_runtime.h>

#include "b2pt_types.h"

namespace b2pt
{

struct LaunchCfg
{
  int numSMs;
  int traceBlocksPerSM[2][3]; // [primary][0 small scene, 1 binary BVH, 2 8-wide BVH]
  int shadeBlocksPerSM[2][2];
  int bounceBlocksPerSM;
  int leanBlocksPerSM; // k_bvh_hits // k_bounce (one-kernel pipeline of small scenes)
};

// Queries occupancy of the bounce kernels on the current device.
cudaError_t query_launch_cfg(LaunchCfg* cfg);

// One bounce of every ray of the input queue (or, primary=true, of freshly generated camera rays): k_trace
// (K1+K2: raygen + closest hit, hits binned by shading strategy) then k_shade (K3+K5: fused shading, survivors
// compacted into the output queue).  scene is B2SmallScene or B2BvhScene.  betweenStages (optional) is recorded
// after k_trace.  mode: per-warp regions in and out / regions in, flat global queue out / global queue and bins
// (tail of the bounce loop, see k_trace).
enum
{
  B2PT_BOUNCE_REGIONS = 0,
  B2PT_BOUNCE_TO_GLOBAL = 1,
  B2PT_BOUNCE_TAIL = 2
};
cudaError_t launch_bounce(const LaunchCfg& cfg, bool primary, int mode, const B2Camera& cam, const B2SmallScene* small,
                          const B2BvhScene* bvh, const B2Lights& lights, const B2RenderArgs& args,
                          cudaStream_t stream, cudaEvent_t betweenStages = nullptr);
// One-kernel pipeline of small scenes (b2pt_kernels.cu k_bounce): bounce 0, bounce args.depth >= 1 (the closing shade
// pass when args.depth == args.maxDepth) in one of the three modes above, and every bounce from args.depth >= 2
// (global bins) to the closing pass inside one cluster launch.
cudaError_t launch_primary(const LaunchCfg& cfg, const B2Camera& cam, const B2SmallScene& S, const B2RenderArgs& args,
                           cudaStream_t stream);
cudaError_t launch_bounce_fused(const LaunchCfg& cfg, int mode, const B2SmallScene& S, const B2Lights& lights,
                                const B2RenderArgs& args, cudaStream_t stream);
cudaError_t launch_bounce_tail_loop(const B2SmallScene& S, const B2Lights& lights, const B2RenderArgs& args,
                                    cudaStream_t stream);
// Spatial sort of the ray queue of a BVH scene (region mode, after k_shade of bounce args.depth - 1): fills perm[] with
// the queue entries ordered by origin cell (64^3 cells of [lo, hi]) and direction octant.  hist: sort_buckets()
// counters, keys / perm: one uint32 per queue entry, temp: sort_temp_bytes() of scan scratch.
size_t sort_temp_bytes();
int sort_buckets();
cudaError_t launch_sort_rays(const B2RenderArgs& args, const float lo[3], const float hi[3], uint32_t* hist,
                             uint32_t* keys, uint32_t* perm, void* temp, size_t tempBytes, cudaStream_t stream);
// Every bounce from args.depth (>= 1, global-queue mode) to args.maxDepth-1 in one launch of a single thread-block
// cluster; stops early when the queue runs empty.
cudaError_t launch_tail_loop(const B2Camera& cam, const B2SmallScene* small, const B2BvhScene* bvh,
                             const B2Lights& lights, const B2RenderArgs& args, cudaStream_t stream);
// Primary-ray specialisation of small scenes: per (view, tile of 32 pixels) candidate masks + per-view quad constants
// (views == nullptr: the one camera `cam`).
cudaError_t launch_primary_prep(const B2SmallScene& S, const B2Camera& cam, const B2Camera* views, int nViews,
                                int tilesPerView, uint2* masks, B2PrimQuad* pq, cudaStream_t stream);
// K4: color[p] += sum_b rad[b*N + p] in sample order; counts NaN samples into *nanCounter.
int warps_per_block();

// Multiplier and shift of the device's fastdiv (b2pt_kernels.cu) for a divisor d >= 1: with l = ceil(log2 d) and
// m = floor(2^32 (2^l - d) / d) + 1,  n / d = (t + ((n - t) >> 1)) >> (l - 1),  t = umulhi(n, m), for every 32-bit n
// (Granlund & Montgomery 1994, fig. 4.1 as used by libdivide's branch-free u32 divider).  d = 1: shift = 0xffffffff.
inline void make_fastdiv(uint32_t d, uint32_t& magic, uint32_t& shift)
{
  if (d <= 1)
  {
    magic = 0;
    shift = 0xffffffffu;
    return;
  }
  uint32_t l = 0;
  while (((uint64_t)1 << l) < d)
    ++l;
  magic = (uint32_t)((((uint64_t)1 << 32) * (((uint64_t)1 << l) - d)) / d + 1);
  shift = l - 1;
}
cudaError_t launch_accumulate(float4* color, const float4* rad, int nPixels, int samplesPerView, int nViews,
                              unsigned long long* nanCounter, cudaStream_t stream);
cudaError_t launch_primary_hits(const B2Camera& cam, const B2SmallScene* small, const B2BvhScene* bvh,
                                uint32_t seedOffset, int32_t* primOut, float* tOut, cudaStream_t stream);
// -direct G-buffers of nViews views (k_direct_views): per view the camera basis, its look-at point and its up vector
// as Camera::SetUp stores it.  Outputs [view][pixel]: normals / albedo float4, depth float, prim ids; any may be null.
// bvh != nullptr traverses its binary tree (nodes / primSlots in binary leaf order), else the small scene.
// nViews * nPixels must stay below 2^32.
struct DirectView
{
  B2Camera cam;
  float lookAt[3], upN[3];
};
cudaError_t launch_direct_views(const B2SmallScene* small, const B2BvhScene* bvh, const DirectView* views, int nViews,
                                int nPixels, float4* normals, float4* albedo, float* depth, int32_t* primOut,
                                cudaStream_t stream);
cudaError_t launch_create_rays(const B2Camera& cam, uint32_t* seeds, float* dx, float* dy, float* dz, float* ox,
                               float* oy, float* oz, long long* pixelIdx, cudaStream_t stream);
cudaError_t launch_intersect(const B2SmallScene* small, const B2BvhScene* bvh, int64_t n, const float* ox,
                             const float* oy, const float* oz, const float* dx, const float* dy, const float* dz,
                             float tmin, float tmax, int32_t* primId, float* hrec9, int32_t* matId, int32_t* texId,
                             cudaStream_t stream);
cudaError_t launch_normalize(float4* color, int64_t n, int spp, cudaStream_t stream);
cudaError_t launch_pnm16(const float4* color, int64_t n, int spp, uint16_t* rgb, cudaStream_t stream);
cudaError_t launch_fill_seeds(uint32_t* seeds, int n, uint32_t seedOffset, cudaStream_t stream);
// dst[i-begin] = sum_g srcs[g][i] over [begin,end) float4 elements; srcs may be peer-device pointers.
cudaError_t launch_sum_peers(float4* dst, const float4* const* srcs, int G, int64_t begin, int64_t end,
                             cudaStream_t stream);

} // namespace b2pt
#endif
