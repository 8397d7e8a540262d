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
                          cudaStream_t stream, cudaEvent_t betweenStages = nullptr, const B2Lens* lens = nullptr);
// One-kernel pipeline of small scenes (b2pt_kernels.cu k_bounce): bounce 0, bounce args.depth >= 1 (the closing shade
// pass when args.depth == args.maxDepth) in one of the three modes above, and every bounce from args.depth >= 2
// (global bins) to the closing pass inside one cluster launch.
// lens (device array, nullptr = pinhole) in launch_bounce (primary) and launch_primary: the thin-lens records of the
// cameras, [view] of args.views or [0] for cam; the primary rays then run through k_trace_lens.
cudaError_t launch_primary(const LaunchCfg& cfg, const B2Camera& cam, const B2SmallScene& S, const B2RenderArgs& args,
                           cudaStream_t stream, const B2Lens* lens = nullptr);
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
// launch_accumulate that also stores the running sums at sample counts count[0..n-2] (k_accumulate_checkpoints).
// Slices are sliceStride float4 apart; entry0 + P is canvas entry P's index in every slice.  snap: n-1 slices, written
// once each; moment (nullptr: none): n slices of sums of squares, slice n-1 the running one (cleared before the first
// batch).  sampleBase: global sample index of the batch's first slot.
constexpr int kMaxCheckpoints = 32;
struct CheckpointArgs
{
  int n;
  int sampleBase;
  int count[kMaxCheckpoints]; // strictly increasing
  float4* snap;
  float4* moment;
  int64_t sliceStride, entry0;
};
cudaError_t launch_accumulate_checkpoints(float4* color, const float4* rad, int nPixels, int samplesPerView, int nViews,
                                          unsigned long long* nanCounter, const CheckpointArgs& ck, cudaStream_t stream);
// lens (host pointer, nullptr = pinhole): sample 0's ray through this thin lens, t measured from its origin.
cudaError_t launch_primary_hits(const B2Camera& cam, const B2SmallScene* small, const B2BvhScene* bvh,
                                uint32_t seedOffset, int32_t* primOut, float* tOut, cudaStream_t stream,
                                const B2Lens* lens = nullptr);
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
// First-hit features of nViews views over their path samples (k_view_features): per (view, pixel) the primary rays of
// samples s = 0 .. count[n-1]-1 (the render's streams: rng = pixel + seedOffset + s * B2PT_GOLDEN), summed in sample
// order; at s + 1 == count[k] the sums go to slice k, outputs [k][view][pixel] with slices nViews * nPixels apart.
// albedo: (albedo rgb, hit); normalDepth: (normal xyz, t); either may be null.  The trace structure is the one the
// renders use (bvh->wide: the 8-wide tree).  nViews * nPixels must stay below 2^32.  lenses (device, nullptr = pinhole):
// the thin-lens record of every camera, the rays then go through lenses[view] as the render's do.
struct FeatureCheckpoints
{
  int n;
  int count[kMaxCheckpoints]; // strictly increasing
};
cudaError_t launch_view_features(const B2SmallScene* small, const B2BvhScene* bvh, const B2Camera* cams, int nViews,
                                 int nPixels, uint32_t seedOffset, const FeatureCheckpoints& ck, float4* albedo,
                                 float4* normalDepth, cudaStream_t stream, const B2Lens* lenses = nullptr);
// Motion vectors of nViews views towards prevCams (k_view_motion): the primary rays of launch_view_features (same
// streams, trace structure and lenses), per sample that hits the motion to prevCams[view] in pixels, its visibility
// there and a valid flag; motion = (sum dx, sum dy, sum visible, sum valid) over the valid samples, stored at the
// checkpoints as launch_view_features stores its sums.  nViews * nPixels must stay below 2^32.
cudaError_t launch_view_motion(const B2SmallScene* small, const B2BvhScene* bvh, const B2Camera* cams,
                               const B2Camera* prevCams, int nViews, int nPixels, uint32_t seedOffset,
                               const FeatureCheckpoints& ck, float4* motion, cudaStream_t stream,
                               const B2Lens* lenses = nullptr);
// launch_view_features and launch_view_motion in one pass (k_view_guides_motion): each sample's primary ray traced
// once, the three outputs (all required) hold the bits the two launches store.
cudaError_t launch_view_guides_motion(const B2SmallScene* small, const B2BvhScene* bvh, const B2Camera* cams,
                                      const B2Camera* prevCams, int nViews, int nPixels, uint32_t seedOffset,
                                      const FeatureCheckpoints& ck, float4* albedo, float4* normalDepth,
                                      float4* motion, cudaStream_t stream, const B2Lens* lenses = nullptr);
// Spatial denoiser of b2pt_denoise_views over one chunk of nImages = K * nViews images of W x H pixels, stored
// [k][view][pixel] (image z = k * nViews + v; its checkpoint count is count[z / nViews]).
// launch_denoise_prep: in place, x (color sums in, (m, V0) out), moment (sums of squares, may be null; read only),
// ga (albedo sums in, (a/c, h/c) out), gnz (normal/depth sums in, (N/c, z) out).
// launch_atrous: one level of step `step` from xIn to xOut (float4 (x.rgb, V)); guides as prep leaves them.
struct DenoiseArgs
{
  int n;                      // checkpoints
  int count[kMaxCheckpoints]; // strictly increasing
  int nViews;                 // views in the chunk
  int hasMoments;
  float sigmaLum, sigmaAlbedo, sigmaNormal, sigmaDepth; // +inf switches a term off
};
cudaError_t launch_denoise_prep(float4* x, const float4* moment, float4* ga, float4* gnz, int nPixels,
                                const DenoiseArgs& a, cudaStream_t stream);
cudaError_t launch_atrous(const float4* xIn, float4* xOut, const float4* ga, const float4* gnz, int W, int H,
                          int step, const DenoiseArgs& a, cudaStream_t stream);
// Temporal accumulation of one view of a sweep (b2pt_denoise_views_temporal, k_temporal) in all nSlices slices: slice k
// of the view's (m, V0) in x[k * stride .. + W*H), turned in place into (x_bar, V_bar), with its guides ga / gnz as
// launch_denoise_prep leaves them, its motion sums and its history n written to hist, at the same offsets.  The
// previous view's state px / pga / pgnz / phist sits at k * pstride; px == nullptr means there is no previous view.
struct TemporalArgs
{
  B2Camera cam;   // camera of the view (pixel-centre ray of the expected distance)
  float prevPos[3]; // position of the previous view's camera
  float alpha, minVisible, normalTol, albedoTol, depthTol; // +inf switches a test off
};
cudaError_t launch_temporal(float4* x, const float4* ga, const float4* gnz, const float4* motion, float* hist,
                            int64_t stride, const float4* px, const float4* pga, const float4* pgnz, const float* phist,
                            int64_t pstride, int nSlices, const TemporalArgs& t, cudaStream_t stream);
// Adaptive sampling of a view sweep (b2pt_render_views_adaptive).  Canvas entries P = view * W*H + pixel, n of them.
// launch_accumulate_list: for e < nReal, the samples rad[b * nPad + e] (b < nSamples) onto color[list[e]] and their
// squares onto moment[list[e]], in sample order (k_accumulate_checkpoints' operations).
// launch_adaptive_mark: after round a.c, unconv[P] = the convergence test failed (first: counts set to a.c first).
// launch_adaptive_select: active[P] = count a.c and an unconverged entry within a.radius in its view, counts of the
// active entries set to a.next; then the active P in ascending order into list and their number into *numActive
// (device), through cub (temp: adaptive_select_temp_bytes(n)).
// launch_list_pad: list[n .. nPad) = list[n-1], nPad - n < 32.
struct AdaptiveArgs
{
  float tau, eps; // threshold and luminance floor (b2pt_adaptive_params)
  int radius, W, H;
  int c, next; // samples of the round just finished, samples after the next one
  int first;   // round 0: the counts are not yet written
};
cudaError_t launch_accumulate_list(float4* color, float4* moment, const float4* rad, const uint32_t* list, int nReal,
                                   int nPad, int nSamples, unsigned long long* nanCounter, cudaStream_t stream);
cudaError_t launch_adaptive_mark(const float4* color, const float4* moment, int32_t* counts, uint8_t* unconv, int64_t n,
                                 const AdaptiveArgs& a, cudaStream_t stream);
size_t adaptive_select_temp_bytes(int64_t n);
cudaError_t launch_adaptive_select(const uint8_t* unconv, int32_t* counts, uint8_t* active, int64_t n,
                                   const AdaptiveArgs& a, uint32_t* list, int32_t* numActive, void* temp,
                                   size_t tempBytes, cudaStream_t stream);
cudaError_t launch_list_pad(uint32_t* list, int n, int nPad, cudaStream_t stream);
// launch_normalize / launch_pnm16 with spp = counts[i] per entry
cudaError_t launch_normalize_counts(float4* color, int64_t n, const int32_t* counts, cudaStream_t stream);
cudaError_t launch_pnm16_counts(const float4* color, int64_t n, const int32_t* counts, uint16_t* rgb,
                                cudaStream_t stream);
// Denoising an adaptive sweep (b2pt_render_views_adaptive_denoised), over one chunk of whole views with each
// (view, pixel) entry's own sample count counts[idx] (the chunk's slice of the adaptive counts).
// launch_view_features_counts: launch_view_features' sums over samples s < counts[idx], stored once per entry (both
// outputs required).  launch_denoise_prep_counts: launch_denoise_prep's arithmetic with c = counts[idx] >= 2 and the
// sums of squares always used; color and moment are read only, (m, V0) goes to x, ga and gnz are converted in place.
cudaError_t launch_view_features_counts(const B2SmallScene* small, const B2BvhScene* bvh, const B2Camera* cams,
                                        int nViews, int nPixels, uint32_t seedOffset, const int32_t* counts,
                                        float4* albedo, float4* normalDepth, cudaStream_t stream,
                                        const B2Lens* lenses = nullptr);
cudaError_t launch_denoise_prep_counts(const float4* color, const float4* moment, const int32_t* counts, float4* x,
                                       float4* ga, float4* gnz, int64_t n, cudaStream_t stream);
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
