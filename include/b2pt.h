/*
 * b2pt.h -- C-ABI of libb2pt.so, the B200-native (sm_100a) replacement for the Monte-Carlo
 * render path of m-kim/raytracingtherestofyourlife.
 *
 * The reference has no FFI: its boundary is the C++ class surface MapperPathTracer / PathTracer /
 * Camera / ChannelBuffer / Ray (SURVEY.md 8b).  The C++ facade under
 * raytracingtherestofyourlife_b200/host/ keeps those signatures and calls ONLY the functions
 * declared here; each entry point cites the reference code it replaces (paths relative to the
 * reference root).
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  Every function returns 0 on success
 * or a negative b2pt_status; b2pt_last_error() returns the message of the calling thread's last
 * failure (the facade converts it to vtkm::cont::ErrorBadValue, as MapperPathTracer.cxx:162 and
 * pathtracing/Camera.cxx:645,667,700,720-724 throw).  The caller owns all host pointers; the
 * library owns all device memory unless an external buffer is attached.  One context per GPU;
 * calls on one context must be serialised by the caller; different contexts are independent
 * (each has its own CUDA stream), so G contexts can be driven from one host thread.
 * There is NO CPU fallback: every entry point that computes fails with B2PT_ERR_CUDA when no
 * sm_100-class device is usable.
 */
#ifndef B2PT_H
#define B2PT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2pt_ctx b2pt_ctx;

typedef enum b2pt_status
{
  B2PT_OK = 0,
  B2PT_ERR_BAD_VALUE = -1, /* vtkm::cont::ErrorBadValue in the reference */
  B2PT_ERR_CUDA = -2,      /* CUDA runtime failure or no usable device */
  B2PT_ERR_STATE = -3,     /* call order violated (e.g. render before set_scene) */
  B2PT_ERR_ALLOC = -4,
  B2PT_ERR_UNSUPPORTED = -5
} b2pt_status;

/* b2pt_render flags */
#define B2PT_FLAG_REFERENCE_STREAM 0x1u /* per-pixel persistent RNG stream; dead paths burn the draws the reference \
                                           still consumes (SURVEY A.3) so every trajectory equals the reference's. \
                                           One sample per pass; for parity runs, not for speed. */
#define B2PT_FLAG_KILL_ZERO_THROUGHPUT 0x2u /* stop paths whose throughput is exactly (0,0,0); not valid together   \
                                               with B2PT_FLAG_REFERENCE_STREAM */
#define B2PT_FLAG_NO_DEDUP 0x4u             /* keep bit-identical duplicate quads in the trace list */
#define B2PT_FLAG_FORCE_BVH 0x8u            /* use the BVH traversal kernels even for small scenes */
#define B2PT_FLAG_NO_TAIL 0x20u             /* never switch deep bounces to the global-queue tail mode (A/B parity checks) */
#define B2PT_FLAG_NO_OVERLAP 0x40u          /* run the sample batches one after the other on the context's stream */
#define B2PT_FLAG_GPU_LBVH 0x80u            /* build the BVH on the device (Morton LBVH) instead of the host binned-SAH builder */
#define B2PT_FLAG_VIEWS_NORMALIZE 0x100u     /* b2pt_render_views: apply b2pt_normalize's sqrt(de_nan(sum)/spp) to every view */
#define B2PT_FLAG_VIEWS_PNM16 0x200u         /* b2pt_render_views: rgbaOut receives uint16_t[nViews*W*H*3], the integers of b2pt_read_pnm16 */
#define B2PT_FLAG_NO_PRIMARY_MASKS 0x400u    /* trace primary rays with the generic per-ray candidate filter instead of the per-tile candidate masks (A/B parity checks) */
#define B2PT_FLAG_ONE_KERNEL_BOUNCE 0x800u   /* small scenes: ONE kernel per bounce (k_bounce: shade the hits of bounce d-1, trace bounce d, bin; no ray queue) instead of k_trace + k_shade; bit-identical images, half the HBM traffic, measured slower on B200 (DESIGN.md 4) */
#define B2PT_FLAG_WIDE_BVH 0x1000u           /* BVH scenes: traverse the 8-wide compressed tree (80-byte nodes, 8-bit quantised child boxes) collapsed from the binary tree instead of the binary tree itself; identical hits, fewer dependent fetches, more instructions -- measured slower on B200 (DESIGN.md 4), hence opt-in */
#define B2PT_FLAG_SPLIT_TRACE 0x4000u        /* BVH scenes, binary tree, sorted rays: a lean traversal kernel (k_bvh_hits) followed by k_resolve_hits instead of one k_trace per bounce; bit-identical, measured 0.4 % slower on configs[3] (A/B runs) */
#define B2PT_FLAG_NO_RAY_SORT 0x2000u        /* BVH scenes: trace the ray queue in the order k_shade left it instead of sorted by origin cell and direction octant (A/B runs) */
#define B2PT_FLAG_NO_AA 0x10u               /* do not use the axis-aligned quad specialisation (A/B parity checks) */
/* The build flags: the ones that choose and shape the trace structures (b2pt_build_bvh_ex); every other flag only
 * affects a render. */
#define B2PT_BUILD_FLAGS \
  (B2PT_FLAG_FORCE_BVH | B2PT_FLAG_NO_DEDUP | B2PT_FLAG_NO_AA | B2PT_FLAG_GPU_LBVH | B2PT_FLAG_WIDE_BVH)

typedef struct b2pt_stats
{
  int64_t paths;      /* path samples rendered by the last b2pt_render* call */
  int64_t segments;   /* live ray segments traced */
  int64_t nanSamples; /* path samples with a NaN radiance channel */
  int64_t launches;   /* kernels launched by the call */
  int64_t queueBytes; /* bytes read+written on the SoA ray queues */
  double renderMs;    /* CUDA-event time of the call on the context's stream */
  int32_t batches;    /* sample batches */
  int32_t samplesPerBatch;
  int32_t tracePath;  /* 0 = small-scene (kernel-parameter resident) trace, 1 = BVH traversal */
  int32_t bvhNodes;
  int32_t tracedQuads; /* quads in the trace list after dedup */
  int32_t tracedSpheres;
  int32_t tailDepth;  /* first bounce run in tail mode (global queue); == maxDepth when never */
  int32_t loopDepth;  /* first bounce run inside the persistent cluster launch; == maxDepth when never */
} b2pt_stats;

/* ---- lifetime ------------------------------------------------------------------------------ */
/* Replaces MapperPathTracer::InternalsType (MapperPathTracer.cxx:79-92) + VTK-m device selection
 * (DeviceAdapterTagAny, MapperPathTracer.cxx:220). */
b2pt_ctx* b2pt_create(int device, int* err);
void b2pt_destroy(b2pt_ctx* ctx);
const char* b2pt_last_error(void);
/* Run the context's work on an existing CUDA stream (cudaStream_t as void*); NULL restores its own. */
int b2pt_set_stream(b2pt_ctx* ctx, void* cudaStream);

/* ---- scene --------------------------------------------------------------------------------- */
/* Replaces MapperPathTracer::extract (MapperPathTracer.cxx:178-197), the per-primitive material
 * lookups (Surface.h:191-192, 391-392; EmitWorklet.h:60-64) and the hard-coded light lists
 * (MapperPathTracer.cxx:141-148).  quadIds = Vec<Id,5>(cell,p0..p3); spherePt = point id per sphere.
 * lightQuadIds / lightSpherePt / lightSphereR as used by QuadGenerateDir.h / SphereGenerateDir.h. */
int b2pt_set_scene(b2pt_ctx* ctx, const float* pts, int64_t nPts, const int64_t* quadIds, int64_t nQuads,
                   const int64_t* spherePt, const float* sphereR, int64_t nSpheres, const int64_t* matIdxQuad,
                   const int64_t* texIdxQuad, const int64_t* matIdxSph, const int64_t* texIdxSph, const int* matType,
                   int nMatType, const int* texType, int nTexType, const float* tex, int nTex,
                   const int64_t* lightQuadIds, int nLightQuads, const int64_t* lightSpherePt,
                   const float* lightSphereR, int nLightSpheres, int lightables, float refIdx);
/* Replaces MapperPathTracer::buildBVH (MapperPathTracer.cxx:437-449): QuadIntersector::SetData
 * (pathtracing/QuadIntersector.cxx:109-135), SphereIntersector::SetData
 * (pathtracing/SphereIntersector.cxx:46-76), FindQuadAABBs / FindSphereAABBs (pathtracing/AABBSurface.h) and
 * VTK-m's LinearBVH::Construct.  One tree over quads and spheres; small scenes skip the tree. */
int b2pt_build_bvh(b2pt_ctx* ctx);
/* Same with build-affecting flags (B2PT_BUILD_FLAGS); a later render with other build flags rebuilds. */
int b2pt_build_bvh_ex(b2pt_ctx* ctx, uint32_t flags);

/* Moved spheres: new centres (3 floats per sphere, the order of b2pt_set_scene) and, optionally, radii; counts and
 * materials stay.  A light sphere moves with its scene sphere and takes its new radius.  The reference has no
 * counterpart (its scene is static); this is the input side of b2pt_refit_bvh.  Waits for renders in flight.  Every
 * later trace sees the moved spheres: the kernel-parameter path takes them at once, and on a BVH the next trace call
 * first refits the binary tree (as b2pt_refit_bvh does) or rebuilds the 8-wide one with its build flags, unless
 * b2pt_refit_bvh ran in between.  NULL centres: B2PT_ERR_BAD_VALUE; before b2pt_set_scene: B2PT_ERR_STATE. */
int b2pt_update_spheres(b2pt_ctx* ctx, const float* centers, const float* radii);
/* Refit instead of rebuild: the tree built by b2pt_build_bvh keeps its topology and every node box is recomputed
 * bottom-up on the device from the primitives' current geometry (one kernel, atomic arrival counters as in the LBVH
 * build).  The reference's equivalent is a full LinearBVH::Construct on every RenderCells (QuadIntersector.cxx:134,
 * SphereIntersector.cxx:75).  Closest hits equal a fresh build's (they do not depend on the tree); traversal slows
 * down as primitives drift away from the positions the tree was built for.  Optional after b2pt_update_spheres (the
 * next trace refits a tree the update left behind); calling it keeps the refit out of the next trace call.  Binary
 * tree only: B2PT_ERR_UNSUPPORTED under B2PT_FLAG_WIDE_BVH, whose tree the next trace rebuilds.  B2PT_ERR_STATE before
 * b2pt_build_bvh. */
int b2pt_refit_bvh(b2pt_ctx* ctx);

/* ---- camera -------------------------------------------------------------------------------- */
/* Replaces pathtracing::Camera::SetParameters / CreateRaysImpl set-up (pathtracing/Camera.cxx:625-637,
 * 880-960) and the RayGen constructor (:438-476).  fovDeg in (0,180]; W,H > 0 else B2PT_ERR_BAD_VALUE. */
int b2pt_set_camera(b2pt_ctx* ctx, const float pos[3], const float lookAt[3], const float up[3], float fovDeg, int W,
                    int H);
/* Upper bound, in bytes, of the device memory the context's batch buffers (ray records in flight) may take; 0 = 0.85
 * of the memory that is free at the context's first render.  The reference has no counterpart (its buffers are sized
 * by the canvas, MapperPathTracer.cxx:94-149); results never depend on it. */
int b2pt_set_memory_budget(b2pt_ctx* ctx, int64_t bytes);
/* seeds[i] = i + seedOffset (0 = the reference, MapperPathTracer.cxx:265-267). */
int b2pt_seed(b2pt_ctx* ctx, uint32_t seedOffset);
/* Thin-lens depth of field (DESIGN.md 8h; the book's camera with an aperture and a focus distance, which the reference's
 * camera dropped).  aperture = lens diameter in scene units, finite and >= 0; 0 (the default) is the pinhole: the
 * current behaviour bit for bit, with no extra RNG draws.  focusDistance, finite: > 0 is the distance from the camera
 * position to the plane of focus along the view direction; <= 0 (the default) focuses every camera at its own
 * |lookAt - pos| (a hemisphere sweep that looks at the box centre keeps the box in focus in every view).  NaN, +-inf or
 * a negative aperture gives B2PT_ERR_BAD_VALUE and leaves the state unchanged; the state persists until the next call
 * ((0, 0) restores the pinhole).  With aperture > 0, the primary ray of pixel p, sample s (rng = p + seedOffset +
 * s*0x9E3779B9) of a camera with basis nlook, dx, dy, pos is, in float32 with no FMA and in this order:
 *   1. d0 = the pinhole ray (two jitter draws, unchanged);
 *   2. for k = 0..15: a = 2 randf - 1, b = 2 randf - 1, stop at the first pair with a*a + b*b < 1; after 16 rejections
 *      a = b = 0 (the book's random_in_unit_disk, bounded);
 *   3. per camera: u = dx/|dx|, v = dy/|dy| (|x| = sqrtf((x0*x0 + x1*x1) + x2*x2)), r = aperture/2, f = focusDistance
 *      or |lookAt - pos|;
 *   4. o = (pos + u*(r*a)) + v*(r*b);
 *   5. F = pos + d0*(f / ((d0.x*nlook.x + d0.y*nlook.y) + d0.z*nlook.z)), where the pinhole ray meets the plane of focus;
 *   6. d = F - o, zero components nudged by 1e-7 and normalised by division as the pinhole raygen does;
 *   7. the path continues from (o, d) with the stream after the lens draws.
 * The lens applies to b2pt_render, b2pt_render_range, b2pt_render_views and its _checkpoints, _features, _adaptive and
 * _adaptive_denoised forms, and b2pt_primary_hits (sample 0's lens ray; t, like the features' depth, is measured from
 * o).  View v of a sweep stays bit-identical to b2pt_set_camera(view v) + b2pt_render under the same lens.  It does not
 * apply to the reference's stage hooks b2pt_create_rays and b2pt_intersect, to the -direct G-buffers
 * (b2pt_render_direct, b2pt_render_direct_views: un-jittered corner rays as in the reference), or to
 * b2pt_denoise_views (a pure function of its inputs).  Every render flag works under a lens except
 * B2PT_FLAG_REFERENCE_STREAM, which the reference's lens-less camera defines: b2pt_render and b2pt_render_range with it
 * and aperture > 0 fail with B2PT_ERR_BAD_VALUE before anything runs.  Small scenes trace lens rays without the per-tile
 * primary masks (as under B2PT_FLAG_NO_PRIMARY_MASKS), which assume one ray origin per view. */
int b2pt_set_lens(b2pt_ctx* ctx, float aperture, float focusDistance);

/* ---- render -------------------------------------------------------------------------------- */
/* Replaces MapperPathTracer::RenderCellsImpl's sample x depth loop (MapperPathTracer.cxx:278-350):
 * clears the radiance sum (:222-223) and accumulates spp samples of depth maxDepth into it. */
int b2pt_render(b2pt_ctx* ctx, int spp, int maxDepth, uint32_t flags);
/* Same without clearing, rendering global sample indices [sampleBegin, sampleBegin+sampleCount):
 * the multi-GPU sharding primitive (each rank renders a disjoint sample range of every pixel). */
int b2pt_render_range(b2pt_ctx* ctx, int sampleBegin, int sampleCount, int maxDepth, uint32_t flags);
/* View-batched render.  Replaces the camera loop around runPath of generateHemisphere / fibonacciHemisphere
 * (main.cc:431-561 calling generate() :386-429): nViews independent path-traced images of the resident scene, every
 * one bit-identical to b2pt_set_camera(view) + b2pt_render(spp, maxDepth, flags).  views holds 10 floats per view
 * (pos[3], lookAt[3], up[3], fovDeg); all views share the canvas size W x H.  While W*H*spp fits a sample batch,
 * (view, sample, pixel) is one flat path index space and many views share each launch, so small canvases (the
 * reference's 128 x 128 x 10 spp default) fill the GPU; larger views are rendered one after the other.  The sums land
 * in a library-owned device array [nViews][W*H] of float4 (b2pt_views_device_ptr) and, when rgbaOut is not NULL, are
 * copied to the host array rgbaOut = float[nViews*W*H*4] (the call then synchronises); with B2PT_FLAG_VIEWS_PNM16
 * rgbaOut is uint16_t[nViews*W*H*3] instead (see b2pt_read_pnm16).  The context's own camera and canvas
 * are left untouched.  B2PT_FLAG_REFERENCE_STREAM is rejected (B2PT_ERR_BAD_VALUE). */
int b2pt_render_views(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int spp, int maxDepth,
                      uint32_t flags, void* rgbaOut);
/* b2pt_render_views at several sample counts from one render: renders checkpoints[K-1] samples of every view as
 * b2pt_render_views does (same batching rule) and keeps the running sums at every checkpoint.  checkpoints holds
 * K = nCheckpoints strictly increasing counts >= 1, 1 <= K <= 32.  Slice k of rgbaOut, [k][view][j*W+i], holds the
 * bits b2pt_render_views(..., spp = checkpoints[k], flags) returns: float4 sums, normalised with checkpoints[k] under
 * B2PT_FLAG_VIEWS_NORMALIZE, uint16_t[3] integers computed with checkpoints[k] under B2PT_FLAG_VIEWS_PNM16.
 * moment2Out receives, whatever the flags, the float4 per-pixel sums of squared samples r*r (alpha lane 0, sample
 * order) at every checkpoint, [k][view][j*W+i]: with the sums they give each checkpoint's sample variance.  Either
 * output may be NULL; the call synchronises when one is not.  Afterwards b2pt_views_device_ptr holds the last
 * checkpoint as b2pt_render_views(checkpoints[K-1]) leaves it, and stats.paths is W*H*checkpoints[K-1]*nViews.  The
 * context's own camera and canvas are left untouched.  B2PT_ERR_BAD_VALUE, before anything runs: a bad checkpoint
 * list, B2PT_FLAG_REFERENCE_STREAM, a bad view (b2pt_set_camera's message), or more than 2^30 float4 of device output
 * ((K-1) snapshots, K sums of squares when moment2Out is not NULL, and the image, of nViews*W*H each).  nViews == 0
 * does nothing.  The reference has no counterpart: it renders one sample count per sweep (main.cc:386-561). */
int b2pt_render_views_checkpoints(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                                  const int* checkpoints, int maxDepth, uint32_t flags, void* rgbaOut,
                                  float* moment2Out);
/* Denoiser guide buffers of a view sweep: per pixel, the first-hit albedo, normal and depth of the SAME path samples
 * b2pt_render_views_checkpoints averages, summed over the first checkpoints[k] samples.  For view v, pixel
 * p = j*W+i (j = 0 bottom row) and sample s, the primary ray is the renderer's: rng = p + seedOffset + s*0x9E3779B9
 * (b2pt_seed), the jittered raygen of the path tracer, origin at the camera (under b2pt_set_lens: the lens ray, depth
 * measured from its origin on the lens), closest hit in (0.001, FLT_MAX) through
 * the trace structure a render with `flags` uses (quads and spheres).  Per sample, on a hit:
 *   albedo = lambertian (matType 0): the primitive's texture colour; dielectric (2): (1,1,1), the attenuation of the
 *            specular bounce; emitter (1): its colour clamped per channel to [0,1];
 *   hit = 1;  normal = the shading normal (quads: geometric normal flipped to oppose the ray; spheres: (p-c)/r);
 *   depth = t (the ray is unit length: a distance);
 * and all zero on a miss.  albedoOut = (sum albedo.rgb, sum hit) and normalDepthOut = (sum normal.xyz, sum depth),
 * float32 sums over s = 0 .. c-1 in sample order from +0.0, c = checkpoints[k]; layout [k][view][j*W+i] float4,
 * K*nViews*W*H*4 floats each; either may be NULL.  Means are sum / c; the mean depth of the hitting samples is
 * sum depth / sum hit.  views holds 10 floats per view as in b2pt_render_views.  flags may hold only the build flags
 * (B2PT_BUILD_FLAGS), and (re)builds the trace structures as a render would.
 * B2PT_ERR_BAD_VALUE, before anything runs: a bad view list or view (b2pt_set_camera's message), a checkpoint list of
 * other than 1..32 strictly increasing counts >= 1, checkpoints[K-1] > 2^24 (the hit count must stay an exact float),
 * another flag, or K*W*H > 2^30.  nViews == 0 does nothing; no scene gives B2PT_ERR_STATE.  Views run in chunks of
 * whole views through library-owned staging of at most max(2^23, K*W*H) float4 per requested output.  The context's
 * camera, canvas, b2pt_views_device_ptr image and statistics are left untouched.  Synchronises the stream.  The
 * reference has no counterpart. */
int b2pt_render_views_features(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                               const int* checkpoints, uint32_t flags, float* albedoOut, float* normalDepthOut);
/* Motion vectors and disocclusion between the views of a sweep (DESIGN.md 8i), from the primary hits of the SAME path
 * samples b2pt_render_views_features traces.  views and prevViews hold 10 floats per view as in b2pt_render_views, on
 * one W x H canvas; prevViews[v] is the camera view v is reprojected into (for a sweep, view v-1).  For view v with
 * camera C and C' = prevViews[v], pixel p = j*W+i (j = 0 bottom row) and sample s:
 *   1. (o, d) = the primary ray of b2pt_render_views_features (same stream, jittered raygen, under b2pt_set_lens the
 *      lens ray), t = its closest hit in (0.001, FLT_MAX) through the trace structure `flags` selects; on a miss the
 *      sample adds nothing;
 *   2. X = o + d*t per component;
 *   3. proj(C, X): D = X - pos, w = (D.x*nlook.x + D.y*nlook.y) + D.z*nlook.z, x = (D.dx) / (w * (dx.dx)) + W*0.5,
 *      y = (D.dy) / (w * (dy.dy)) + H*0.5, every dot product in that order, with the camera basis of b2pt_set_camera
 *      (nlook unit, |dx| = 2 tan(fov/2) / W, |dy| = 2 tan(fov/2) / H).  Raygen's sample of pixel (i, j) with jitter
 *      (fx, fy) sits at (i + fx, j + fy); the projection ignores any lens (the camera's centre of projection);
 *   4. the sample is valid when w > 0 for C and w' > 0 for C' (NaN is not > 0); an invalid sample adds nothing;
 *   5. motion m = (x' - x, y' - y) in pixels, x to the right and y up;
 *   6. visible = 1 when 0 <= x' < W and 0 <= y' < H and the closest hit from pos' along e = X - pos' (components equal
 *      to 0 nudged by 1e-7, then L = sqrtf((e.x*e.x + e.y*e.y) + e.z*e.z) and e / L per component, as raygen
 *      normalises) in (0.001, FLT_MAX) is absent or has t' >= L * 0.999755859375f (L*(1 - 2^-12)); else 0.  Off the
 *      canvas no visibility ray is traced.
 * motionOut = (sum m.x, sum m.y, sum visible, sum valid) over the valid samples s < checkpoints[k], float32 sums in
 * sample order from +0.0, every operation in float32 without FMA; layout [k][view][j*W+i] float4, K*nViews*W*H*4
 * floats.  Means are sum / sum valid; with prevViews == views the motion sums are exactly 0 and sum valid is the
 * features' hit count.  The scene is the context's, static within the call (spheres moved by b2pt_update_spheres are
 * not tracked: visibility is tested against the current scene).  flags may hold only the build flags.
 * B2PT_ERR_BAD_VALUE, before anything runs: a bad view list or view in either list (b2pt_set_camera's message), a NULL
 * prevViews or motionOut with nViews > 0, a checkpoint list of other than 1..32 strictly increasing counts >= 1,
 * checkpoints[K-1] > 2^24, another flag, or K*W*H > 2^30.  nViews == 0 does nothing; no scene gives B2PT_ERR_STATE.
 * Views run in chunks of whole views through library-owned staging of at most max(2^23, K*W*H) float4; the result does
 * not depend on the chunking.  The context's camera, canvas, b2pt_views_device_ptr image and statistics are left
 * untouched.  Synchronises the stream.  The reference has no counterpart. */
int b2pt_render_views_motion(b2pt_ctx* ctx, int nViews, const float* views, const float* prevViews, int W, int H,
                             int nCheckpoints, const int* checkpoints, uint32_t flags, float* motionOut);
/* Parameters of b2pt_denoise_views.  A sigma may be +inf, which switches its term off. */
typedef struct b2pt_denoise_params
{
  int32_t levels;    /* a-trous levels, 0..10; 0 = no filtering (the output is the mean) */
  float sigmaLum;    /* colour edge-stop, in standard deviations of the mean luminance */
  float sigmaAlbedo; /* albedo + hit-fraction edge-stop */
  float sigmaNormal; /* mean-normal edge-stop */
  float sigmaDepth;  /* relative depth edge-stop, per pixel footprint */
} b2pt_denoise_params;
/* levels 5, sigmaLum 4, sigmaAlbedo 0.1, sigmaNormal 0.3, sigmaDepth 2 (DESIGN.md 8e). */
void b2pt_denoise_defaults(b2pt_denoise_params* p);
/* Spatial denoiser of a view sweep: the edge-avoiding a-trous wavelet filter of SVGF (Schied et al. 2017; Dammertz et
 * al. 2010), its colour edge-stop scaled by the per-pixel standard deviation, guided by the sweep's own buffers.  All
 * inputs are host arrays [k][view][j*W+i] of float4, K*nViews*W*H*4 floats each: color = the radiance sums of
 * b2pt_render_views_checkpoints (flags 0), moment2 = its sums of squares (may be NULL), albedo and normalDepth = the sums
 * of b2pt_render_views_features.  Every (slice k, view v) image is filtered on its own; taps never cross a view, a slice
 * or the image border (taps outside are skipped, the weights renormalised).  With c = checkpoints[k], a pixel's inputs
 * S, Q, A = (a, h), ND = (N, D), dn(x) = x with NaN replaced by 0 and luminance L(x) = 0.2126 x.r + 0.7152 x.g +
 * 0.0722 x.b:
 *   m = dn(S.rgb) / c;  V0 = sum_ch w_ch max(0, dn(Q_ch)/c - m_ch^2) / (c - 1), w = the luminance weights; V0 exists
 *   only when moment2 is given and c >= 2, otherwise the colour term e_l is left out and V is 0 throughout;
 *   guides g_a = (a/c, h/c), g_n = N/c, z = D/h when h > 0.
 * Level i = 0..levels-1, step s = 2^i, taps q = p + s (dx, dy), dx, dy in -2..2, h = (1,4,6,4,1)/16:
 *   w = h[dx] h[dy] exp(-(e_l + e_a + e_n + e_z)),
 *   e_l = |L(x_i(p)) - L(x_i(q))| / (sigmaLum sqrt(V_i(p)) + 1e-6),
 *   e_a = |g_a(p) - g_a(q)|^2 / sigmaAlbedo^2,  e_n = |g_n(p) - g_n(q)|^2 / sigmaNormal^2,
 *   e_z = |z_p - z_q| H / (sigmaDepth z_p s sqrt(dx^2 + dy^2) + 1e-6) when both pixels have h > 0, else 0,
 *   x_{i+1}(p) = sum w x_i(q) / sum w,  V_{i+1}(p) = sum w^2 V_i(q) / (sum w)^2,  x_0 = m, V_0 = V0.
 * out: float4 (x_L.rgb, V_L) per pixel in the input layout; with B2PT_FLAG_VIEWS_PNM16 instead uint16_t[K*nViews*W*H*3],
 * the integers b2pt_read_pnm16 gives for x_L with spp = 1 (levels = 0: the integers of
 * b2pt_render_views_checkpoints(..., B2PT_FLAG_VIEWS_PNM16)).  params NULL = b2pt_denoise_defaults.  A pure function
 * of its inputs: needs no scene, leaves the context's camera, canvas, view images and statistics untouched, and the
 * result depends neither on chunking nor on launch shape.  B2PT_ERR_BAD_VALUE, before anything runs: a bad checkpoint
 * list, NULL color / albedo / normalDepth, W or H <= 0, nViews < 0, levels outside 0..10, a sigma that is NaN or
 * <= 0, a flag other than B2PT_FLAG_VIEWS_PNM16, or one view's K*W*H above 2^30.  nViews == 0 does nothing.  Views run
 * in chunks of whole views through library-owned staging of at most max(2^23, K*W*H) float4 per buffer (four buffers).
 * Synchronises the stream.  The reference has no counterpart (it has no denoiser). */
int b2pt_denoise_views(b2pt_ctx* ctx, int nViews, int W, int H, int nCheckpoints, const int* checkpoints,
                       const float* color, const float* moment2, const float* albedo, const float* normalDepth,
                       const b2pt_denoise_params* params, uint32_t flags, void* out);
/* Parameters of b2pt_denoise_views_temporal.  A tolerance may be +inf, which switches its test off. */
typedef struct b2pt_temporal_params
{
  float alpha;      /* least weight of the new view, (0, 1]; 1 = no history at all */
  float minVisible; /* a pixel takes history only when sum visible >= minVisible * sum valid, [0, 1] */
  float normalTol;  /* tap consistent when |g_n(p) - g_n(q)|^2 <= normalTol^2 */
  float albedoTol;  /* ... and |g_a(p) - g_a(q)|^2 <= albedoTol^2 (four lanes, as the a-trous filter) */
  float depthTol;   /* ... and |z_q - d'| <= depthTol * d' (relative) */
} b2pt_temporal_params;
/* alpha 0.1, minVisible 0.5, normalTol 0.3, albedoTol 0.03, depthTol 0.05 (DESIGN.md 8j). */
void b2pt_temporal_defaults(b2pt_temporal_params* p);
/* Temporal accumulation of a view sweep (the temporal half of SVGF, Schied et al. 2017), then b2pt_denoise_views'
 * a-trous filter.  The inputs are those of b2pt_denoise_views plus views (10 floats per view, the sweep in order, as in
 * b2pt_render_views) and motion = the sums of b2pt_render_views_motion(views, prevViews) with prevViews[v] = views[v-1]
 * for v >= 1 (row 0 of motion is not read), [k][view][j*W+i] float4 like the other inputs.  Every slice k is its own
 * chain: view v takes its history from view v-1 of the same slice, view 0 has none.  The history is the UNFILTERED
 * temporal result (x_bar, V_bar, n) of view v-1 (SVGF feeds back its first filtered level instead; DESIGN.md 8j).
 * Float32 in this order, without FMA.  Pixel p = (i, j) of view v, slice k, c = checkpoints[k]: m, V0, g_a = (a, h),
 * g_n and z as b2pt_denoise_views computes them, (Sx, Sy, Svis, Sval) its motion sums; the state of view v-1 at pixel
 * q is (x_bar_q, V_bar_q), n_q and that view's g_a, g_n, z.
 *   p takes history when v >= 1, alpha < 1, h_p > 0, Sval > 0 and Svis >= minVisible * Sval; otherwise
 *   x_bar = m, V_bar = V0, n = 1.
 *   Reprojection (pixel centres): u = (float)i + Sx/Sval, y = (float)j + Sy/Sval, u0 = floorf(u), y0 = floorf(y),
 *   fu = u - u0, fy = y - y0; taps in the order (0,0), (1,0), (0,1), (1,1) at (u0 + dx, y0 + dy) with the bilinear
 *   weights b = (1-fu)*(1-fy), fu*(1-fy), (1-fu)*fy, fu*fy.  A tap's column and row are tested for [0, W-1] x [0, H-1]
 *   in float before any conversion to int, so NaN or huge motion only gives inconsistent taps.
 *   Expected distance from the previous camera: d_hat = raygen's pinhole direction of camera C for pixel p at jitter
 *   (0.5, 0.5), i.e. sx = (2*((float)i + 0.5f) - W)/2, sy = (2*((float)j + 0.5f) - H)/2, d = (nlook + dx*sx) + dy*sy,
 *   zero components nudged by 1e-7, divided by sqrtf((d.x*d.x + d.y*d.y) + d.z*d.z); X_hat = pos + d_hat*z_p;
 *   e = X_hat - pos' (pos' = the position of views[v-1]); d' = sqrtf((e.x*e.x + e.y*e.y) + e.z*e.z).
 *   Tap q is consistent when it is inside the canvas, h_q > 0, ((dn0*dn0 + dn1*dn1) + dn2*dn2) <= normalTol^2 with
 *   dn = g_n(p) - g_n(q), (((da0*da0 + da1*da1) + da2*da2) + da3*da3) <= albedoTol^2 with da = g_a(p) - g_a(q), and
 *   fabsf(z_q - d') <= depthTol * d'; a tolerance of +inf switches its test off.
 *   Over the consistent taps in tap order, sums from +0: sb = sum b, sx = sum b*x_bar_q (per channel),
 *   sv = sum (b*b)*V_bar_q, sn = sum b*n_q.  If sb > 0: xh = sx/sb, Vh = sv/(sb*sb), nh = sn/sb, n = nh + 1,
 *   a = fmaxf(alpha, 1/n), x_bar = (1-a)*xh + a*m, V_bar = ((1-a)*(1-a))*Vh + (a*a)*V0; if sb = 0, no history.
 * Then denoise.levels levels of b2pt_denoise_views' filter with x_0 = x_bar, V_0 = V_bar and view v's own guides.
 * out: float4 (x_L.rgb, V_L), or under B2PT_FLAG_VIEWS_PNM16 the uint16_t integers of b2pt_denoise_views;
 * historyOut (may be NULL): float32 n per pixel, [k][view][j*W+i].  Guarantees: with alpha = 1, out is bit for bit
 * b2pt_denoise_views(...) with the same denoise parameters and the history is 1 everywhere; with levels = 0, out is
 * (x_bar, V_bar).  temporal NULL = b2pt_temporal_defaults, denoise NULL = b2pt_denoise_defaults.  A pure function of
 * its inputs: needs no scene, leaves the context's camera, canvas, view images and statistics untouched, and the
 * result depends neither on chunking nor on launch shape.  B2PT_ERR_BAD_VALUE, before anything runs: whatever
 * b2pt_denoise_views rejects, a NULL views or motion with nViews > 0, a bad view (b2pt_set_camera's message), alpha NaN
 * or outside (0, 1], minVisible NaN or outside [0, 1], a tolerance NaN or <= 0.  nViews == 0 does nothing.  Views run
 * in chunks of whole views through library-owned staging of at most max(2^23, K*W*H) float4 per buffer (five buffers,
 * plus max(2^23, K*W*H) floats of history); the state of the last view of a chunk (K*W*H float4 of (x_bar, V_bar), two
 * of guides and K*W*H floats of n) is carried into the next.  Steady state allocates nothing.  One small launch per view
 * (view v reads view v-1's result).  Synchronises the stream.  The reference has no counterpart. */
int b2pt_denoise_views_temporal(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                                const int* checkpoints, const float* color, const float* moment2, const float* albedo,
                                const float* normalDepth, const float* motion, const b2pt_temporal_params* temporal,
                                const b2pt_denoise_params* denoise, uint32_t flags, void* out, float* historyOut);
/* A view sweep rendered and temporally denoised in one call, its state kept on the device (DESIGN.md 8k).  Defined as
 * the chain of four calls, bit for bit: with prevViews = (views[0], views[0], views[1], ..., views[nViews-2]),
 * rf = flags & ~B2PT_FLAG_VIEWS_PNM16 and bf = flags & B2PT_BUILD_FLAGS,
 *   colorOut, moment2Out  = b2pt_render_views_checkpoints(views, checkpoints, maxDepth, rf): float4 sums and sums of
 *                           squares;
 *   albedoOut, normalDepthOut = b2pt_render_views_features(views, checkpoints, bf);
 *   motionOut             = b2pt_render_views_motion(views, prevViews, checkpoints, bf);
 *   out, historyOut       = b2pt_denoise_views_temporal(views, checkpoints, color, moment2, albedo, normalDepth,
 *                           motion, temporal, denoise, flags & B2PT_FLAG_VIEWS_PNM16): float4 (x_L.rgb, V_L), or
 *                           uint16_t[3] under B2PT_FLAG_VIEWS_PNM16; float32 n.
 * Every array is [k][view][j*W+i], K*nViews*W*H entries.  out is required when nViews > 0; every other output may be
 * NULL and is only a copy of a buffer the call computes anyway, so one call gives a whole denoiser-dataset record
 * (noisy sums, variance, guides, motion, denoised target).  The seed offset (b2pt_seed) and the lens (b2pt_set_lens)
 * apply as they do to the four calls.  Each primary ray of the guides and the motion is traced once for both.
 * Afterwards b2pt_views_device_ptr and the statistics are what b2pt_render_views_checkpoints leaves, and the context's
 * camera and canvas are untouched.  B2PT_ERR_BAD_VALUE, before anything runs: whatever one of the four calls rejects,
 * B2PT_FLAG_VIEWS_NORMALIZE (the sums stay raw), B2PT_FLAG_REFERENCE_STREAM, a NULL out with nViews > 0,
 * checkpoints[K-1] > 2^24, or more than 2^30 float4 of render state (2K nViews W H).  nViews == 0 does nothing; no
 * scene gives B2PT_ERR_STATE.  Views are denoised in chunks of whole views through b2pt_denoise_views_temporal's
 * staging; only the requested outputs are copied to the host.  Synchronises the stream once.  The reference has no
 * counterpart. */
int b2pt_render_views_temporal_denoised(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nCheckpoints,
                                        const int* checkpoints, int maxDepth, const b2pt_temporal_params* temporal,
                                        const b2pt_denoise_params* denoise, uint32_t flags, void* out,
                                        float* historyOut, float* colorOut, float* moment2Out, float* albedoOut,
                                        float* normalDepthOut, float* motionOut);
/* Parameters of b2pt_render_views_adaptive. */
typedef struct b2pt_adaptive_params
{
  float threshold; /* tau: target relative standard error of a pixel's mean luminance, >= 0 (0 = never converged;
                      +inf = stop after round 0) */
  float epsilon;   /* absolute floor added to the mean luminance, > 0 */
  int32_t radius;  /* 0..4: a pixel keeps sampling while any pixel within this Chebyshev radius in its view is
                      unconverged */
} b2pt_adaptive_params;
/* threshold 0.02, epsilon 0.01, radius 1 (DESIGN.md 8f). */
void b2pt_adaptive_defaults(b2pt_adaptive_params* p);
/* Adaptive sampling of a view sweep: every pixel stops at the first round its own variance calls converged.  views
 * holds 10 floats per view as in b2pt_render_views; rounds is a list of K = nRounds sample counts as
 * b2pt_render_views_checkpoints takes it (1..32 strictly increasing counts), with rounds[0] >= 2.
 * Round 0 renders rounds[0] samples of every pixel (b2pt_render_views_checkpoints with sums of squares).  After round
 * k < K-1, with c = rounds[k], a pixel is unconverged when its count is c and, in float32 in this order (no FMA),
 *   m = dn(S)/c and V0 as b2pt_denoise_views computes them (dn: NaN -> 0; V0 with the luminance weights),
 *   L = 0.2126 m.r + 0.7152 m.g + 0.0722 m.b,  e = tau (L + epsilon),
 * the test V0 <= e*e fails (a NaN V0 or L fails it; tau = 0 converges nothing).  A pixel is active in round k+1 when
 * its count is c and some pixel of its view within Chebyshev distance `radius` is unconverged; active pixels get
 * samples [rounds[k], rounds[k+1]), the others keep their count n_p.  Sample s of a pixel is the stream of every
 * render (p + seedOffset + s * GOLDEN), added in sample order, so at every pixel S is the bits of
 * b2pt_render_views(spp = n_p, flags) and Q the sums of squares of b2pt_render_views_checkpoints(rounds) at n_p.
 * Outputs, [view][j*W+i], any may be NULL: rgbaOut float4 S (VIEWS_NORMALIZE: normalised with each pixel's n_p;
 * VIEWS_PNM16: uint16[3] computed with n_p), moment2Out float4 Q whatever the flags, countOut int32 n_p, activeOut K
 * entries: the pixels sampled in round k (activeOut[0] = nViews*W*H).  params NULL = b2pt_adaptive_defaults.
 * B2PT_ERR_BAD_VALUE, before anything runs: a bad view list, view or round list, REFERENCE_STREAM or
 * ONE_KERNEL_BOUNCE, a NaN or negative threshold, epsilon <= 0 or NaN, a radius outside 0..4, or more than 2^30
 * float4 of device state (2 nViews W H).  nViews == 0 does nothing.  The context's camera and canvas are untouched;
 * afterwards b2pt_views_device_ptr holds the image (S, normalised in place under VIEWS_NORMALIZE as b2pt_render_views
 * does); stats.paths counts the paths of every round.  One 4-byte device-to-host read per round.  Synchronises the
 * stream.  The reference has no counterpart. */
int b2pt_render_views_adaptive(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nRounds,
                               const int* rounds, int maxDepth, const b2pt_adaptive_params* params, uint32_t flags,
                               void* rgbaOut, float* moment2Out, int32_t* countOut, int64_t* activeOut);
/* An adaptive sweep denoised on the device: b2pt_render_views_adaptive, then b2pt_denoise_views' filter at every
 * pixel's own sample count n_p, from the sums the render leaves on the device (only the outputs are copied).
 * rgbaOut and countOut are, bit for bit, what b2pt_render_views_adaptive returns for the same arguments (flags 0,
 * VIEWS_NORMALIZE or VIEWS_PNM16), and afterwards b2pt_views_device_ptr and the statistics are as it leaves them.
 * Guides, [view][j*W+i] float4, either may be NULL: albedoOut = (sum albedo.rgb, sum hit) and normalDepthOut =
 * (sum normal.xyz, sum depth) over the pixel's own samples s = 0 .. n_p-1 with b2pt_render_views_features' per-sample
 * rule, so a pixel holds the bits of b2pt_render_views_features(views, rounds) in the slice k with rounds[k] == n_p.
 * denoisedOut: b2pt_denoise_views' filter with checkpoints[k] replaced by n_p in the prep (c = n_p >= rounds[0] >= 2,
 * so V0 always exists): m = dn(S)/n_p, V0 = sum_ch w_ch max(0, dn(Q_ch)/n_p - m_ch^2)/(n_p - 1), g_a = (a/n_p, h/n_p),
 * g_n = N/n_p, z = D/h where h > 0, from S before any VIEWS_NORMALIZE conversion; then `levels` a-trous levels.  Per
 * pixel float4 (x_L.rgb, V_L), or under VIEWS_PNM16 uint16_t[3], the integers b2pt_read_pnm16 gives for x_L with
 * spp = 1 (levels = 0: the adaptive rgbaOut integers).  adaptive NULL = b2pt_adaptive_defaults, denoise NULL =
 * b2pt_denoise_defaults.  B2PT_ERR_BAD_VALUE, before anything runs: whatever b2pt_render_views_adaptive rejects,
 * levels outside 0..10, a sigma that is NaN or <= 0, or rounds[K-1] > 2^24.  nViews == 0 does nothing; no scene gives
 * B2PT_ERR_STATE.  Views are denoised in chunks of whole views through library-owned staging of at most
 * max(2^23, W*H) float4 per buffer; the result depends neither on the chunking nor on the launch shape.  The context's
 * camera and canvas are untouched.  Synchronises the stream.  The reference has no counterpart. */
int b2pt_render_views_adaptive_denoised(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, int nRounds,
                                        const int* rounds, int maxDepth, const b2pt_adaptive_params* adaptive,
                                        const b2pt_denoise_params* denoise, uint32_t flags, void* rgbaOut,
                                        int32_t* countOut, float* albedoOut, float* normalDepthOut, void* denoisedOut);
void* b2pt_views_device_ptr(b2pt_ctx* ctx);
int b2pt_clear_color(b2pt_ctx* ctx);
/* Host-side planning rule of the renders above, exposed for tests and capacity planning (no GPU needed): `units`
 * (samples of one view, or whole views) of unitPaths paths each are cut into equal batches -- as few as
 * maxPathsPerBatch allows, but up to `sets` (buffer sets in flight, 4 by default) while every batch keeps at least
 * 32 Mi paths.  The reference has no counterpart: it renders one sample of every pixel per pass
 * (MapperPathTracer.cxx:278). */
int b2pt_plan_batches(int64_t units, int64_t unitPaths, int64_t maxPathsPerBatch, int sets, int64_t* unitsPerBatch,
                      int64_t* nBatches);
/* Attach a caller-owned device buffer of W*H float4 as the radiance sum (NULL detaches). */
int b2pt_set_color_buffer(b2pt_ctx* ctx, void* deviceFloat4);
void* b2pt_color_device_ptr(b2pt_ctx* ctx);
/* Device->host copy of the un-normalised radiance sum, canvas.GetColorBuffer() layout
 * (Vec<Float32,4>[W*H], index j*W+i, j=0 bottom row; alpha lane 0). Synchronises the stream. */
int b2pt_read_color(b2pt_ctx* ctx, float* rgba);
int b2pt_write_color(b2pt_ctx* ctx, const float* rgba);
/* Replaces NormalizeFunctor (main.cc:253-287): in-place sqrt(de_nan(sum)/spp) on the device buffer. */
int b2pt_normalize(b2pt_ctx* ctx, int spp);
/* Replaces NormalizeFunctor + the per-pixel arithmetic of save() (main.cc:253-287, 325-384) without touching the
 * canvas: rgb[3*i+k] = int(255.99 * sqrt(de_nan(sum[i][k]) / spp)), the integers the reference prints into its P3
 * file (Float64 product, truncated; not clamped to 255 -- the light prints 991 -- but saturating at 65535).
 * 6 B per pixel cross PCIe instead of 16.  Synchronises the stream. */
int b2pt_read_pnm16(b2pt_ctx* ctx, int spp, uint16_t* rgb);
int b2pt_synchronize(b2pt_ctx* ctx);
int b2pt_get_stats(b2pt_ctx* ctx, b2pt_stats* out);
/* Per-launch CUDA-event durations (ms, on the context's stream) and input ray counts of the first bounce
 * launches of the last render's first sample batch; returns the number of entries written (<= maxEntries,
 * <= 16) or a negative status.  Feeds the live roofline measurement of bench.py. */
int b2pt_get_bounce_profile(b2pt_ctx* ctx, int maxEntries, float* ms, int64_t* raysIn);
/* Same launches split by stage: duration of the k_trace launch and of the k_shade launch of each bounce. */
int b2pt_get_stage_profile(b2pt_ctx* ctx, int maxEntries, float* traceMs, float* shadeMs, int64_t* raysIn);

/* ---- parity hooks and stage-level entry points --------------------------------------------- */
/* Sample-0 primary rays with seeds[i] = i + seedOffset through the production raygen + trace device
 * code: hit primitive id per pixel (quad q -> q, sphere s -> nQuads+s, miss -> -1) and hit t.
 * Either output may be NULL.  Under b2pt_set_lens the rays are sample 0's lens rays and t is measured from their
 * origin on the lens. */
int b2pt_primary_hits(b2pt_ctx* ctx, int32_t* primId, float* t);
/* Replaces the -direct G-buffer passes of main.cc:402-422 (runNorms / runAlbedo through MapperQuadNormals / MapperQuadAlbedo,
 * raytracing/RayTracerNormals.cxx:47-143 and :234-281, RayTracerAlbedo.cxx:100-143, MapperQuad.cxx:86-150) and the
 * depth image: one un-jittered ray per pixel (Camera::PerspectiveRayGen, pathtracing/Camera.cxx:394-423), the
 * closest QUAD hit (the MapperQuad family extracts quads only), then per hit pixel
 *   normals = (n.x, n.y, n.z, 1)   with n the geometric normal flipped to oppose the ray,
 *   albedo  = (cosPhi R / (cosTheta L), 1) per channel, L / R / cosines as the reference's Shade computes them with the
 *             light at camera + 2 up,
 *   depth   = hit distance along the unit ray (VTK-m's canvas stores a projected depth; not restated),
 * and (0,0,0,0) / 0 / -1 where nothing is hit.  Host outputs W*H*4, W*H*4, W*H floats and W*H ids; any may be NULL.
 * Every scene: small scenes on the kernel-parameter path, larger ones (or B2PT_FLAG_FORCE_BVH) through the binary BVH
 * the context holds, whichever builder made it; spheres are never hit.  Synchronises the stream.  The Phong colour
 * image of VTK-m's stock shader is out of scope. */
int b2pt_render_direct(b2pt_ctx* ctx, float* normals, float* albedo, float* depth, int32_t* primId);
/* The same G-buffers for nViews views in one call: the camera loop of generateHemisphere / fibonacciHemisphere with
 * -direct (main.cc:386-561).  views holds 10 floats per view as in b2pt_render_views (pos[3], lookAt[3], up[3],
 * fovDeg); all views share W x H.  Outputs are [view][j*W+i]: normals and albedo nViews*W*H*4 floats, depth nViews*W*H
 * floats, primId nViews*W*H ids; any may be NULL.  View v gets the bits b2pt_set_camera(view v) + b2pt_render_direct
 * give.  A bad view fails with b2pt_set_camera's message and nothing is rendered; nViews == 0 does nothing.  Device
 * memory is bounded: views run in chunks of whole views of at most 2^22 pixels (one view per chunk when a view is
 * larger), each chunk one launch into library-owned staging buffers copied to its slice of the outputs.  The context's
 * own camera and canvas are left untouched.  Synchronises the stream. */
int b2pt_render_direct_views(b2pt_ctx* ctx, int nViews, const float* views, int W, int H, float* normals,
                             float* albedo, float* depth, int32_t* primId);
/* Replaces pathtracing::Camera::CreateRays (pathtracing/Camera.cxx:880-960): one jittered primary ray
 * per pixel from the current per-pixel seeds; host outputs, any may be NULL. seedsInOut (W*H) is
 * read as the RNG state and updated (2 draws per pixel). */
int b2pt_create_rays(b2pt_ctx* ctx, uint32_t* seedsInOut, float* dirX, float* dirY, float* dirZ, float* originX,
                     float* originY, float* originZ, int64_t* pixelIdx);
/* Replaces MapperPathTracer::intersect (MapperPathTracer.cxx:410-435) for host ray arrays:
 * closest hit in (tmin, tmax) per ray; hrec is 9 planar arrays [U,V,T,Nx,Ny,Nz,Px,Py,Pz] (n each),
 * primId/matId/texId n each. */
int b2pt_intersect(b2pt_ctx* ctx, int64_t n, const float* ox, const float* oy, const float* oz, const float* dx,
                   const float* dy, const float* dz, float tmin, float tmax, int32_t* primId, float* hrec9,
                   int32_t* matId, int32_t* texId);

/* ---- multi-GPU (single process, G contexts) ------------------------------------------------ */
/* Sum the radiance buffers of G contexts (one per GPU) into every context's buffer: the exchange
 * step of the sample-sharded render.  Uses peer access over NVLink. */
int b2pt_allreduce(b2pt_ctx* const* ctxs, int G);

/* ---- host-side scene builders (restated inputs, not kernels) -------------------------------- */
/* CornellBox::buildDataSet (CornellBox.cpp:141-418): 89 points, 22 quads, 1 sphere. */
int b2pt_scene_cornell(float* pts /*3*89*/, int64_t* quadIds /*5*22*/, int64_t* spherePt /*1*/, float* sphereR /*1*/,
                       int64_t* matIdxQuad /*22*/, int64_t* texIdxQuad /*22*/, int64_t* matIdxSph /*1*/,
                       int64_t* texIdxSph /*1*/, int* matType /*5*/, int* texType /*5*/, float* tex /*3*4*/);
/* BASELINE.json configs[3]: nSpheres random lambertian spheres + emissive quad + floor (SURVEY 8d-4).
 * pts: 3*(nSpheres+8); quadIds: 5*2; spherePt/sphereR/matIdxSph/texIdxSph: nSpheres; mat/tex idx quad: 2;
 * matType/texType: 5; tex: 3*4. */
int b2pt_scene_spheres(int64_t nSpheres, float* pts, int64_t* quadIds, int64_t* spherePt, float* sphereR,
                       int64_t* matIdxQuad, int64_t* texIdxQuad, int64_t* matIdxSph, int64_t* texIdxSph, int* matType,
                       int* texType, float* tex);

/* Host-only self-check of the BVH builders (no GPU): the configs[3]-style scene with nSpheres spheres through the binned-SAH
 * builder and the collapse into 8-wide compressed nodes, both validated structurally (every primitive reachable exactly
 * once, boxes nested, quantised boxes conservative).  stats4 = { binary nodes, binary depth, wide nodes, wide depth }. */
int b2pt_bvh_selfcheck(int64_t nSpheres, int64_t* stats4);

int b2pt_version(void);

#ifdef __cplusplus
}
#endif
#endif
