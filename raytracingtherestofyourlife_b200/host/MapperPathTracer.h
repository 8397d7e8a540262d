// MapperPathTracer.h -- facade of vtkm::rendering::MapperPathTracer (reference MapperPathTracer.h:45-160).
// Same constructor, SetCanvas/GetCanvas, RenderCells, stage methods and public data members, so the
// reference's driver (main.cc::runPath, lines 289-323) compiles and runs unchanged.  RenderCells hands the
// scene to the B200 library and runs the whole sample x depth loop of MapperPathTracer.cxx:278-350 on the GPU
// (b2pt_set_scene / b2pt_build_bvh / b2pt_set_camera / b2pt_render / b2pt_read_color); the canvas colour
// buffer receives the un-normalised radiance sum exactly like MapperPathTracer.cxx:350.
#ifndef b2pt_facade_MapperPathTracer_h
#define b2pt_facade_MapperPathTracer_h

#include <memory>
#include <vector>
#include <tuple>

#include <vtkm/rendering/Rendering.h>

#include "pathtracing/Intersectors.h"
#include "raytracing/Ray.h"

namespace vtkm
{
namespace rendering
{

class MapperPathTracer : public Mapper
{
public:
  using ExtractResult = std::tuple<vtkm::cont::ArrayHandle<vtkm::Id>, vtkm::cont::ArrayHandle<vtkm::Float32>,
                                   vtkm::cont::ArrayHandle<vtkm::Id>, vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>>;

  // sc = samples per pixel, dc = maximum path depth.  matIdx / texIdx point at two-element arrays
  // ([0] quads, [1] spheres) owned by the caller, which must outlive the mapper (reference :133).
  MapperPathTracer(int sc, int dc, vtkm::cont::ArrayHandle<vtkm::Id>* matIdx, vtkm::cont::ArrayHandle<vtkm::Id>* texIdx,
                   vtkm::cont::ArrayHandle<int>& matType, vtkm::cont::ArrayHandle<int>& texType,
                   vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 3>>& tex);
  ~MapperPathTracer() override;

  void SetCanvas(vtkm::rendering::Canvas* canvas) override;
  vtkm::rendering::Canvas* GetCanvas() const override;

  void RenderCells(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                   const vtkm::cont::Field& scalarField, const vtkm::cont::ColorTable& colorTable,
                   const vtkm::rendering::Camera& camera, const vtkm::Range& scalarRange) override;

  // Closest hit of every ray whose status has the scatter bit: fills Distance (t), Normal*, Intersection*,
  // matIdArray/texIdArray of the last buildBVH, kills rays that miss and writes attenuation=1 / emitted=0 for
  // dead rays at `depth` (reference MapperPathTracer.cxx:410-435 + CollectIntersecttWorklet).
  template <typename emittedType, typename attenType>
  void intersect(vtkm::rendering::raytracing::Ray<vtkm::Float32>& rays, vtkm::cont::ArrayHandle<float>& tmin,
                 emittedType& emitted, attenType& attenuation, const vtkm::Id depth);

  void buildBVH(const vtkm::cont::CoordinateSystem& coord, vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>& QuadIds,
                vtkm::cont::ArrayHandle<vtkm::Id>& SphereIds, vtkm::cont::ArrayHandle<vtkm::Float32>& SphereRadii,
                vtkm::cont::ArrayHandle<vtkm::Int32>& matIdArray, vtkm::cont::ArrayHandle<vtkm::Int32>& texIdArray,
                vtkm::cont::ArrayHandle<vtkm::Id>* matIdx, vtkm::cont::ArrayHandle<vtkm::Id>* texIdx);

  // The three per-depth stages below are fused into the bounce kernel together with intersect (one launch per
  // bounce) and have no stand-alone device entry point; calling them throws vtkm::cont::ErrorBadValue.
  template <typename HitRecord, typename HitId, typename ScatterRecord, typename emittedType>
  void applyMaterials(vtkm::rendering::raytracing::Ray<vtkm::Float32>&, HitRecord&, HitId&, ScatterRecord&,
                      vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 3>>&, vtkm::cont::ArrayHandle<int>&,
                      vtkm::cont::ArrayHandle<int>&, emittedType&, vtkm::cont::ArrayHandle<unsigned int>&, vtkm::Id,
                      vtkm::Id)
  {
    FusedStage("applyMaterials");
  }
  template <typename HitRecord, typename ScatterRecord, typename attenType, typename GenDirType>
  void applyPDFs(const vtkm::cont::CoordinateSystem&, vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>&,
                 vtkm::cont::ArrayHandle<vtkm::Id>&, vtkm::cont::ArrayHandle<vtkm::Float32>&,
                 vtkm::cont::ArrayHandle<vtkm::Id>*, vtkm::cont::ArrayHandle<vtkm::Id>*,
                 vtkm::rendering::raytracing::Ray<vtkm::Float32>&, HitRecord&, ScatterRecord&,
                 vtkm::cont::ArrayHandle<vtkm::Float32>&, GenDirType, attenType&, vtkm::cont::ArrayHandle<unsigned int>&,
                 int, vtkm::Id, vtkm::Id)
  {
    FusedStage("applyPDFs");
  }
  void generateRays(const vtkm::cont::CoordinateSystem&, vtkm::cont::ArrayHandle<vtkm::Float32>&,
                    vtkm::cont::ArrayHandle<int>&, vtkm::rendering::raytracing::Ray<vtkm::Float32>&,
                    vtkm::cont::ArrayHandle<vtkm::UInt32>&)
  {
    FusedStage("generateRays");
  }

  // (SphereIds, SphereRadii, ShapeOffset, QuadIds): VERTEX cells become spheres of radius 90/555, QUAD cells
  // become (cell, p0..p3) records (reference MapperPathTracer.cxx:178-197).
  ExtractResult extract(const vtkm::cont::DynamicCellSet& cellset) const;

  void StartScene() override;
  void EndScene() override;
  void SetCompositeBackground(bool on);
  vtkm::rendering::Mapper* NewCopy() const override;

  // B200 additions (not in the reference): render flags (B2PT_FLAG_*) and the statistics of the last render.
  void SetRenderFlags(unsigned int flags) { RenderFlags = flags; }
  // Thin-lens depth of field (b2pt_set_lens): lens diameter and focus distance (<= 0: each camera focuses at its
  // look-at point), passed to the context before every path-traced render and sweep.  (0, 0), the default, is the
  // reference's pinhole; the reference has no counterpart.  The -direct buffers never use it.
  void SetLens(float aperture, float focusDistance)
  {
    LensAperture = aperture;
    LensFocus = focusDistance;
  }
  // The GPUs RenderCells uses (CUDA device ordinals; default: the one of B2PT_DEVICE).  With G > 1 devices the samples
  // of every pixel are partitioned over them -- device g renders a contiguous range of the global sample indices with
  // the same per-(pixel, sample) streams a single GPU would use -- and the radiance sums are added over NVLink
  // (b2pt_allreduce) before the canvas is read back: the single-process form of the sample-sharded render.
  void SetDevices(const std::vector<int>& devices) { Devices = devices; }
  const std::vector<int>& GetDevices() const { return Devices; }
  // Many cameras, one call: what main.cc's generateHemisphere / fibonacciHemisphere loops do by calling RenderCells
  // per view point (main.cc:431-561).  Every camera renders onto a canvas of the size of the canvas set with
  // SetCanvas; image v lands in colors[v] exactly as RenderCells would leave it in canvas->GetColorBuffer()
  // (un-normalised sums, same bits).  Small canvases share GPU launches across views (b2pt_render_views).
  void RenderCellsViews(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                        const std::vector<vtkm::rendering::Camera>& cameras,
                        std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& colors);
  // Same, returning for every view the integers main.cc's save() prints into the P3 file (:325-384) after
  // NormalizeFunctor (:253-287): pnm[(v * W*H + i) * 3 + k] = int(255.99 * sqrt(de_nan(sum) / samplecount)).
  // Packed on the GPU, 6 bytes per pixel cross PCIe instead of 16.
  void RenderCellsViewsPnm(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                           const std::vector<vtkm::rendering::Camera>& cameras, std::vector<unsigned short>& pnm);
  // Same for several sample counts from one render of samplecount samples per view: checkpoints is strictly increasing
  // and ends with samplecount (else ErrorBadValue); pnm[((k * V + v) * W*H + i) * 3 + c] holds the integers
  // RenderCellsViewsPnm gives with samplecount = checkpoints[k] (b2pt_render_views_checkpoints).
  void RenderCellsViewsCheckpointsPnm(const vtkm::cont::DynamicCellSet& cellset,
                                      const vtkm::cont::CoordinateSystem& coords,
                                      const std::vector<vtkm::rendering::Camera>& cameras,
                                      const std::vector<int>& checkpoints, std::vector<unsigned short>& pnm);
  // Denoiser guides of the same sweep (b2pt_render_views_features, on the first device of SetDevices): for every
  // checkpoint c (strictly increasing, ending with samplecount, else ErrorBadValue) and view v, the float4 sums over the
  // primary hits of path samples 0 .. c-1, the samples RenderCellsViewsCheckpointsPnm renders:
  // albedo[((k * V + v) * W*H + i) * 4 + ...] = (albedo rgb, hit count), normalDepth = (normal xyz, depth).
  void RenderCellsViewsFeatures(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                const std::vector<vtkm::rendering::Camera>& cameras, const std::vector<int>& checkpoints,
                                std::vector<float>& albedo, std::vector<float>& normalDepth);
  // Motion vectors of the same sweep (b2pt_render_views_motion, on the first device of SetDevices): prevCameras[v]
  // (one per camera, else ErrorBadValue) is the camera view v is reprojected into; same checkpoint rule.
  // motion[((k * V + v) * W*H + i) * 4 + ...] = the sums over the primary hits of path samples 0 .. c-1 of
  // (motion x, motion y, visible, valid), motion in pixels from view v to prevCameras[v], y up.
  void RenderCellsViewsMotion(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                              const std::vector<vtkm::rendering::Camera>& cameras,
                              const std::vector<vtkm::rendering::Camera>& prevCameras,
                              const std::vector<int>& checkpoints, std::vector<float>& motion);
  // RenderCellsViewsCheckpointsPnm's integers (same checkpoint rule, same bytes in pnm) and, in denoisedPnm, the same
  // layout for the sweep denoised with b2pt_denoise_views' defaults: one render of the float sums and their squares,
  // the guides of RenderCellsViewsFeatures, then the filter (levels 0 for pnm, which is the unfiltered mean).
  void RenderCellsViewsDenoisedPnm(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                   const std::vector<vtkm::rendering::Camera>& cameras,
                                   const std::vector<int>& checkpoints, std::vector<unsigned short>& pnm,
                                   std::vector<unsigned short>& denoisedPnm);
  // The same sweep with temporal accumulation, in the layout of RenderCellsViewsCheckpointsPnm: the float sums and
  // their squares, the guides of RenderCellsViewsFeatures and the motion of RenderCellsViewsMotion towards the view
  // before each in the order of `cameras`, through b2pt_denoise_views_temporal with the default temporal and filter
  // parameters (same checkpoint rule).
  void RenderCellsViewsTemporalPnm(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                   const std::vector<vtkm::rendering::Camera>& cameras,
                                   const std::vector<int>& checkpoints, std::vector<unsigned short>& temporalPnm);
  // Adaptive sampling of the sweep (b2pt_render_views_adaptive with its default epsilon and radius): rounds is a
  // checkpoint list ending with the sample count; every pixel stops at the first round whose variance test it passes.
  // pnm: [view][pixel] the integers of RenderCellsViewsPnm computed with each pixel's own count; counts: [view][pixel]
  // the samples each pixel received.
  void RenderCellsViewsAdaptivePnm(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                   const std::vector<vtkm::rendering::Camera>& cameras, const std::vector<int>& rounds,
                                   float threshold, std::vector<unsigned short>& pnm, std::vector<int>& counts);
  // RenderCellsViewsAdaptivePnm's integers and counts (same rounds rule, same bytes) and, in denoisedPnm, the same
  // layout for the adaptive sweep denoised on the GPU at every pixel's own count with b2pt_denoise_views' defaults
  // (b2pt_render_views_adaptive_denoised).
  void RenderCellsViewsAdaptiveDenoisedPnm(const vtkm::cont::DynamicCellSet& cellset,
                                           const vtkm::cont::CoordinateSystem& coords,
                                           const std::vector<vtkm::rendering::Camera>& cameras,
                                           const std::vector<int>& rounds, float threshold,
                                           std::vector<unsigned short>& pnm, std::vector<int>& counts,
                                           std::vector<unsigned short>& denoisedPnm);
  // The -direct G-buffers of main.cc:402-422 (what MapperQuadNormals / MapperQuadAlbedo leave in the canvas colour
  // buffer, raytracing/RayTracerNormals.cxx / RayTracerAlbedo.cxx, and a depth image) for the canvas set with
  // SetCanvas: one un-jittered ray per pixel, closest quad hit, the reference's two Shade rules (b2pt_render_direct).
  // depth holds the hit distance along the ray (VTK-m's projected canvas depth is not restated).
  void RenderDirectBuffers(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                           const vtkm::rendering::Camera& camera,
                           vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& normals,
                           vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& albedo,
                           vtkm::cont::ArrayHandle<vtkm::Float32>& depth);
  // The same G-buffers for many cameras in one call: what main.cc's generateHemisphere / fibonacciHemisphere do with
  // -direct by calling generate() per view point (main.cc:386-561).  Every camera is validated against the canvas set
  // with SetCanvas; view v lands in normals[v] / albedo[v] / depth[v] with the bits RenderDirectBuffers gives for that
  // camera (b2pt_render_direct_views, on the first device of SetDevices).
  void RenderDirectBuffersViews(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                const std::vector<vtkm::rendering::Camera>& cameras,
                                std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& normals,
                                std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& albedo,
                                std::vector<vtkm::cont::ArrayHandle<vtkm::Float32>>& depth);
  double GetLastRenderMilliseconds() const { return LastRenderMs; }
  long long GetLastSegments() const { return LastSegments; }

  const int depthcount, samplecount;
  vtkm::cont::ArrayHandle<vtkm::Id>*MatIdx, *TexIdx;
  vtkm::cont::ArrayHandle<int> whichPDF;
  vtkm::cont::ArrayHandle<int> MatType, TexType;
  vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 3>> Tex;
  vtkm::rendering::pathtracing::QuadIntersector::ScatterRecord srecs;
  vtkm::rendering::pathtracing::QuadIntersector::HitRecord hrecs;
  vtkm::rendering::pathtracing::QuadIntersector::HitId hids;

private:
  struct InternalsType;
  std::shared_ptr<InternalsType> Internals;
  // The set-up every camera sweep shares: needs a canvas, validates every camera against it, uploads the scene
  // (buildBVH) and returns the view list of the C-ABI (10 floats per camera).
  std::vector<float> PrepareSweep(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                  const std::vector<vtkm::rendering::Camera>& cameras);
  void RenderViewsImpl(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                       const std::vector<vtkm::rendering::Camera>& cameras, unsigned int flags, void* out,
                       const std::vector<int>* checkpoints = nullptr, float* moment2 = nullptr);
  void RenderCellsImpl(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                       const vtkm::cont::Field& scalarField, const vtkm::rendering::Camera& camera);
  void UploadScene(const vtkm::cont::CoordinateSystem& coord, vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>& QuadIds,
                   vtkm::cont::ArrayHandle<vtkm::Id>& SphereIds, vtkm::cont::ArrayHandle<vtkm::Float32>& SphereRadii,
                   vtkm::cont::ArrayHandle<vtkm::Id>* matIdx, vtkm::cont::ArrayHandle<vtkm::Id>* texIdx);
  void IntersectImpl(vtkm::rendering::raytracing::Ray<vtkm::Float32>& rays, vtkm::cont::ArrayHandle<float>& tmin,
                     std::vector<unsigned char>& missed);
  [[noreturn]] static void FusedStage(const char* name);

  unsigned int RenderFlags = 0;
  float LensAperture = 0.f, LensFocus = 0.f;
  std::vector<int> Devices; // empty = the default device
  double LastRenderMs = 0.0;
  long long LastSegments = 0;
  vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>> light_box_pointids;
  vtkm::cont::ArrayHandle<vtkm::Id> light_box_indices, light_sphere_pointids, light_sphere_indices;
  vtkm::cont::ArrayHandle<vtkm::Int32> MatIdArray, TexIdArray;
  vtkm::rendering::pathtracing::QuadIntersector quadIntersector;
  vtkm::rendering::pathtracing::SphereIntersector sphereIntersector;
};

template <typename emittedType, typename attenType>
void MapperPathTracer::intersect(vtkm::rendering::raytracing::Ray<vtkm::Float32>& rays,
                                 vtkm::cont::ArrayHandle<float>& tmin, emittedType& emitted, attenType& attenuation,
                                 const vtkm::Id depth)
{
  std::vector<unsigned char> missed;
  IntersectImpl(rays, tmin, missed);
  const vtkm::Id n = rays.NumRays;
  for (vtkm::Id i = 0; i < n; ++i)
    if (missed[static_cast<size_t>(i)])
    { // SurfaceWorklets.h:98-111: depth-major planar layout [depth*N + i]
      attenuation.Set(i + n * depth, vtkm::Vec<vtkm::Float32, 3>(1.0f));
      emitted.Set(i + n * depth, vtkm::Vec<vtkm::Float32, 3>(0.0f));
    }
}

} // namespace rendering
} // namespace vtkm
#endif
