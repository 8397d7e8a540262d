// MapperPathTracer.cxx -- see MapperPathTracer.h.  Host-side marshalling only; every computation happens in
// libb2pt (sm_100a kernels) through the C-ABI.
#include "MapperPathTracer.h"
#include <cstring>

#include <cfloat>
#include <string>
#include <vector>

#include "b2pt_facade.h"

#include <algorithm>
#include "pathtracing/Camera.h"
#include "pathtracing/PathTracer.h"

namespace vtkm
{
namespace rendering
{

struct MapperPathTracer::InternalsType
{
  vtkm::rendering::CanvasRayTracer* Canvas = nullptr;
  vtkm::rendering::pathtracing::PathTracer Tracer;
  vtkm::rendering::pathtracing::Camera RayCamera;
  vtkm::rendering::raytracing::Ray<vtkm::Float32> Rays;
  bool CompositeBackground = true;
};

MapperPathTracer::MapperPathTracer(int sc, int dc, vtkm::cont::ArrayHandle<vtkm::Id>* matIdx,
                                   vtkm::cont::ArrayHandle<vtkm::Id>* texIdx, vtkm::cont::ArrayHandle<int>& matType,
                                   vtkm::cont::ArrayHandle<int>& texType,
                                   vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 3>>& tex)
  : depthcount(dc)
  , samplecount(sc)
  , MatIdx(matIdx)
  , TexIdx(texIdx)
  , MatType(matType)
  , TexType(texType)
  , Tex(tex)
  , Internals(new InternalsType)
{
  // The reference registers 27 named per-ray buffers here (MapperPathTracer.cxx:111-139).  They stay
  // addressable by name for API compatibility; the depth-layered ones are never materialised by the fused
  // kernels (per-path throughput lives in registers), so only their names and channel counts are kept.
  auto& rays = Internals->Rays;
  rays.EnableIntersectionData();
  for (const char* n : { "specular_Ox", "specular_Oy", "specular_Oz", "specular_Dx", "specular_Dy", "specular_Dz",
                         "specular_Ax", "specular_Ay", "specular_Az" })
    rays.AddBuffer(1, n);
  for (const char* n : { "attenuationX", "attenuationY", "attenuationZ", "emittedX", "emittedY", "emittedZ" })
    rays.AddBuffer(depthcount, n);
  for (const char* n : { "generated_dirX", "generated_dirY", "generated_dirZ", "sumtotlx", "sumtotly", "sumtotlz",
                         "sum_values" })
    rays.AddBuffer(1, n);
  rays.AddBuffer(depthcount, "alphaChannelAE");
  rays.AddBuffer(1, "alphaChannel");

  // hard-coded light lists of the reference (MapperPathTracer.cxx:141-148): the quad made of points 8..11
  // and the sphere centred at point 48
  const vtkm::Vec<vtkm::Id, 5> lightQuad(0, 8, 9, 10, 11);
  light_box_pointids = vtkm::cont::make_ArrayHandle(&lightQuad, 1, vtkm::CopyFlag::On);
  const vtkm::Id zero = 0, spherePoint = 4 * 12;
  light_box_indices = vtkm::cont::make_ArrayHandle(&zero, 1, vtkm::CopyFlag::On);
  light_sphere_pointids = vtkm::cont::make_ArrayHandle(&spherePoint, 1, vtkm::CopyFlag::On);
  light_sphere_indices = vtkm::cont::make_ArrayHandle(&zero, 1, vtkm::CopyFlag::On);
}

MapperPathTracer::~MapperPathTracer() {}

void MapperPathTracer::SetCanvas(vtkm::rendering::Canvas* canvas)
{
  if (canvas == nullptr)
  {
    Internals->Canvas = nullptr;
    return;
  }
  Internals->Canvas = dynamic_cast<CanvasRayTracer*>(canvas);
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("Ray Tracer: bad canvas type. Must be CanvasRayTracer");
  whichPDF.Allocate(canvas->GetWidth() * canvas->GetHeight());
}

vtkm::rendering::Canvas* MapperPathTracer::GetCanvas() const { return Internals->Canvas; }

MapperPathTracer::ExtractResult MapperPathTracer::extract(const vtkm::cont::DynamicCellSet& cellset) const
{
  const auto& cs = cellset.Cast<vtkm::cont::CellSetExplicit<>>();
  std::vector<vtkm::Id> sphereIds;
  std::vector<vtkm::Vec<vtkm::Id, 5>> quadIds;
  const vtkm::Id nCells = cs.GetNumberOfCells();
  for (vtkm::Id c = 0; c < nCells; ++c)
  {
    const vtkm::UInt8 shape = cs.Shapes.ReadPortal().Get(c);
    const vtkm::Id off = cs.Offsets.ReadPortal().Get(c);
    auto conn = cs.Connectivity.ReadPortal();
    if (shape == vtkm::CELL_SHAPE_VERTEX)
      sphereIds.push_back(conn.Get(off));
    else if (shape == vtkm::CELL_SHAPE_QUAD)
      quadIds.push_back(vtkm::Vec<vtkm::Id, 5>(c, conn.Get(off), conn.Get(off + 1), conn.Get(off + 2), conn.Get(off + 3)));
  }
  std::vector<vtkm::Float32> radii(sphereIds.size(), static_cast<vtkm::Float32>(90 / 555.0)); // :182
  return std::make_tuple(vtkm::cont::make_ArrayHandle(sphereIds), vtkm::cont::make_ArrayHandle(radii), cs.Offsets,
                         vtkm::cont::make_ArrayHandle(quadIds));
}

void MapperPathTracer::UploadScene(const vtkm::cont::CoordinateSystem& coord,
                                   vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>& QuadIds,
                                   vtkm::cont::ArrayHandle<vtkm::Id>& SphereIds,
                                   vtkm::cont::ArrayHandle<vtkm::Float32>& SphereRadii,
                                   vtkm::cont::ArrayHandle<vtkm::Id>* matIdx, vtkm::cont::ArrayHandle<vtkm::Id>* texIdx)
{
  const auto& pts = coord.GetPoints();
  const vtkm::Id nPts = pts.GetNumberOfValues(), nQ = QuadIds.GetNumberOfValues(), nS = SphereIds.GetNumberOfValues();
  if (matIdx[0].GetNumberOfValues() < nQ || texIdx[0].GetNumberOfValues() < nQ || matIdx[1].GetNumberOfValues() < nS ||
      texIdx[1].GetNumberOfValues() < nS || SphereRadii.GetNumberOfValues() < nS)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: material/texture index arrays shorter than the primitive lists");
  static_assert(sizeof(vtkm::Vec<vtkm::Float32, 3>) == 12 && sizeof(vtkm::Vec<vtkm::Id, 5>) == 40, "packed Vec");
  static_assert(sizeof(vtkm::Id) == sizeof(int64_t), "vtkm::Id is 64-bit");
  std::vector<float> lightR;
  for (vtkm::Id l = 0; l < light_sphere_pointids.GetNumberOfValues(); ++l)
    lightR.push_back(l < nS ? SphereRadii.ReadPortal().Get(l) : 0.f); // radii.Get(i), PdfWorklet.h:205
  const int nLightSph = nS > 0 ? static_cast<int>(light_sphere_pointids.GetNumberOfValues()) : 0;
  // every device of SetDevices gets the scene (replicated: a few KB for the Cornell box, < 100 MB for a million spheres)
  std::vector<int> devs = Devices;
  if (devs.empty())
    devs.push_back(-1);
  for (int dev : devs)
  {
    b2pt_ctx* ctx = b2pt_facade::Context(dev);
    b2pt_facade::Check(b2pt_set_scene(
      ctx, reinterpret_cast<const float*>(pts.GetStorage()), nPts, reinterpret_cast<const int64_t*>(QuadIds.GetStorage()),
      nQ, reinterpret_cast<const int64_t*>(SphereIds.GetStorage()), SphereRadii.GetStorage(), nS,
      reinterpret_cast<const int64_t*>(matIdx[0].GetStorage()), reinterpret_cast<const int64_t*>(texIdx[0].GetStorage()),
      reinterpret_cast<const int64_t*>(matIdx[1].GetStorage()), reinterpret_cast<const int64_t*>(texIdx[1].GetStorage()),
      MatType.GetStorage(), static_cast<int>(MatType.GetNumberOfValues()), TexType.GetStorage(),
      static_cast<int>(TexType.GetNumberOfValues()), reinterpret_cast<const float*>(Tex.GetStorage()),
      static_cast<int>(Tex.GetNumberOfValues()), reinterpret_cast<const int64_t*>(light_box_pointids.GetStorage()),
      static_cast<int>(light_box_pointids.GetNumberOfValues()),
      reinterpret_cast<const int64_t*>(light_sphere_pointids.GetStorage()), lightR.data(), nLightSph, /*lightables*/ 2,
      /*ref_idx, MapperPathTracer.cxx:467*/ 1.5f));
    b2pt_facade::Check(b2pt_build_bvh(ctx));
  }
}

void MapperPathTracer::buildBVH(const vtkm::cont::CoordinateSystem& coord,
                                vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Id, 5>>& QuadIds,
                                vtkm::cont::ArrayHandle<vtkm::Id>& SphereIds,
                                vtkm::cont::ArrayHandle<vtkm::Float32>& SphereRadii,
                                vtkm::cont::ArrayHandle<vtkm::Int32>& matIdArray,
                                vtkm::cont::ArrayHandle<vtkm::Int32>& texIdArray,
                                vtkm::cont::ArrayHandle<vtkm::Id>* matIdx, vtkm::cont::ArrayHandle<vtkm::Id>* texIdx)
{
  quadIntersector.SetData(coord, QuadIds, matIdx[0], texIdx[0], matIdArray, texIdArray);
  sphereIntersector.SetData(coord, SphereIds, SphereRadii, matIdx[1], texIdx[1], matIdArray, texIdArray);
  MatIdArray = matIdArray;
  TexIdArray = texIdArray;
  UploadScene(coord, QuadIds, SphereIds, SphereRadii, matIdx, texIdx);
}

void MapperPathTracer::IntersectImpl(vtkm::rendering::raytracing::Ray<vtkm::Float32>& rays,
                                     vtkm::cont::ArrayHandle<float>& tmin, std::vector<unsigned char>& missed)
{
  const vtkm::Id n = rays.NumRays;
  rays.EnableIntersectionData();
  if (tmin.GetNumberOfValues() != n)
    tmin.Allocate(n);
  for (vtkm::Id i = 0; i < n; ++i)
  { // MapperPathTracer.cxx:419-420
    rays.Distance.GetStorage()[i] = FLT_MAX;
    tmin.GetStorage()[i] = 0.001f;
  }
  std::vector<int32_t> prim(static_cast<size_t>(n)), mat(static_cast<size_t>(n)), texi(static_cast<size_t>(n));
  std::vector<float> rec(static_cast<size_t>(9 * n));
  b2pt_facade::Check(b2pt_intersect(b2pt_facade::Context(), n, rays.OriginX.GetStorage(), rays.OriginY.GetStorage(),
                                    rays.OriginZ.GetStorage(), rays.DirX.GetStorage(), rays.DirY.GetStorage(),
                                    rays.DirZ.GetStorage(), 0.001f, FLT_MAX, prim.data(), rec.data(), mat.data(),
                                    texi.data()));
  if (MatIdArray.GetNumberOfValues() != n)
    MatIdArray.Allocate(n);
  if (TexIdArray.GetNumberOfValues() != n)
    TexIdArray.Allocate(n);
  missed.assign(static_cast<size_t>(n), 0);
  vtkm::UInt8* status = rays.Status.GetStorage();
  float* out[9] = { rays.U.GetStorage(),       rays.V.GetStorage(),       rays.Distance.GetStorage(),
                    rays.NormalX.GetStorage(), rays.NormalY.GetStorage(), rays.NormalZ.GetStorage(),
                    rays.IntersectionX.GetStorage(), rays.IntersectionY.GetStorage(), rays.IntersectionZ.GetStorage() };
  for (vtkm::Id i = 0; i < n; ++i)
  {
    const bool alive = (status[i] & (1u << 3)) != 0;
    const bool hit = alive && prim[static_cast<size_t>(i)] >= 0;
    if (hit)
    {
      for (int f = 2; f < 9; ++f) // u,v are never consumed downstream and are left untouched
        out[f][i] = rec[static_cast<size_t>(f * n + i)];
      MatIdArray.GetStorage()[i] = mat[static_cast<size_t>(i)];
      TexIdArray.GetStorage()[i] = texi[static_cast<size_t>(i)];
    }
    else
    { // CollectIntersecttWorklet: clear the scatter bit of rays that did not hit
      status[i] = static_cast<vtkm::UInt8>(status[i] & ~(1u << 3));
      missed[static_cast<size_t>(i)] = 1;
    }
    status[i] = static_cast<vtkm::UInt8>(status[i] & ~(1u << 2));
  }
}

void MapperPathTracer::FusedStage(const char* name)
{
  throw vtkm::cont::ErrorBadValue(std::string("MapperPathTracer::") + name +
                                  " is fused into the per-bounce GPU kernel; use RenderCells");
}

void MapperPathTracer::RenderCellsImpl(const vtkm::cont::DynamicCellSet& cellset,
                                       const vtkm::cont::CoordinateSystem& coords, const vtkm::cont::Field&,
                                       const vtkm::rendering::Camera& camera)
{
  auto* canvas = Internals->Canvas;
  const vtkm::Id nx = canvas->GetWidth(), ny = canvas->GetHeight();
  auto tup = extract(cellset);
  auto SphereIds = std::get<0>(tup);
  auto SphereRadii = std::get<1>(tup);
  auto QuadIds = std::get<3>(tup);
  vtkm::cont::ArrayHandle<vtkm::Int32> matIdArray, texIdArray;
  matIdArray.Allocate(nx * ny);
  texIdArray.Allocate(nx * ny);
  buildBVH(coords, QuadIds, SphereIds, SphereRadii, matIdArray, texIdArray, MatIdx, TexIdx);

  const auto pos = camera.GetPosition(), at = camera.GetLookAt(), up = camera.GetViewUp();
  const float p[3] = { pos[0], pos[1], pos[2] }, a[3] = { at[0], at[1], at[2] }, u[3] = { up[0], up[1], up[2] };
  std::vector<int> devs = Devices;
  if (devs.empty())
    devs.push_back(-1);
  const int G = static_cast<int>(devs.size());
  std::vector<b2pt_ctx*> ctxs;
  for (int dev : devs)
    ctxs.push_back(b2pt_facade::Context(dev));
  // Device g renders the global samples [g*S/G, (g+1)*S/G) of every pixel.  The calls return once the work is queued
  // on the device's own stream, so the G GPUs render side by side; the sums are then added across the devices.
  for (int g = 0; g < G; ++g)
  {
    b2pt_ctx* ctx = ctxs[static_cast<size_t>(g)];
    b2pt_facade::Check(
      b2pt_set_camera(ctx, p, a, u, camera.GetFieldOfView(), static_cast<int>(nx), static_cast<int>(ny)));
    b2pt_facade::Check(b2pt_seed(ctx, 0)); // seeds[i] = i, MapperPathTracer.cxx:265-267
    b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
    const int begin = static_cast<int>(static_cast<long long>(samplecount) * g / G);
    const int end = static_cast<int>(static_cast<long long>(samplecount) * (g + 1) / G);
    b2pt_facade::Check(b2pt_clear_color(ctx)); // MapperPathTracer.cxx:222-223
    b2pt_facade::Check(b2pt_render_range(ctx, begin, end - begin, depthcount, RenderFlags));
  }
  if (G > 1)
    b2pt_facade::Check(b2pt_allreduce(ctxs.data(), G));
  b2pt_ctx* ctx = ctxs[0];
  auto& cols = canvas->GetColorBuffer();
  if (cols.GetNumberOfValues() != nx * ny)
    cols.Allocate(nx * ny);
  static_assert(sizeof(vtkm::Vec<vtkm::Float32, 4>) == 16, "packed Vec4");
  b2pt_facade::Check(b2pt_read_color(ctx, reinterpret_cast<float*>(cols.GetStorage())));
  b2pt_stats st;
  LastRenderMs = 0.0;
  LastSegments = 0;
  for (b2pt_ctx* c : ctxs)
  {
    b2pt_facade::Check(b2pt_get_stats(c, &st));
    LastRenderMs = std::max(LastRenderMs, st.renderMs);
    LastSegments += st.segments;
  }
}

void MapperPathTracer::RenderCells(const vtkm::cont::DynamicCellSet& cellset, const vtkm::cont::CoordinateSystem& coords,
                                   const vtkm::cont::Field& scalarField, const vtkm::cont::ColorTable&,
                                   const vtkm::rendering::Camera& camera, const vtkm::Range&)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  Internals->RayCamera.SetParameters(camera, *Internals->Canvas); // validates like the reference (:372)
  RenderCellsImpl(cellset, coords, scalarField, camera);
}

void MapperPathTracer::RenderDirectBuffers(const vtkm::cont::DynamicCellSet& cellset,
                                           const vtkm::cont::CoordinateSystem& coords,
                                           const vtkm::rendering::Camera& camera,
                                           vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& normals,
                                           vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& albedo,
                                           vtkm::cont::ArrayHandle<vtkm::Float32>& depth)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  auto* canvas = Internals->Canvas;
  const vtkm::Id nx = canvas->GetWidth(), ny = canvas->GetHeight();
  Internals->RayCamera.SetParameters(camera, *canvas);
  auto tup = extract(cellset);
  auto SphereIds = std::get<0>(tup);
  auto SphereRadii = std::get<1>(tup);
  auto QuadIds = std::get<3>(tup);
  vtkm::cont::ArrayHandle<vtkm::Int32> matIdArray, texIdArray;
  matIdArray.Allocate(nx * ny);
  texIdArray.Allocate(nx * ny);
  buildBVH(coords, QuadIds, SphereIds, SphereRadii, matIdArray, texIdArray, MatIdx, TexIdx);
  b2pt_ctx* ctx = b2pt_facade::Context(Devices.empty() ? -1 : Devices[0]);
  const auto pos = camera.GetPosition(), at = camera.GetLookAt(), up = camera.GetViewUp();
  const float p[3] = { pos[0], pos[1], pos[2] }, a[3] = { at[0], at[1], at[2] }, u[3] = { up[0], up[1], up[2] };
  b2pt_facade::Check(
    b2pt_set_camera(ctx, p, a, u, camera.GetFieldOfView(), static_cast<int>(nx), static_cast<int>(ny)));
  normals.Allocate(nx * ny);
  albedo.Allocate(nx * ny);
  depth.Allocate(nx * ny);
  b2pt_facade::Check(b2pt_render_direct(ctx, reinterpret_cast<float*>(normals.GetStorage()),
                                        reinterpret_cast<float*>(albedo.GetStorage()), depth.GetStorage(), nullptr));
}

// b2pt_render_views / b2pt_render_direct_views view list: pos[3], lookAt[3], up[3], fovDeg per camera
static std::vector<float> packViews(const std::vector<vtkm::rendering::Camera>& cameras)
{
  std::vector<float> views(cameras.size() * 10);
  for (size_t v = 0; v < cameras.size(); ++v)
  {
    const auto pos = cameras[v].GetPosition(), at = cameras[v].GetLookAt(), up = cameras[v].GetViewUp();
    float* p = &views[10 * v];
    for (int k = 0; k < 3; ++k)
      p[k] = pos[k], p[3 + k] = at[k], p[6 + k] = up[k];
    p[9] = cameras[v].GetFieldOfView();
  }
  return views;
}

// A sweep's checkpoint list: strictly increasing counts >= 1 that end with the sample count.
static void CheckCheckpoints(const std::vector<int>& checkpoints, int samplecount)
{
  if (checkpoints.empty() || checkpoints.back() != samplecount)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: the checkpoint list must end with the sample count");
  for (size_t k = 0; k < checkpoints.size(); ++k)
    if (checkpoints[k] < 1 || (k > 0 && checkpoints[k] <= checkpoints[k - 1]))
      throw vtkm::cont::ErrorBadValue("MapperPathTracer: checkpoints must be >= 1 and strictly increasing");
}

std::vector<float> MapperPathTracer::PrepareSweep(const vtkm::cont::DynamicCellSet& cellset,
                                                  const vtkm::cont::CoordinateSystem& coords,
                                                  const std::vector<vtkm::rendering::Camera>& cameras)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  auto* canvas = Internals->Canvas;
  const vtkm::Id nx = canvas->GetWidth(), ny = canvas->GetHeight();
  for (const auto& camera : cameras)
    Internals->RayCamera.SetParameters(camera, *canvas); // validates every view like the reference (:372)
  auto tup = extract(cellset);
  auto SphereIds = std::get<0>(tup);
  auto SphereRadii = std::get<1>(tup);
  auto QuadIds = std::get<3>(tup);
  vtkm::cont::ArrayHandle<vtkm::Int32> matIdArray, texIdArray;
  matIdArray.Allocate(nx * ny);
  texIdArray.Allocate(nx * ny);
  buildBVH(coords, QuadIds, SphereIds, SphereRadii, matIdArray, texIdArray, MatIdx, TexIdx);
  return packViews(cameras);
}

void MapperPathTracer::RenderDirectBuffersViews(const vtkm::cont::DynamicCellSet& cellset,
                                                const vtkm::cont::CoordinateSystem& coords,
                                                const std::vector<vtkm::rendering::Camera>& cameras,
                                                std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& normals,
                                                std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& albedo,
                                                std::vector<vtkm::cont::ArrayHandle<vtkm::Float32>>& depth)
{
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  const size_t n = static_cast<size_t>(nx * ny), V = cameras.size();
  std::vector<float> nrm(V * n * 4), alb(V * n * 4), dep(V * n);
  b2pt_ctx* ctx = b2pt_facade::Context(Devices.empty() ? -1 : Devices[0]);
  b2pt_facade::Check(b2pt_render_direct_views(ctx, static_cast<int>(V), views.data(), static_cast<int>(nx),
                                              static_cast<int>(ny), nrm.data(), alb.data(), dep.data(), nullptr));
  normals.resize(V);
  albedo.resize(V);
  depth.resize(V);
  for (size_t v = 0; v < V; ++v)
  {
    normals[v].Allocate(static_cast<vtkm::Id>(n));
    albedo[v].Allocate(static_cast<vtkm::Id>(n));
    depth[v].Allocate(static_cast<vtkm::Id>(n));
    std::memcpy(static_cast<void*>(normals[v].GetStorage()), &nrm[v * n * 4], sizeof(float) * 4 * n);
    std::memcpy(static_cast<void*>(albedo[v].GetStorage()), &alb[v * n * 4], sizeof(float) * 4 * n);
    std::memcpy(depth[v].GetStorage(), &dep[v * n], sizeof(float) * n);
  }
}

void MapperPathTracer::RenderViewsImpl(const vtkm::cont::DynamicCellSet& cellset,
                                       const vtkm::cont::CoordinateSystem& coords,
                                       const std::vector<vtkm::rendering::Camera>& cameras, unsigned int flags,
                                       void* out, const std::vector<int>* checkpoints, float* moment2)
{
  std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  b2pt_ctx* ctx = b2pt_facade::Context();
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // seeds[i] = i, MapperPathTracer.cxx:265-267
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  if (checkpoints)
    b2pt_facade::Check(b2pt_render_views_checkpoints(
      ctx, static_cast<int>(cameras.size()), views.data(), static_cast<int>(nx), static_cast<int>(ny),
      static_cast<int>(checkpoints->size()), checkpoints->data(), depthcount, RenderFlags | flags, out, moment2));
  else
    b2pt_facade::Check(b2pt_render_views(ctx, static_cast<int>(cameras.size()), views.data(), static_cast<int>(nx),
                                         static_cast<int>(ny), samplecount, depthcount, RenderFlags | flags, out));
  b2pt_stats st;
  b2pt_facade::Check(b2pt_get_stats(ctx, &st));
  LastRenderMs = st.renderMs;
  LastSegments = st.segments;
}

void MapperPathTracer::RenderCellsViews(const vtkm::cont::DynamicCellSet& cellset,
                                        const vtkm::cont::CoordinateSystem& coords,
                                        const std::vector<vtkm::rendering::Camera>& cameras,
                                        std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>>& colors)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  const size_t n = static_cast<size_t>(Internals->Canvas->GetWidth()) * Internals->Canvas->GetHeight();
  std::vector<float> rgba(cameras.size() * n * 4);
  RenderViewsImpl(cellset, coords, cameras, 0, rgba.data());
  colors.resize(cameras.size());
  for (size_t v = 0; v < cameras.size(); ++v)
  {
    colors[v].Allocate(static_cast<vtkm::Id>(n));
    std::memcpy(colors[v].GetStorage(), &rgba[v * n * 4], sizeof(float) * 4 * n);
  }
}

void MapperPathTracer::RenderCellsViewsPnm(const vtkm::cont::DynamicCellSet& cellset,
                                           const vtkm::cont::CoordinateSystem& coords,
                                           const std::vector<vtkm::rendering::Camera>& cameras,
                                           std::vector<unsigned short>& pnm)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  static_assert(sizeof(unsigned short) == 2, "16-bit PNM integers");
  const size_t n = static_cast<size_t>(Internals->Canvas->GetWidth()) * Internals->Canvas->GetHeight();
  pnm.assign(cameras.size() * n * 3, 0);
  RenderViewsImpl(cellset, coords, cameras, B2PT_FLAG_VIEWS_PNM16, pnm.data());
}

void MapperPathTracer::RenderCellsViewsCheckpointsPnm(const vtkm::cont::DynamicCellSet& cellset,
                                                      const vtkm::cont::CoordinateSystem& coords,
                                                      const std::vector<vtkm::rendering::Camera>& cameras,
                                                      const std::vector<int>& checkpoints,
                                                      std::vector<unsigned short>& pnm)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(checkpoints, samplecount);
  const size_t n = static_cast<size_t>(Internals->Canvas->GetWidth()) * Internals->Canvas->GetHeight();
  pnm.assign(checkpoints.size() * cameras.size() * n * 3, 0);
  RenderViewsImpl(cellset, coords, cameras, B2PT_FLAG_VIEWS_PNM16, pnm.data(), &checkpoints);
}

void MapperPathTracer::RenderCellsViewsFeatures(const vtkm::cont::DynamicCellSet& cellset,
                                                const vtkm::cont::CoordinateSystem& coords,
                                                const std::vector<vtkm::rendering::Camera>& cameras,
                                                const std::vector<int>& checkpoints, std::vector<float>& albedo,
                                                std::vector<float>& normalDepth)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(checkpoints, samplecount);
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  const size_t n = checkpoints.size() * cameras.size() * static_cast<size_t>(nx * ny) * 4;
  albedo.assign(n, 0.f);
  normalDepth.assign(n, 0.f);
  b2pt_ctx* ctx = b2pt_facade::Context(Devices.empty() ? -1 : Devices[0]);
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // the streams RenderCellsViews* render with
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  b2pt_facade::Check(b2pt_render_views_features(ctx, static_cast<int>(cameras.size()), views.data(),
                                                static_cast<int>(nx), static_cast<int>(ny),
                                                static_cast<int>(checkpoints.size()), checkpoints.data(),
                                                RenderFlags & B2PT_BUILD_FLAGS, albedo.data(), normalDepth.data()));
}

void MapperPathTracer::RenderCellsViewsMotion(const vtkm::cont::DynamicCellSet& cellset,
                                              const vtkm::cont::CoordinateSystem& coords,
                                              const std::vector<vtkm::rendering::Camera>& cameras,
                                              const std::vector<vtkm::rendering::Camera>& prevCameras,
                                              const std::vector<int>& checkpoints, std::vector<float>& motion)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  if (prevCameras.size() != cameras.size())
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: one previous camera per camera");
  CheckCheckpoints(checkpoints, samplecount);
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras), prevViews = packViews(prevCameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  motion.assign(checkpoints.size() * cameras.size() * static_cast<size_t>(nx * ny) * 4, 0.f);
  b2pt_ctx* ctx = b2pt_facade::Context(Devices.empty() ? -1 : Devices[0]);
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // the streams RenderCellsViews* render with
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  b2pt_facade::Check(b2pt_render_views_motion(ctx, static_cast<int>(cameras.size()), views.data(), prevViews.data(),
                                              static_cast<int>(nx), static_cast<int>(ny),
                                              static_cast<int>(checkpoints.size()), checkpoints.data(),
                                              RenderFlags & B2PT_BUILD_FLAGS, motion.data()));
}

void MapperPathTracer::RenderCellsViewsDenoisedPnm(const vtkm::cont::DynamicCellSet& cellset,
                                                   const vtkm::cont::CoordinateSystem& coords,
                                                   const std::vector<vtkm::rendering::Camera>& cameras,
                                                   const std::vector<int>& checkpoints, std::vector<unsigned short>& pnm,
                                                   std::vector<unsigned short>& denoisedPnm)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(checkpoints, samplecount);
  std::vector<float> color, moment2, albedo, normalDepth;
  const size_t n = static_cast<size_t>(Internals->Canvas->GetWidth()) * Internals->Canvas->GetHeight();
  const size_t n4 = checkpoints.size() * cameras.size() * n * 4;
  color.assign(n4, 0.f);
  moment2.assign(n4, 0.f);
  RenderViewsImpl(cellset, coords, cameras, 0, color.data(), &checkpoints, moment2.data());
  RenderCellsViewsFeatures(cellset, coords, cameras, checkpoints, albedo, normalDepth);
  b2pt_ctx* ctx = b2pt_facade::Context();
  const int V = static_cast<int>(cameras.size()), K = static_cast<int>(checkpoints.size());
  const int nx = static_cast<int>(Internals->Canvas->GetWidth()), ny = static_cast<int>(Internals->Canvas->GetHeight());
  pnm.assign(n4 / 4 * 3, 0);
  denoisedPnm.assign(n4 / 4 * 3, 0);
  b2pt_denoise_params unfiltered;
  b2pt_denoise_defaults(&unfiltered);
  unfiltered.levels = 0;
  b2pt_facade::Check(b2pt_denoise_views(ctx, V, nx, ny, K, checkpoints.data(), color.data(), moment2.data(),
                                        albedo.data(), normalDepth.data(), &unfiltered, B2PT_FLAG_VIEWS_PNM16,
                                        pnm.data()));
  b2pt_facade::Check(b2pt_denoise_views(ctx, V, nx, ny, K, checkpoints.data(), color.data(), moment2.data(),
                                        albedo.data(), normalDepth.data(), nullptr, B2PT_FLAG_VIEWS_PNM16,
                                        denoisedPnm.data()));
}

void MapperPathTracer::RenderCellsViewsTemporalPnm(const vtkm::cont::DynamicCellSet& cellset,
                                                   const vtkm::cont::CoordinateSystem& coords,
                                                   const std::vector<vtkm::rendering::Camera>& cameras,
                                                   const std::vector<int>& checkpoints,
                                                   std::vector<unsigned short>& temporalPnm)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(checkpoints, samplecount);
  if (cameras.empty())
  {
    temporalPnm.clear();
    return;
  }
  // one call: the render, its guides, the motion of every view towards the one before it in sweep order, and the
  // temporal denoiser, with nothing but the result copied to the host
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const int nx = static_cast<int>(Internals->Canvas->GetWidth()), ny = static_cast<int>(Internals->Canvas->GetHeight());
  temporalPnm.assign(checkpoints.size() * cameras.size() * static_cast<size_t>(nx) * ny * 3, 0);
  b2pt_ctx* ctx = b2pt_facade::Context();
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // the streams RenderCellsViews* render with
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  b2pt_facade::Check(b2pt_render_views_temporal_denoised(
    ctx, static_cast<int>(cameras.size()), views.data(), nx, ny, static_cast<int>(checkpoints.size()),
    checkpoints.data(), depthcount, nullptr, nullptr, RenderFlags | B2PT_FLAG_VIEWS_PNM16, temporalPnm.data(), nullptr,
    nullptr, nullptr, nullptr, nullptr, nullptr));
  b2pt_stats st;
  b2pt_facade::Check(b2pt_get_stats(ctx, &st));
  LastRenderMs = st.renderMs;
  LastSegments = st.segments;
}

void MapperPathTracer::RenderCellsViewsAdaptivePnm(const vtkm::cont::DynamicCellSet& cellset,
                                                   const vtkm::cont::CoordinateSystem& coords,
                                                   const std::vector<vtkm::rendering::Camera>& cameras,
                                                   const std::vector<int>& rounds, float threshold,
                                                   std::vector<unsigned short>& pnm, std::vector<int>& counts)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(rounds, samplecount);
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  const size_t n = cameras.size() * static_cast<size_t>(nx * ny);
  pnm.assign(n * 3, 0);
  counts.assign(n, 0);
  b2pt_ctx* ctx = b2pt_facade::Context();
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // the streams RenderCellsViews* render with
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  b2pt_adaptive_params params;
  b2pt_adaptive_defaults(&params);
  params.threshold = threshold;
  b2pt_facade::Check(b2pt_render_views_adaptive(ctx, static_cast<int>(cameras.size()), views.data(),
                                                static_cast<int>(nx), static_cast<int>(ny),
                                                static_cast<int>(rounds.size()), rounds.data(), depthcount, &params,
                                                RenderFlags | B2PT_FLAG_VIEWS_PNM16, pnm.data(), nullptr,
                                                counts.data(), nullptr));
  b2pt_stats st;
  b2pt_facade::Check(b2pt_get_stats(ctx, &st));
  LastRenderMs = st.renderMs;
  LastSegments = st.segments;
}

void MapperPathTracer::RenderCellsViewsAdaptiveDenoisedPnm(const vtkm::cont::DynamicCellSet& cellset,
                                                           const vtkm::cont::CoordinateSystem& coords,
                                                           const std::vector<vtkm::rendering::Camera>& cameras,
                                                           const std::vector<int>& rounds, float threshold,
                                                           std::vector<unsigned short>& pnm, std::vector<int>& counts,
                                                           std::vector<unsigned short>& denoisedPnm)
{
  if (Internals->Canvas == nullptr)
    throw vtkm::cont::ErrorBadValue("MapperPathTracer: no canvas set");
  CheckCheckpoints(rounds, samplecount);
  const std::vector<float> views = PrepareSweep(cellset, coords, cameras);
  const vtkm::Id nx = Internals->Canvas->GetWidth(), ny = Internals->Canvas->GetHeight();
  const size_t n = cameras.size() * static_cast<size_t>(nx * ny);
  pnm.assign(n * 3, 0);
  counts.assign(n, 0);
  denoisedPnm.assign(n * 3, 0);
  b2pt_ctx* ctx = b2pt_facade::Context();
  b2pt_facade::Check(b2pt_seed(ctx, 0)); // the streams RenderCellsViews* render with
  b2pt_facade::Check(b2pt_set_lens(ctx, LensAperture, LensFocus));
  b2pt_adaptive_params params;
  b2pt_adaptive_defaults(&params);
  params.threshold = threshold;
  b2pt_facade::Check(b2pt_render_views_adaptive_denoised(
    ctx, static_cast<int>(cameras.size()), views.data(), static_cast<int>(nx), static_cast<int>(ny),
    static_cast<int>(rounds.size()), rounds.data(), depthcount, &params, nullptr, RenderFlags | B2PT_FLAG_VIEWS_PNM16,
    pnm.data(), counts.data(), nullptr, nullptr, denoisedPnm.data()));
  b2pt_stats st;
  b2pt_facade::Check(b2pt_get_stats(ctx, &st));
  LastRenderMs = st.renderMs;
  LastSegments = st.segments;
}

void MapperPathTracer::SetCompositeBackground(bool on) { Internals->CompositeBackground = on; }

void MapperPathTracer::StartScene()
{
  auto& rays = Internals->Rays;
  vtkm::UInt8* s = rays.Status.GetStorage();
  for (vtkm::Id i = 0; i < rays.Status.GetNumberOfValues(); ++i)
    s[i] = static_cast<vtkm::UInt8>(1u << 3);
}

void MapperPathTracer::EndScene() {}

vtkm::rendering::Mapper* MapperPathTracer::NewCopy() const { return new vtkm::rendering::MapperPathTracer(*this); }

} // namespace rendering
} // namespace vtkm
