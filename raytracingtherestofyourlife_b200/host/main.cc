// main.cc -- command-line driver with the reference's flags (main.cc:54-113) for the path-traced image:
//   ./CornellBox_b2pt -x 128 -y 128 -samplecount 10 -raydepth 5
// Builds the Cornell box, renders it through MapperPathTracer (GPU), normalises with the reference's
// NormalizeFunctor semantics and writes output.pnm (ASCII P3, bottom row first) like main.cc:361-384.
// -hemisphere [-phicount P -thetacount T] sweeps the camera over the reference's hemisphere of view points
// (generateHemisphere, main.cc:504-561): one path-traced image per view, named output-<phi>-<theta>.pnm as the
// reference's generate() names them (main.cc:386-429).  Every view is an independent render through the same mapper;
// scene tables and trace structures stay resident on the GPU between views.
// -fibonacci [-viewcount N -viewseed R] is the reference's other sweep, fibonacciHemisphere (main.cc:430-503; its call
// at main.cc:612 is commented out, N = 10000 there): the points of an N-point Fibonacci lattice on the unit sphere
// around the box centre that lie on the camera's side (z < 0), rotated by R steps (the reference draws R = rand() % N
// from an unseeded rand(); here it is an option, default 0); images are named output-0.0000-<i>.0000.pnm like
// generate(cam, ..., 0, i) names them.
// -direct writes the G-buffers of generate()'s direct branch (main.cc:402-422) instead of the path-traced image:
// normals.pnm, albedo.pnm and depth.pnm for the default view, and with -hemisphere or -fibonacci, for every view point,
// normals-<phi>-<theta>.pnm, albedo-<phi>-<theta>.pnm and depth-<phi>-<theta>.pnm (phi and theta formatted as in the
// path-traced names; the Fibonacci sweep uses phi = 0, theta = i).  All views of a sweep are rendered in one call.
// The reference's own file names for the swept G-buffers are not restated here: this rule is the driver's.
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <sstream>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "CornellBox.h"
#include "MapperPathTracer.h"
#include "b2pt_facade.h"

namespace
{

struct Options
{
  int x = 128, y = 128, samples = 10, depth = 5; // reference defaults, main.cc:56-62
  std::string out = "output";
  bool stats = false;
  bool hemi = false;
  bool direct = false;
  bool fibonacci = false;
  int viewCount = 10000, viewSeed = 0; // main.cc:612 / :468
  int phiCount = 15, thetaCount = 15;  // main.cc:59-60
};

Options parse(int argc, char** argv)
{
  Options o;
  for (int i = 1; i < argc; ++i)
  {
    auto next = [&](int& dst) {
      if (i + 1 < argc)
        dst = std::atoi(argv[++i]);
    };
    if (!std::strcmp(argv[i], "-x"))
      next(o.x);
    else if (!std::strcmp(argv[i], "-y"))
      next(o.y);
    else if (!std::strcmp(argv[i], "-samplecount"))
      next(o.samples);
    else if (!std::strcmp(argv[i], "-raydepth"))
      next(o.depth);
    else if (!std::strcmp(argv[i], "-o") && i + 1 < argc)
      o.out = argv[++i];
    else if (!std::strcmp(argv[i], "-stats"))
      o.stats = true;
    else if (!std::strcmp(argv[i], "-hemisphere"))
      o.hemi = true;
    else if (!std::strcmp(argv[i], "-phicount"))
      next(o.phiCount);
    else if (!std::strcmp(argv[i], "-thetacount"))
      next(o.thetaCount);
    else if (!std::strcmp(argv[i], "-direct"))
      o.direct = true;
    else if (!std::strcmp(argv[i], "-fibonacci"))
      o.fibonacci = true;
    else if (!std::strcmp(argv[i], "-viewcount"))
      next(o.viewCount);
    else if (!std::strcmp(argv[i], "-viewseed"))
      next(o.viewSeed);
  }
  return o;
}

// NormalizeFunctor (main.cc:253-287): sqrt(de_nan(sum) / samplecount), alpha through the same sqrt
void normalizeColors(vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& colors, int samplecount)
{
  auto cols = colors.WritePortal();
  const float sc = static_cast<float>(samplecount);
  for (vtkm::Id i = 0; i < cols.GetNumberOfValues(); ++i)
  {
    auto c = cols.Get(i);
    for (int k = 0; k < 3; ++k)
      if (!(c[k] == c[k]))
        c[k] = 0;
    for (int k = 0; k < 4; ++k)
      c[k] = std::sqrt(c[k] / sc);
    cols.Set(i, c);
  }
}

// the reference's runPath (main.cc:289-323): this body is what a reference user already has
void runPath(CornellBox& cb, int samplecount, int depthcount, vtkm::rendering::Canvas& canvas,
             vtkm::rendering::Camera& cam, bool stats)
{
  vtkm::rendering::MapperPathTracer mapper(samplecount, depthcount, cb.matIdx, cb.texIdx, cb.matType, cb.texType,
                                           cb.tex);
  mapper.SetCanvas(&canvas);
  vtkm::cont::Field field;
  vtkm::cont::ColorTable ct;
  vtkm::Range sr;
  mapper.RenderCells(cb.ds.GetCellSet(), cb.coord, field, ct, cam, sr);
  if (stats)
    std::cout << " GPU render ms = " << mapper.GetLastRenderMilliseconds()
              << "  path samples/s = " << double(canvas.GetWidth()) * canvas.GetHeight() * samplecount /
        (mapper.GetLastRenderMilliseconds() * 1e-3)
              << "  segments = " << mapper.GetLastSegments() << std::endl;
  normalizeColors(canvas.GetColorBuffer(), samplecount);
}

void savePnm(const std::string& stem, int nx, int ny, const vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>& colors)
{
  std::ofstream fs(stem + ".pnm");
  if (!fs)
  {
    std::cout << "Couldn't save pnm." << std::endl;
    return;
  }
  fs << "P3\n" << nx << " " << ny << " 255" << std::endl;
  auto cols = colors.ReadPortal();
  for (vtkm::Id i = 0; i < cols.GetNumberOfValues(); ++i)
  {
    auto col = cols.Get(i);
    if ((col[0] != col[0]) || (col[1] != col[1]) || (col[2] != col[2]))
      col = 0.0f;
    fs << int(255.99 * col[0]) << " " << int(255.99 * col[1]) << " " << int(255.99 * col[2]) << std::endl;
  }
}

// save() for a scalar image (main.cc:343-359, the depth buffer): de_nan, sqrt, one value on three channels
void savePnmScalar(const std::string& stem, int nx, int ny, const vtkm::cont::ArrayHandle<vtkm::Float32>& values)
{
  std::ofstream fs(stem + ".pnm");
  if (!fs)
  {
    std::cout << "Couldn't save pnm." << std::endl;
    return;
  }
  fs << "P3\n" << nx << " " << ny << " 255" << std::endl;
  auto v = values.ReadPortal();
  for (vtkm::Id i = 0; i < v.GetNumberOfValues(); ++i)
  {
    float col = v.Get(i);
    if (col != col)
      col = 0.f;
    col = std::sqrt(col);
    const int g = int(255.99 * col);
    fs << g << " " << g << " " << g << std::endl;
  }
}

// the G-buffer half of generate() with direct = true (main.cc:402-422): "normals", "albedo" and "depth" images of the
// view.  The "direct" colour image needs VTK-m's stock Phong shader and colour table and is not produced.
void runDirect(CornellBox& cb, const Options& o, vtkm::rendering::Canvas& canvas, vtkm::rendering::Camera& cam)
{
  vtkm::rendering::MapperPathTracer mapper(o.samples, o.depth, cb.matIdx, cb.texIdx, cb.matType, cb.texType, cb.tex);
  mapper.SetCanvas(&canvas);
  vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>> normals, albedo;
  vtkm::cont::ArrayHandle<vtkm::Float32> depth;
  mapper.RenderDirectBuffers(cb.ds.GetCellSet(), cb.coord, cam, normals, albedo, depth);
  savePnm("normals", o.x, o.y, normals);
  savePnm("albedo", o.x, o.y, albedo);
  savePnmScalar("depth", o.x, o.y, depth);
  std::cout << " wrote normals.pnm albedo.pnm depth.pnm (direct.pnm, the stock Phong image, is out of scope)" << std::endl;
}

// The same file from the integers packed on the GPU (RenderCellsViewsPnm): "r g b\n" per pixel, formatted into one
// buffer and written once.
void savePnm16(const std::string& stem, int nx, int ny, const unsigned short* rgb)
{
  std::ofstream fs(stem + ".pnm", std::ios::binary);
  if (!fs)
  {
    std::cout << "Couldn't save pnm." << std::endl;
    return;
  }
  std::string buf = "P3\n" + std::to_string(nx) + " " + std::to_string(ny) + " 255\n";
  const size_t n = static_cast<size_t>(nx) * ny;
  buf.reserve(buf.size() + n * 18);
  char tmp[8];
  for (size_t i = 0; i < 3 * n; ++i)
  {
    unsigned v = rgb[i];
    int len = 0;
    do
    {
      tmp[len++] = static_cast<char>('0' + v % 10);
      v /= 10;
    } while (v);
    while (len)
      buf.push_back(tmp[--len]);
    buf.push_back(i % 3 == 2 ? '\n' : ' ');
  }
  fs.write(buf.data(), static_cast<std::streamsize>(buf.size()));
}

std::string viewName(const std::string& stem, float phi, float theta)
{ // generate(): "output-" << fixed << setw(4) << setprecision(4) << phi << "-" << theta
  std::stringstream name;
  name << stem << "-" << std::fixed << std::setw(4) << std::setprecision(4) << phi << "-";
  name << std::fixed << std::setw(4) << std::setprecision(4) << theta;
  return name.str();
}

using ViewAngles = std::vector<std::pair<float, float>>; // (phi, theta) of every view point, for the file names

// generate() for a list of view points (main.cc:386-429, direct branch): ONE call renders the G-buffers of every
// view; each view's three images are written with save()'s arithmetic.
int renderDirectViews(CornellBox& cb, const Options& o, const std::vector<vtkm::rendering::Camera>& cameras,
                      const ViewAngles& angles)
{
  if (cameras.empty())
    return 0;
  vtkm::rendering::CanvasRayTracer canvas(o.x, o.y);
  vtkm::rendering::MapperPathTracer mapper(o.samples, o.depth, cb.matIdx, cb.texIdx, cb.matType, cb.texType, cb.tex);
  mapper.SetCanvas(&canvas);
  std::vector<vtkm::cont::ArrayHandle<vtkm::Vec<vtkm::Float32, 4>>> normals, albedo;
  std::vector<vtkm::cont::ArrayHandle<vtkm::Float32>> depth;
  mapper.RenderDirectBuffersViews(cb.ds.GetCellSet(), cb.coord, cameras, normals, albedo, depth);
  for (size_t v = 0; v < cameras.size(); ++v)
  {
    savePnm(viewName("normals", angles[v].first, angles[v].second), o.x, o.y, normals[v]);
    savePnm(viewName("albedo", angles[v].first, angles[v].second), o.x, o.y, albedo[v]);
    savePnmScalar(viewName("depth", angles[v].first, angles[v].second), o.x, o.y, depth[v]);
  }
  return static_cast<int>(cameras.size());
}

// generate() for a list of view points (main.cc:386-429, path-traced branch): the reference renders and saves one
// view per call; here ONE call renders them all (small canvases share GPU launches across views), NormalizeFunctor and
// the integer conversion of save() (main.cc:253-287, 325-384) run on the GPU.
int renderViews(CornellBox& cb, const Options& o, const std::vector<vtkm::rendering::Camera>& cameras,
                const ViewAngles& angles)
{
  if (cameras.empty())
    return 0;
  vtkm::rendering::CanvasRayTracer canvas(o.x, o.y);
  vtkm::rendering::MapperPathTracer mapper(o.samples, o.depth, cb.matIdx, cb.texIdx, cb.matType, cb.texType, cb.tex);
  mapper.SetCanvas(&canvas);
  std::vector<unsigned short> pnm;
  mapper.RenderCellsViewsPnm(cb.ds.GetCellSet(), cb.coord, cameras, pnm);
  if (o.stats)
    std::cout << " GPU render ms = " << mapper.GetLastRenderMilliseconds() << " for " << cameras.size() << " views"
              << "  path samples/s = " << double(o.x) * o.y * o.samples * double(cameras.size()) /
        (mapper.GetLastRenderMilliseconds() * 1e-3)
              << "  segments = " << mapper.GetLastSegments() << std::endl;
  for (size_t v = 0; v < cameras.size(); ++v)
    savePnm16(viewName(o.out, angles[v].first, angles[v].second), o.x, o.y,
              &pnm[v * static_cast<size_t>(o.x) * o.y * 3]);
  return static_cast<int>(cameras.size());
}

vtkm::rendering::Camera sweepCamera()
{ // main.cc:463-467 / :516-521
  vtkm::rendering::Camera cam;
  cam.SetClippingRange(01.f, 5.f);
  cam.SetPosition(vec3(278 / 555.0, 278 / 555.0, -800 / 555.0));
  cam.SetFieldOfView(40.f);
  cam.SetViewUp(vec3(0, 1, 0));
  cam.SetLookAt(vec3(278 / 555.0, 278 / 555.0, 278 / 555.0));
  return cam;
}

// the reference's generateHemisphere (main.cc:504-561), path-traced or -direct: view points on a sphere of
// radius 1078/555 around the box centre, phi in [0,1) in phiCount steps, theta in [0,2pi) in thetaCount steps
int generateHemisphere(CornellBox& cb, const Options& o)
{
  vtkm::rendering::Camera cam = sweepCamera();
  const float phiBegin = 0.0f, phiEnd = 1.0f, thetaBegin = 0.f;
  const float thetaEnd = static_cast<float>(2 * 3.14159265358979323846);
  const float rTheta = thetaEnd / static_cast<float>(o.thetaCount);
  const float rPhi = (phiEnd - phiBegin) / float(o.phiCount);
  const float r = static_cast<float>(-1078 / 555.0);
  std::vector<vtkm::rendering::Camera> cameras;
  ViewAngles angles;
  for (float phi = phiBegin; phi < (phiEnd - 0.5 * rPhi); phi += rPhi)
    for (float theta = thetaBegin; theta < thetaEnd; theta += rTheta)
    {
      const auto x = r * std::cos(theta) * std::sin(phi);
      const auto y = r * std::sin(theta) * std::sin(phi);
      const auto z = r * std::cos(phi);
      cam.SetPosition(vec3(x + 278 / 555.0, y + 278 / 555.0, z + 278 / 555.0));
      cameras.push_back(cam);
      angles.emplace_back(phi, theta);
    }
  return o.direct ? renderDirectViews(cb, o, cameras, angles) : renderViews(cb, o, cameras, angles);
}

// the reference's fibonacciHemisphere (main.cc:430-503): lattice point i of N has height z = (i + 1/2) 2/N - 1 (float),
// radius sqrt(1 - z^2) and azimuth ((i + rnd) mod N) * pi (3 - sqrt 5) (double); points with z < 0 become camera
// positions on the unit sphere around the box centre
int fibonacciHemisphere(CornellBox& cb, const Options& o)
{
  vtkm::rendering::Camera cam = sweepCamera();
  const int n = o.viewCount;
  if (n <= 0)
    return 0;
  const int rnd = ((o.viewSeed % n) + n) % n;
  const float offset = static_cast<float>(2. / n);
  const double increment = 3.14159265358979323846 * (3. - std::sqrt(5.0));
  std::vector<vtkm::rendering::Camera> cameras;
  ViewAngles angles;
  for (int i = 0; i < n; ++i)
  {
    const float z = ((i * offset) - 1) + (offset / 2);
    const float r = static_cast<float>(std::sqrt(1 - std::pow(z, 2)));
    const double phi = ((i + rnd) % n) * increment;
    const float x = static_cast<float>(std::cos(phi) * r);
    const float y = static_cast<float>(std::sin(phi) * r);
    if (z < 0)
    {
      cam.SetPosition(vec3(x + 278 / 555.0, y + 278 / 555.0, z + 278 / 555.0));
      cameras.push_back(cam);
      angles.emplace_back(0.f, static_cast<float>(i));
    }
  }
  return o.direct ? renderDirectViews(cb, o, cameras, angles) : renderViews(cb, o, cameras, angles);
}

} // namespace

int main(int argc, char* argv[])
{
  const Options o = parse(argc, argv);
  const auto t0 = std::chrono::steady_clock::now();
  try
  {
    auto cb = std::make_unique<CornellBox>();
    cb->buildDataSet();
    if (o.hemi || o.fibonacci)
    {
      const int views = o.fibonacci ? fibonacciHemisphere(*cb, o) : generateHemisphere(*cb, o);
      std::cout << " views rendered       = " << views << std::endl;
      b2pt_facade::ReleaseContext();
      const double dth = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      std::cout << " Elapsed time         = " << dth << std::endl;
      return 0;
    }
    vtkm::rendering::CanvasRayTracer canvas(o.x, o.y);
    vtkm::rendering::Camera cam; // main.cc:616-622
    cam.SetClippingRange(0.1f, 5.f);
    cam.SetPosition(vec3(278 / 555.0, 278 / 555.0, -800 / 555.0));
    cam.SetFieldOfView(40.);
    cam.SetViewUp(vec3(0, 1, 0));
    cam.SetLookAt(vec3(278 / 555.0, 278 / 555.0, 278 / 555.0));
    if (o.direct)
      runDirect(*cb, o, canvas, cam);
    else
    {
      runPath(*cb, o.samples, o.depth, canvas, cam, o.stats);
      savePnm(o.out, o.x, o.y, canvas.GetColorBuffer());
    }
  }
  catch (const vtkm::cont::Error& e)
  {
    std::cerr << "error: " << e.GetMessage() << std::endl;
    b2pt_facade::ReleaseContext();
    return 1;
  }
  b2pt_facade::ReleaseContext();
  const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  std::cout << " Elapsed time         = " << dt << std::endl;
  return 0;
}
