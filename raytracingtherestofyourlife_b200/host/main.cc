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
// -checkpoints c1,c2,... (with -hemisphere or -fibonacci, path-traced) also keeps the images at the lower sample counts
// c1 < c2 < ... < samplecount of the same render: <out>-s<c>-<phi>-<theta>.pnm for every listed c, each the file a
// sweep with -samplecount c writes, next to the usual <out>-<phi>-<theta>.pnm of samplecount samples (a denoiser
// dataset's noisy inputs and target from one sweep).  A malformed or non-increasing list, an entry >= samplecount,
// -direct, or no sweep is an error (exit 1).
// -features (with -hemisphere or -fibonacci, path-traced) also writes denoiser guide images of the same path samples,
// for the default sample count and every -checkpoints count c: <stem>-albedo-<phi>-<theta>.pfm (PF, mean first-hit
// albedo), <stem>-normal-<phi>-<theta>.pfm (PF, mean first-hit normal, not renormalised) and
// <stem>-depth-<phi>-<theta>.pfm (Pf, mean hit distance of the samples that hit, 0 where none does), with <stem> =
// <out> for samplecount samples and <out>-s<c> for a checkpoint.  PFM (little-endian float32, scale -1.0, rows bottom
// first as the buffers are) because PNM cannot hold negative normals or distances beyond 255.  The radiance files
// stay byte-identical to a run without -features.  -features with -direct, or without a sweep, is an error (exit 1).
// -denoise (with -hemisphere or -fibonacci, path-traced) also writes <stem>-denoised-<phi>-<theta>.pnm next to every
// radiance file <stem>-<phi>-<theta>.pnm: the same sweep through the edge-avoiding a-trous filter (b2pt_denoise_views
// with its default parameters), guided by the sweep's per-pixel variance, albedo, normal and depth, written with save()'s
// arithmetic.  The radiance files (and the -features PFMs) stay byte-identical to a run without -denoise.  -denoise with
// -direct, or without a sweep, is an error (exit 1).
// -adaptive <tau> (with -hemisphere or -fibonacci and -checkpoints) renders the sweep adaptively instead: the
// checkpoints and samplecount are the rounds, and after each round a pixel stops when the relative standard error of
// its mean luminance is below tau (b2pt_render_views_adaptive, default epsilon and radius).  It writes
// <out>-adaptive-<phi>-<theta>.pnm (save()'s arithmetic with each pixel's own sample count) and
// <out>-spp-<phi>-<theta>.pfm (Pf, the sample count of every pixel).  -adaptive without -checkpoints, with -direct,
// -features or -denoise, or with a tau that is not a number >= 0 is an error (exit 1).
// -adaptive-denoise <tau> is -adaptive <tau> with the adaptive sweep also denoised on the GPU at every pixel's own
// sample count (b2pt_render_views_adaptive_denoised, default filter parameters): the files of -adaptive <tau>,
// byte-identical, and <out>-adaptive-denoised-<phi>-<theta>.pnm.  The same uses as -adaptive are errors, and so is
// -adaptive-denoise with -adaptive.
// -aperture <a> [-focusdist <f>] renders every path-traced image -- the single render, -hemisphere, -fibonacci and
// every sweep option above -- through a thin lens of diameter a (b2pt_set_lens; the reference's camera has none):
// defocus blur away from the plane of focus, f scene units in front of each camera, or, with f <= 0 (the default), at
// each camera's look-at point (the box centre in the sweeps).  a = 0 is the pinhole; without the flags every file is
// what it was.  With -direct, or with a value that is not a finite number (a < 0 too), they are an error (exit 1).
// -motion (with -hemisphere, path-traced) also writes <stem>-motion-<phi>-<theta>.pfm for every <stem> of -features:
// motion vectors and disocclusion of the same path samples towards the previous view of the sweep (the first view
// towards itself), b2pt_render_views_motion: PF with the mean motion x and y in pixels (y up) and the fraction of the
// samples whose surface the previous view sees, over the samples whose hit lies in front of both cameras; 0 where there
// is none.  It works with -checkpoints, -features, -denoise and -aperture, and every other file stays byte-identical to
// a run without -motion.  -motion with -direct, without a sweep, with -fibonacci (consecutive lattice points are a
// golden angle apart, not neighbours) or with -adaptive / -adaptive-denoise is an error (exit 1).
// -temporal (with -hemisphere, path-traced) also writes <stem>-temporal-<phi>-<theta>.pnm next to every radiance file
// <stem>-<phi>-<theta>.pnm: the sweep with temporal accumulation along the motion of -motion's view chain (every view
// towards the one before it), then the a-trous filter (b2pt_denoise_views_temporal with its default parameters),
// written with save()'s arithmetic.  Every other file stays byte-identical to a run without -temporal.  -temporal is
// refused where -motion is: with -direct, without a sweep, with -fibonacci or with -adaptive / -adaptive-denoise.
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
  bool checkpointsGiven = false;
  std::string checkpointsArg;
  std::vector<int> checkpoints; // -checkpoints, parsed and checked by checkCheckpoints
  bool features = false;
  bool denoise = false;
  bool motion = false;
  bool temporal = false;
  bool adaptiveGiven = false;
  std::string adaptiveArg;
  bool adaptiveDenoiseGiven = false;
  std::string adaptiveDenoiseArg;
  float adaptive = 0.f; // -adaptive or -adaptive-denoise, parsed and checked by checkAdaptive
  bool apertureGiven = false, focusGiven = false;
  std::string apertureArg, focusArg;
  float aperture = 0.f, focus = 0.f; // -aperture / -focusdist, parsed and checked by checkLens
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
    else if (!std::strcmp(argv[i], "-features"))
      o.features = true;
    else if (!std::strcmp(argv[i], "-denoise"))
      o.denoise = true;
    else if (!std::strcmp(argv[i], "-motion"))
      o.motion = true;
    else if (!std::strcmp(argv[i], "-temporal"))
      o.temporal = true;
    else if (!std::strcmp(argv[i], "-adaptive"))
    {
      o.adaptiveGiven = true;
      if (i + 1 < argc)
        o.adaptiveArg = argv[++i];
    }
    else if (!std::strcmp(argv[i], "-adaptive-denoise"))
    {
      o.adaptiveDenoiseGiven = true;
      if (i + 1 < argc)
        o.adaptiveDenoiseArg = argv[++i];
    }
    else if (!std::strcmp(argv[i], "-checkpoints"))
    {
      o.checkpointsGiven = true;
      if (i + 1 < argc)
        o.checkpointsArg = argv[++i];
    }
    else if (!std::strcmp(argv[i], "-aperture"))
    {
      o.apertureGiven = true;
      if (i + 1 < argc)
        o.apertureArg = argv[++i];
    }
    else if (!std::strcmp(argv[i], "-focusdist"))
    {
      o.focusGiven = true;
      if (i + 1 < argc)
        o.focusArg = argv[++i];
    }
  }
  return o;
}

// Parses -checkpoints into o.checkpoints; returns an error message, empty when the list is usable.
std::string checkCheckpoints(Options& o)
{
  if (!o.checkpointsGiven)
    return "";
  if (o.direct)
    return "-checkpoints cannot be combined with -direct";
  if (!o.hemi && !o.fibonacci)
    return "-checkpoints needs -hemisphere or -fibonacci";
  const std::string malformed =
    "-checkpoints takes strictly increasing positive integers separated by commas, got '" + o.checkpointsArg + "'";
  std::stringstream list(o.checkpointsArg + ","); // every item, the last one too, ends with a comma
  std::string item;
  while (std::getline(list, item, ','))
  {
    if (item.empty() || item.size() > 9 || item.find_first_not_of("0123456789") != std::string::npos)
      return malformed;
    const int c = std::atoi(item.c_str());
    if (c < 1 || (!o.checkpoints.empty() && c <= o.checkpoints.back()))
      return malformed;
    o.checkpoints.push_back(c);
  }
  if (o.checkpoints.back() >= o.samples)
    return "-checkpoints entries must be below -samplecount (" + std::to_string(o.samples) + ")";
  return "";
}

// Returns an error message for an unusable -features, empty when it is usable or absent.
std::string checkFeatures(const Options& o)
{
  if (!o.features)
    return "";
  if (o.direct)
    return "-features cannot be combined with -direct";
  if (!o.hemi && !o.fibonacci)
    return "-features needs -hemisphere or -fibonacci";
  return "";
}

// Returns an error message for an unusable -denoise, empty when it is usable or absent.
std::string checkDenoise(const Options& o)
{
  if (!o.denoise)
    return "";
  if (o.direct)
    return "-denoise cannot be combined with -direct";
  if (!o.hemi && !o.fibonacci)
    return "-denoise needs -hemisphere or -fibonacci";
  return "";
}

// Returns an error message for an unusable -motion or -temporal (flag: the switch, given: whether it was), empty when
// it is usable or absent: both need the view chain of a hemisphere sweep.
std::string checkViewChain(const Options& o, const std::string& flag, bool given)
{
  if (!given)
    return "";
  if (o.direct)
    return flag + " cannot be combined with -direct";
  if (o.fibonacci)
    return flag + " cannot be combined with -fibonacci (consecutive lattice points are not neighbouring views)";
  if (!o.hemi)
    return flag + " needs -hemisphere";
  if (o.adaptiveGiven || o.adaptiveDenoiseGiven)
    return flag + " cannot be combined with -adaptive or -adaptive-denoise";
  return "";
}

// Parses the threshold arg of the adaptive switch `flag` into o.adaptive; returns an error message, empty when the
// switch is usable.
std::string checkAdaptiveSwitch(Options& o, const std::string& flag, const std::string& arg)
{
  if (o.direct)
    return flag + " cannot be combined with -direct";
  if (o.features || o.denoise)
    return flag + " cannot be combined with -features or -denoise";
  if (!o.hemi && !o.fibonacci)
    return flag + " needs -hemisphere or -fibonacci";
  if (!o.checkpointsGiven)
    return flag + " needs -checkpoints (the rounds before samplecount)";
  char* end = nullptr;
  const float tau = std::strtof(arg.c_str(), &end);
  if (arg.empty() || *end != '\0' || !(tau >= 0.f))
    return flag + " takes a threshold >= 0, got '" + arg + "'";
  o.adaptive = tau;
  return "";
}

// Parses -adaptive or -adaptive-denoise; returns an error message, empty when it is usable or absent.
std::string checkAdaptive(Options& o)
{
  if (o.adaptiveGiven && o.adaptiveDenoiseGiven)
    return "-adaptive-denoise cannot be combined with -adaptive";
  if (o.adaptiveGiven)
    return checkAdaptiveSwitch(o, "-adaptive", o.adaptiveArg);
  if (o.adaptiveDenoiseGiven)
    return checkAdaptiveSwitch(o, "-adaptive-denoise", o.adaptiveDenoiseArg);
  return "";
}

// Parses -aperture and -focusdist into o.aperture / o.focus; returns an error message, empty when they are usable or
// absent.
std::string checkLens(Options& o)
{
  if (!o.apertureGiven && !o.focusGiven)
    return "";
  if (o.direct)
    return "-aperture and -focusdist cannot be combined with -direct (its G-buffers use the pinhole corner rays)";
  auto number = [](const std::string& arg, float& out) {
    char* end = nullptr;
    out = std::strtof(arg.c_str(), &end);
    return !arg.empty() && *end == '\0' && std::isfinite(out);
  };
  if (o.apertureGiven && (!number(o.apertureArg, o.aperture) || o.aperture < 0.f))
    return "-aperture takes a finite lens diameter >= 0, got '" + o.apertureArg + "'";
  if (o.focusGiven && !number(o.focusArg, o.focus))
    return "-focusdist takes a finite distance, got '" + o.focusArg + "'";
  return "";
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
// (plus the -aperture / -focusdist lens, an extension)
void runPath(CornellBox& cb, int samplecount, int depthcount, vtkm::rendering::Canvas& canvas,
             vtkm::rendering::Camera& cam, bool stats, float aperture, float focus)
{
  vtkm::rendering::MapperPathTracer mapper(samplecount, depthcount, cb.matIdx, cb.texIdx, cb.matType, cb.texType,
                                           cb.tex);
  mapper.SetCanvas(&canvas);
  mapper.SetLens(aperture, focus);
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

// Portable float map: "PF" (rgb) or "Pf" (grey), scale -1.0 (little-endian float32: the host's own layout on the
// x86-64 and aarch64 hosts of a B200), rows bottom first.
void savePfm(const std::string& stem, int nx, int ny, int channels, const std::vector<float>& values)
{
  std::ofstream fs(stem + ".pfm", std::ios::binary);
  if (!fs)
  {
    std::cout << "Couldn't save pfm." << std::endl;
    return;
  }
  fs << (channels == 3 ? "PF" : "Pf") << "\n" << nx << " " << ny << "\n-1.0\n";
  fs.write(reinterpret_cast<const char*>(values.data()), static_cast<std::streamsize>(values.size() * sizeof(float)));
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
  mapper.SetLens(o.aperture, o.focus);
  std::vector<unsigned short> pnm, denoised;
  std::vector<int> counts = o.checkpoints; // -checkpoints: one render, its images at every count up to samplecount
  counts.push_back(o.samples);
  if (o.adaptiveGiven || o.adaptiveDenoiseGiven)
  { // the rounds are the counts; one image and one sample-count map per view (and one denoised image)
    std::vector<int> spp;
    if (o.adaptiveDenoiseGiven)
      mapper.RenderCellsViewsAdaptiveDenoisedPnm(cb.ds.GetCellSet(), cb.coord, cameras, counts, o.adaptive, pnm, spp,
                                                 denoised);
    else
      mapper.RenderCellsViewsAdaptivePnm(cb.ds.GetCellSet(), cb.coord, cameras, counts, o.adaptive, pnm, spp);
    const size_t n = static_cast<size_t>(o.x) * o.y;
    std::vector<float> map(n);
    for (size_t v = 0; v < cameras.size(); ++v)
    {
      savePnm16(viewName(o.out + "-adaptive", angles[v].first, angles[v].second), o.x, o.y, &pnm[v * n * 3]);
      if (o.adaptiveDenoiseGiven)
        savePnm16(viewName(o.out + "-adaptive-denoised", angles[v].first, angles[v].second), o.x, o.y,
                  &denoised[v * n * 3]);
      for (size_t i = 0; i < n; ++i)
        map[i] = static_cast<float>(spp[v * n + i]);
      savePfm(viewName(o.out + "-spp", angles[v].first, angles[v].second), o.x, o.y, 1, map);
    }
    return static_cast<int>(cameras.size());
  }
  if (o.denoise) // the same integers as below, from the float sums the filter needs
    mapper.RenderCellsViewsDenoisedPnm(cb.ds.GetCellSet(), cb.coord, cameras, counts, pnm, denoised);
  else if (counts.size() > 1)
    mapper.RenderCellsViewsCheckpointsPnm(cb.ds.GetCellSet(), cb.coord, cameras, counts, pnm);
  else
    mapper.RenderCellsViewsPnm(cb.ds.GetCellSet(), cb.coord, cameras, pnm);
  if (o.stats)
    std::cout << " GPU render ms = " << mapper.GetLastRenderMilliseconds() << " for " << cameras.size() << " views"
              << "  path samples/s = " << double(o.x) * o.y * o.samples * double(cameras.size()) /
        (mapper.GetLastRenderMilliseconds() * 1e-3)
              << "  segments = " << mapper.GetLastSegments() << std::endl;
  const size_t n = static_cast<size_t>(o.x) * o.y, n3 = n * 3, V = cameras.size();
  auto stemOf = [&](size_t k) { // slice k: counts[k] samples; the last is the ordinary image
    return k + 1 < counts.size() ? o.out + "-s" + std::to_string(counts[k]) : o.out;
  };
  for (size_t k = 0; k < counts.size(); ++k)
    for (size_t v = 0; v < V; ++v)
      savePnm16(viewName(stemOf(k), angles[v].first, angles[v].second), o.x, o.y, &pnm[(k * V + v) * n3]);
  if (o.denoise)
    for (size_t k = 0; k < counts.size(); ++k)
      for (size_t v = 0; v < V; ++v)
        savePnm16(viewName(stemOf(k) + "-denoised", angles[v].first, angles[v].second), o.x, o.y,
                  &denoised[(k * V + v) * n3]);
  if (o.features)
  { // the guide images: sums over the samples of each count, as means
    std::vector<float> albedo, normalDepth;
    mapper.RenderCellsViewsFeatures(cb.ds.GetCellSet(), cb.coord, cameras, counts, albedo, normalDepth);
    std::vector<float> alb(n3), nrm(n3), dep(n);
    for (size_t k = 0; k < counts.size(); ++k)
    {
      const float c = static_cast<float>(counts[k]);
      for (size_t v = 0; v < V; ++v)
      {
        const float* a = &albedo[(k * V + v) * n * 4];
        const float* nd = &normalDepth[(k * V + v) * n * 4];
        for (size_t i = 0; i < n; ++i)
        {
          for (int ch = 0; ch < 3; ++ch)
          {
            alb[3 * i + ch] = a[4 * i + ch] / c;
            nrm[3 * i + ch] = nd[4 * i + ch] / c;
          }
          dep[i] = a[4 * i + 3] > 0.f ? nd[4 * i + 3] / a[4 * i + 3] : 0.f;
        }
        const std::string stem = stemOf(k);
        savePfm(viewName(stem + "-albedo", angles[v].first, angles[v].second), o.x, o.y, 3, alb);
        savePfm(viewName(stem + "-normal", angles[v].first, angles[v].second), o.x, o.y, 3, nrm);
        savePfm(viewName(stem + "-depth", angles[v].first, angles[v].second), o.x, o.y, 1, dep);
      }
    }
  }
  if (o.motion)
  { // every view towards the one before it in sweep order, the first towards itself; sums as means over valid samples
    std::vector<vtkm::rendering::Camera> prevCameras(cameras.begin(), cameras.end() - 1);
    prevCameras.insert(prevCameras.begin(), cameras.front());
    std::vector<float> motion, mv(n3);
    mapper.RenderCellsViewsMotion(cb.ds.GetCellSet(), cb.coord, cameras, prevCameras, counts, motion);
    for (size_t k = 0; k < counts.size(); ++k)
      for (size_t v = 0; v < V; ++v)
      {
        const float* m = &motion[(k * V + v) * n * 4];
        for (size_t i = 0; i < n; ++i)
        {
          const float valid = m[4 * i + 3];
          for (int ch = 0; ch < 3; ++ch)
            mv[3 * i + ch] = valid > 0.f ? m[4 * i + ch] / valid : 0.f;
        }
        savePfm(viewName(stemOf(k) + "-motion", angles[v].first, angles[v].second), o.x, o.y, 3, mv);
      }
  }
  if (o.temporal)
  { // the same render, guides and view chain as above, accumulated over the sweep and filtered
    std::vector<unsigned short> temporal;
    mapper.RenderCellsViewsTemporalPnm(cb.ds.GetCellSet(), cb.coord, cameras, counts, temporal);
    for (size_t k = 0; k < counts.size(); ++k)
      for (size_t v = 0; v < V; ++v)
        savePnm16(viewName(stemOf(k) + "-temporal", angles[v].first, angles[v].second), o.x, o.y,
                  &temporal[(k * V + v) * n3]);
  }
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
  Options o = parse(argc, argv);
  std::string bad = checkCheckpoints(o);
  if (bad.empty())
    bad = checkFeatures(o);
  if (bad.empty())
    bad = checkDenoise(o);
  if (bad.empty())
    bad = checkAdaptive(o);
  if (bad.empty())
    bad = checkViewChain(o, "-motion", o.motion);
  if (bad.empty())
    bad = checkViewChain(o, "-temporal", o.temporal);
  if (bad.empty())
    bad = checkLens(o);
  if (!bad.empty())
  {
    std::cerr << "error: " << bad << std::endl;
    return 1;
  }
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
      runPath(*cb, o.samples, o.depth, canvas, cam, o.stats, o.aperture, o.focus);
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
