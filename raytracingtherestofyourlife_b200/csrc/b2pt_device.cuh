// b2pt_device.cuh -- device functions of the path-tracing hot path (sm_100a).
//
// This translation unit is compiled with -fmad=false (and the default -prec-div=true -prec-sqrt=true
// -ftz=false): every geometric predicate below evaluates the same IEEE-754 single-precision operation
// sequence as the reference built for x86-64 without FMA contraction, so ray generation, hit/miss
// decisions, hit points, normals and sampled directions are bit-identical to the CPU oracle (modulo
// libm sinf/cosf).  Radiance-only arithmetic (pdf mixture, attenuation) runs in FP32 where the reference
// promotes to Float64 through vtkm::Pi(); that changes radiance by <= a few ulp and never a trajectory.
//
// Each function cites the reference code it restates (paths relative to the reference root).
#ifndef B2PT_DEVICE_CUH
#define B2PT_DEVICE_CUH

#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "b2pt_types.h"

namespace b2pt
{

struct f3
{
  float x, y, z;
};

__device__ __forceinline__ f3 mk3(float x, float y, float z)
{
  f3 r;
  r.x = x;
  r.y = y;
  r.z = z;
  return r;
}
__device__ __forceinline__ f3 ld3(const float* p) { return mk3(p[0], p[1], p[2]); }
__device__ __forceinline__ f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ f3 operator-(f3 a) { return mk3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ f3 operator*(f3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ f3 mul3(f3 a, f3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
// vtkm::Dot for Vec3: (a0*b0 + a1*b1) + a2*b2
__device__ __forceinline__ float dot3(f3 a, f3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
// vtkm::Cross (plain form)
__device__ __forceinline__ f3 cross3(f3 a, f3 b)
{
  return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// vtkm::RMagnitude = RSqrt(MagnitudeSquared), host form 1/sqrt (not rsqrtf: keeps CPU bit-parity)
__device__ __forceinline__ float rmag3(f3 a) { return 1.0f / sqrtf(dot3(a, a)); }
__device__ __forceinline__ f3 unit3(f3 a) { return a * rmag3(a); } // vec3.h:38-42, vtkm::Normalize
// Radiance-only arithmetic (pdf values, cosines, attenuation: numbers that are multiplied into the throughput and never
// decide a hit, a branch or a direction) uses the hardware reciprocal / reciprocal square root (MUFU, <= 2 ulp) instead
// of the IEEE-rounded sequences: the reference itself evaluates these in a mix of Float32 and Float64 (vtkm::Pi()), so
// they were never bit-comparable; signs, exact zeros, infinities and NaNs -- everything the NaN-poisoning semantics and
// the comparisons depend on -- are preserved.
__device__ __forceinline__ float rmag3_fast(f3 a) { return rsqrtf(dot3(a, a)); }
__device__ __forceinline__ f3 unit3_fast(f3 a) { return a * rmag3_fast(a); }
__device__ __forceinline__ float div_fast(float a, float b) { return __fdividef(a, b); }
__device__ __forceinline__ f3 denan3(f3 c) // PdfWorklet.h:39-45
{
  if (!(c.x == c.x))
    c.x = 0.f;
  if (!(c.y == c.y))
    c.y = 0.f;
  if (!(c.z == c.z))
    c.z = 0.f;
  return c;
}

// ---------------------------------------------------------------------------------------------- RNG
// wangXor.h:30-38
__device__ __forceinline__ uint32_t wang32(uint32_t& seed)
{
  uint32_t s = seed;
  s = (s ^ 61u) ^ (s >> 16);
  s *= 9u;
  s = s ^ (s >> 4);
  s *= 0x27d4eb2du;
  s = s ^ (s >> 15);
  seed = s;
  return s;
}
// wangXor.h:55-59: Float32(t) / 4294967295.f.  The divisor rounds to 2^32 in binary32, so the division is
// an exact scaling and equals the multiplication by 2^-32 below bit for bit.
__device__ __forceinline__ float randf(uint32_t& seed)
{
  uint32_t t = wang32(seed);
  return __uint2float_rn(t) * 2.3283064365386963e-10f;
}
// PdfWorklet.h:19-21 with genDir(3), WhichGenerateDir.cxx:10
__device__ __forceinline__ int draw_which(uint32_t& seed)
{
  int w = (int)(randf(seed) * 3.f + 1.f);
  return w > 3 ? 3 : w;
}
// Draws a dead pixel still consumes in the reference: per remaining depth 1 (which) + the generator's -- cosine 2,
// 3 per light quad, 2 per light sphere: the generators loop over every light whether the pixel is alive or not
// (PdfWorklet.h:122, :203; SURVEY A.3).  Only used by B2PT_FLAG_REFERENCE_STREAM.
__device__ __forceinline__ void burn_depths(uint32_t& seed, int count, int nLightQuads, int nLightSph)
{
  for (int k = 0; k < count; ++k)
  {
    const int w = draw_which(seed);
    const int nd = (w <= 1) ? 2 : (w == 2 ? 3 * nLightQuads : 2 * nLightSph);
    for (int j = 0; j < nd; ++j)
      wang32(seed);
  }
}

// ------------------------------------------------------------------------------------------- camera
// pathtracing/Camera.cxx:483-524 (RayGen::operator()).  Consumes two draws.
__device__ __forceinline__ f3 raygen(const B2Camera& cam, int pixel, uint32_t& seed)
{
  int i = pixel % cam.W;
  int j = pixel / cam.W;
  float ru = randf(seed);
  float rv = randf(seed);
  float sx = (2.f * ((float)i + (1.f - ru)) - (float)cam.W) / 2.0f;
  float sy = (2.f * ((float)j + rv) - (float)cam.H) / 2.0f;
  f3 d = (ld3(cam.nlook) + ld3(cam.dx) * sx) + ld3(cam.dy) * sy;
  if (d.x == 0.f)
    d.x += 0.0000001f;
  if (d.y == 0.f)
    d.y += 0.0000001f;
  if (d.z == 0.f)
    d.z += 0.0000001f;
  float m = sqrtf(dot3(d, d));
  return mk3(d.x / m, d.y / m, d.z / m);
}

// Thin lens (b2pt_set_lens, DESIGN.md 8h) applied to the pinhole ray d0 = raygen(...): a point (a, b) of the unit disk
// by bounded rejection (at most 16 pairs of draws; (0, 0) after 16 rejections), the origin o = pos + u*(r*a) + v*(r*b)
// on the lens, and the direction from o to the point F = pos + d0 * (f / (d0 . nlook)) where the pinhole ray meets
// the plane of focus; zero components nudged and normalised as raygen does.  Consumes 2k draws for k pairs.  The float
// operations and their order are the ones include/b2pt.h fixes (b2pt_set_lens), so the CPU restatement agrees bit for
// bit under -fmad=false.
__device__ __forceinline__ void lens_ray(const B2Camera& cam, const B2Lens& L, f3 d0, uint32_t& seed, f3& o, f3& d)
{
  float a = 0.f, b = 0.f;
#pragma unroll 1
  for (int k = 0; k < 16; ++k)
  {
    const float x = 2.f * randf(seed) - 1.f;
    const float y = 2.f * randf(seed) - 1.f;
    if (x * x + y * y < 1.f)
    {
      a = x, b = y;
      break;
    }
  }
  const f3 pos = ld3(cam.pos);
  const float ra = L.r * a, rb = L.r * b;
  o = (pos + ld3(L.u) * ra) + ld3(L.v) * rb;
  const float k = L.f / dot3(d0, ld3(cam.nlook));
  const f3 F = pos + d0 * k;
  d = F - o;
  if (d.x == 0.f)
    d.x += 0.0000001f;
  if (d.y == 0.f)
    d.y += 0.0000001f;
  if (d.z == 0.f)
    d.z += 0.0000001f;
  const float m = sqrtf(dot3(d, d));
  d = mk3(d.x / m, d.y / m, d.z / m);
}

// Pinhole projection of a world point X into camera cam, the inverse of raygen (b2pt_render_views_motion, DESIGN.md
// 8i): D = X - pos, w = D . nlook, x = (D . dx) / (w * (dx . dx)) + W/2, y likewise with dy and H, continuous pixel
// coordinates in which raygen's sample of pixel (i, j) with jitter (fx, fy) sits at (i + fx, j + fy).  Returns w; X is in
// front of the camera when w > 0.  The float operations and their order are the ones include/b2pt.h fixes, so the CPU
// restatement agrees bit for bit under -fmad=false.
__device__ __forceinline__ float project(const B2Camera& cam, f3 X, float& x, float& y)
{
  const f3 D = X - ld3(cam.pos);
  const f3 dx = ld3(cam.dx), dy = ld3(cam.dy);
  const float w = dot3(D, ld3(cam.nlook));
  x = dot3(D, dx) / (w * dot3(dx, dx)) + 0.5f * (float)cam.W;
  y = dot3(D, dy) / (w * dot3(dy, dy)) + 0.5f * (float)cam.H;
  return w;
}

// pathtracing/Camera.cxx:394-423 (Camera::PerspectiveRayGen, the generator of the -direct modes): the un-jittered ray
// through the pixel's lower-left corner.
__device__ __forceinline__ f3 raygen_corner(const B2Camera& cam, int pixel)
{
  const int i = pixel % cam.W, j = pixel / cam.W;
  f3 d = (ld3(cam.nlook) + ld3(cam.dx) * ((2.f * (float)i - (float)cam.W) / 2.0f)) +
    ld3(cam.dy) * ((2.f * (float)j - (float)cam.H) / 2.0f);
  if (d.x == 0.f)
    d.x += 0.0000001f;
  if (d.y == 0.f)
    d.y += 0.0000001f;
  if (d.z == 0.f)
    d.z += 0.0000001f;
  const float m = sqrtf(dot3(d, d));
  return mk3(d.x / m, d.y / m, d.z / m);
}
// raygen's direction for pixel (i, j) at jitter (0.5, 0.5), the pixel centre, with no draws (the expected distance of
// b2pt_denoise_views_temporal): the same float operations as raygen with ru = rv = 0.5.
__device__ __forceinline__ f3 raygen_centre(const B2Camera& cam, int i, int j)
{
  const float sx = (2.f * ((float)i + 0.5f) - (float)cam.W) / 2.0f;
  const float sy = (2.f * ((float)j + 0.5f) - (float)cam.H) / 2.0f;
  f3 d = (ld3(cam.nlook) + ld3(cam.dx) * sx) + ld3(cam.dy) * sy;
  if (d.x == 0.f)
    d.x += 0.0000001f;
  if (d.y == 0.f)
    d.y += 0.0000001f;
  if (d.z == 0.f)
    d.z += 0.0000001f;
  const float m = sqrtf(dot3(d, d));
  return mk3(d.x / m, d.y / m, d.z / m);
}
// The per-pixel colour rules of the -direct G-buffers: raytracing/RayTracerNormals.cxx:137-140 (the hit normal) and
// RayTracerAlbedo.cxx:100-143 (cosPhi * R / (cosTheta * L) per channel, with the light at camera + 2 up, :154-155).
// Same float operations in the same order as the reference's worklets (pinned through the oracle, tests/).
__device__ __forceinline__ void direct_shade(f3 n, f3 p, f3 camPos, f3 lookAt, f3 upN, float4& normals, float4& albedo)
{
  const f3 lightPosition = camPos + mk3(2.f * upN.x, 2.f * upN.y, 2.f * upN.z);
  const f3 L = unit3(lightPosition - p);
  const f3 V = unit3(camPos - lookAt);
  float cosTheta = dot3(n, L);
  cosTheta = fminf(fmaxf(cosTheta, 0.f), 1.f);
  const float s = 2.f * dot3(L, n);
  const f3 R = unit3(n * s - L);
  const float cosPhi = dot3(R, V);
  normals = make_float4(n.x, n.y, n.z, 1.f);
  albedo = make_float4((cosPhi * R.x) / (cosTheta * L.x), (cosPhi * R.y) / (cosTheta * L.y),
                       (cosPhi * R.z) / (cosTheta * L.z), 1.f);
}

// --------------------------------------------------------------------------------------- primitives
// Surface.h:30-104 (Lagae-Dutre ray/quad test up to t; the bilinear u,v of :106-158 are never consumed
// downstream and are not computed).  Returns true iff the reference's hit() returns true; t is valid then.
__device__ __forceinline__ bool quad_hit(const B2Quad& Q, f3 o, f3 d, float& t)
{
  const float4* q4 = reinterpret_cast<const float4*>(&Q);
  const float4 c0 = q4[0], c1 = q4[1], c2 = q4[2]; // v00 e01 | e01 e03 | e03 v11
  const f3 E03 = mk3(c1.z, c1.w, c2.x);
  f3 P = cross3(d, E03);
  const f3 E01 = mk3(c0.w, c1.x, c1.y);
  float det = dot3(E01, P);
  if (fabsf(det) < 1e-5f) // vtkm::Epsilon<Float32>()
    return false;
  float inv_det = 1.0f / det;
  f3 T = o - mk3(c0.x, c0.y, c0.z);
  float alpha = dot3(T, P) * inv_det;
  if (alpha < 0.0f)
    return false;
  f3 Qv = cross3(T, E01);
  float beta = dot3(d, Qv) * inv_det;
  if (beta < 0.0f)
    return false;
  if ((alpha + beta) > 1.0f)
  {
    // Shortcut (never changes the outcome, B2Quad::secC1): on a parallelogram alpha' = 1 - alpha, beta' = 1 - beta and
    // det' = det, so while alpha and beta stay below 1 by more than the rounding error of both evaluations the
    // second triangle's reject tests cannot fire and t below is all that is left.  Near an edge, for |det| close to
    // the epsilon, for NaNs and for general quads the reference's second-triangle arithmetic runs as written.
    const float need = ((fabsf(T.x) + fabsf(T.y)) + fabsf(T.z) + Q.secC1) * ((fabsf(d.x) + fabsf(d.y)) + fabsf(d.z)) * Q.secC2;
    if (!((1.0f - fmaxf(alpha, beta)) * fabsf(det) > need && fabsf(det) >= 2e-5f))
    {
    const float4 c3 = q4[3], c4 = q4[4]; // v11 e21 | e21 e23 nrm
    const f3 E23 = mk3(c3.w, c4.x, c4.y);
    const f3 E21 = mk3(c3.x, c3.y, c3.z);
    f3 Pp = cross3(d, E21);
    float detp = dot3(E23, Pp);
    if (fabsf(detp) < 1e-5f)
      return false;
    float inv_detp = 1.0f / detp;
    f3 Tp = o - mk3(c2.y, c2.z, c2.w);
    float alphap = dot3(Tp, Pp) * inv_detp;
    if (alphap < 0.0f)
      return false;
    f3 Qp = cross3(Tp, E23);
    float betap = dot3(d, Qp) * inv_detp;
    if (betap < 0.0f)
      return false;
    }
  }
  t = dot3(E03, Qv) * inv_det;
  if (t < 0.0f)
    return false;
  return true;
}
// Surface.h:163-199 acceptance rule.
__device__ __forceinline__ bool quad_accept(const B2Quad& Q, f3 o, f3 d, float tmin, float tmax, float& t)
{
  float tt;
  bool h = quad_hit(Q, o, d, tt);
  h = h && (tt < tmax) && (tt > tmin);
  if (h)
    t = tt;
  return h;
}
// Surface.h:180-186: geometric normal flipped to oppose the ray.
__device__ __forceinline__ f3 quad_normal(const B2Quad& Q, f3 d)
{
  f3 n = ld3(Q.nrm);
  if (dot3(n, d) > 0.f)
    n = -n;
  return n;
}
// Surface.h:319-367: first root in (tmin,tmax) wins.
__device__ __forceinline__ bool sphere_accept(f3 c, float radius, f3 o, f3 d, float tmin, float tmax, float& t)
{
  f3 oc = o - c;
  float a = dot3(d, d);
  float b = dot3(oc, d);
  float cc = dot3(oc, oc) - radius * radius;
  float disc = b * b - a * cc;
  if (disc > 0.f)
  {
    float sq = sqrtf(b * b - a * cc);
    float temp = (-b - sq) / a;
    if (temp < tmax && temp > tmin)
    {
      t = temp;
      return true;
    }
    temp = (-b + sq) / a;
    if (temp < tmax && temp > tmin)
    {
      t = temp;
      return true;
    }
  }
  return false;
}

// BVHTraverser.h:35-79 slab test against one box with rcp_safe'd inverse direction (:90-93, :145-157).
__device__ __forceinline__ bool slab_hit(const float* bmin, const float* bmax, f3 inv, f3 od, float tmin,
                                         float closest, float& tnear)
{
  float xmin = bmin[0] * inv.x - od.x, ymin = bmin[1] * inv.y - od.y, zmin = bmin[2] * inv.z - od.z;
  float xmax = bmax[0] * inv.x - od.x, ymax = bmax[1] * inv.y - od.y, zmax = bmax[2] * inv.z - od.z;
  float mn = fmaxf(fmaxf(fmaxf(fminf(ymin, ymax), fminf(xmin, xmax)), fminf(zmin, zmax)), tmin);
  float mx = fminf(fminf(fminf(fmaxf(ymin, ymax), fmaxf(xmin, xmax)), fmaxf(zmin, zmax)), closest);
  tnear = mn;
  return mx >= mn;
}
// Same slab test with FMA contraction, for the BVH traversal only: there the padded boxes are conservative
// culling volumes (hit / t come from the exact primitive tests), so the last-ulp difference cannot change a result.
__device__ __forceinline__ bool slab_hit_fma(float4 lo, float4 hi, f3 inv, f3 od, float tmin, float closest, float& tnear)
{
  const float xmin = __fmaf_rn(lo.x, inv.x, -od.x), ymin = __fmaf_rn(lo.y, inv.y, -od.y), zmin = __fmaf_rn(lo.z, inv.z, -od.z);
  const float xmax = __fmaf_rn(hi.x, inv.x, -od.x), ymax = __fmaf_rn(hi.y, inv.y, -od.y), zmax = __fmaf_rn(hi.z, inv.z, -od.z);
  const float mn = fmaxf(fmaxf(fmaxf(fminf(ymin, ymax), fminf(xmin, xmax)), fminf(zmin, zmax)), tmin);
  const float mx = fminf(fminf(fminf(fmaxf(ymin, ymax), fmaxf(xmin, xmax)), fmaxf(zmin, zmax)), closest);
  tnear = mn;
  return mx >= mn;
}
__device__ __forceinline__ float rcp_safe(float f) { return 1.0f / ((fabsf(f) < 1e-8f) ? 1e-8f : f); }
// The reference reaches a sphere only through its own leaf box (FindSphereAABBs, AABBSurface.h:82-174: centre +- radius
// per axis, unpadded) with the traverser's slab test (BVHTraverser.h:35-79).  The analytic sphere test cancels badly
// for small spheres far from the ray origin (it reports hits up to ~|oc|^2*2^-24/(2r) outside the surface), so this
// gate decides grazing hits.  It is evaluated with the reference's arithmetic before every sphere test, against tmax
// rather than the running closest distance so that the winner among near-coincident grazing hits does not depend
// on the order in which a tree (or a list) presents the spheres (same rule in the oracle).
__device__ __forceinline__ bool sphere_gate(f3 c, float r, f3 inv, f3 od, float tmin, float tmax)
{
  const float lo[3] = { fminf(c.x + r, c.x - r), fminf(c.y + r, c.y - r), fminf(c.z + r, c.z - r) };
  const float hi[3] = { fmaxf(c.x + r, c.x - r), fmaxf(c.y + r, c.y - r), fmaxf(c.z + r, c.z - r) };
  float tn;
  return slab_hit(lo, hi, inv, od, tmin, tmax, tn);
}

// Culling form of the sphere test (FMA arithmetic, ~20 instructions): false only when the exact test below -- the
// reference's float sequence -- certainly finds disc <= 0, i.e. the ray's line misses the sphere.  Both evaluations of
// disc = b^2 - a*cc lie within 4.2e-7 (B^2 + a (|oc|^2 + r^2)) of the exact value (B = sum |oc_i d_i|; three-term sums
// and products, u = 2^-24), so a margin of 2e-6 of that scale separates them safely.  Most spheres a BVH leaf offers
// are missed by the line, and they never reach the IEEE sqrt / divisions of the exact test.
__device__ __forceinline__ bool sphere_may_hit(f3 c, float r, f3 o, f3 d)
{
  const float ox = o.x - c.x, oy = o.y - c.y, oz = o.z - c.z;
  const float a = __fmaf_rn(d.x, d.x, __fmaf_rn(d.y, d.y, d.z * d.z));
  const float b = __fmaf_rn(ox, d.x, __fmaf_rn(oy, d.y, oz * d.z));
  const float q = __fmaf_rn(ox, ox, __fmaf_rn(oy, oy, oz * oz));
  const float disc = __fmaf_rn(b, b, -a * __fmaf_rn(-r, r, q));
  const float B = __fmaf_rn(fabsf(ox), fabsf(d.x), __fmaf_rn(fabsf(oy), fabsf(d.y), fabsf(oz) * fabsf(d.z)));
  return disc > -2e-6f * __fmaf_rn(B, B, a * __fmaf_rn(r, r, q));
}

struct Hit
{
  f3 p, n, alb;
  float t;
  int kind; // matType of the hit primitive
  int prim; // original primitive id (quad q, sphere nQuads+s), -1 miss
  int mat, texi;
};

// Lagae-Dutre test of an axis-aligned rectangle in its permuted frame (u,v,n): the operations of quad_hit
// that do not multiply by an exact zero, in the same order, so the result is bit-identical (see B2AAQuad).
// Branch-free up to the second-triangle part.  NaN handling follows the reference's comparisons.
__device__ __forceinline__ bool aa_quad_hit(const B2AAQuad& Q, float du, float dv, float dn, float ou, float ov,
                                            float on, float& t)
{
  // three broadcast 16-byte loads (LDS.128 when the scene is staged in shared memory)
  const float4* q4 = reinterpret_cast<const float4*>(&Q);
  const float4 c0 = q4[0]; // v00u v00v v00n bPu
  const float4 c1 = q4[1]; // v11u v11v v11n bPn
  const float4 c2 = q4[2]; // a aQv aQn b
  const float Pu = dn * c0.w, Pn = du * c1.w;
  const float det = c2.x * Pu;
  const float Tu = ou - c0.x, Tv = ov - c0.y, Tn = on - c0.z;
  const float x1 = Tu * Pu, x2 = Tn * Pn;
  const float TP = x1 + x2;
  const float Qv = Tn * c2.y, Qn = Tv * c2.z;
  const float y1 = dv * Qv, y2 = dn * Qn;
  const float DQ = y1 + y2;
  const float inv_det = 1.0f / det;
  const float alpha = TP * inv_det;
  const float beta = DQ * inv_det;
  t = (c2.w * Qv) * inv_det;
  bool ok = !(fabsf(det) < 1e-5f) && !(alpha < 0.0f) && !(beta < 0.0f) && !(t < 0.0f);
  if (ok && (alpha + beta) > 1.0f)
  {
    // Second-triangle test (Surface.h:72-98).  For a consistent rectangle (host-verified: a2 = -a, b2 = -b,
    // v11 = v00 + E01 + E03 to 2e-6) its barycentrics are alpha' = 1 - alpha, beta' = 1 - beta in exact
    // arithmetic, and the float evaluations of alpha, beta, alpha', beta' are each within
    // u*(4R+14), u = 2^-24, of their exact values, R = (|x1|+|x2|)/|det| resp. (|y1|+|y2|)/|det| (standard
    // forward error of the two-term sums and the division).  Outside a band E = 1e-6*R + 1e-5 > 2x that
    // bound around 1 the outcome of the exact test is therefore known; only inside the band is it evaluated.
    const float ainv = fabsf(inv_det);
    const float Ea = __fmaf_rn(1e-6f, (fabsf(x1) + fabsf(x2)) * ainv, 1e-5f);
    const float Eb = __fmaf_rn(1e-6f, (fabsf(y1) + fabsf(y2)) * ainv, 1e-5f);
    const bool rect = Q.cls >= 8;
    const bool sureOut = rect && (alpha > 1.0f + Ea || beta > 1.0f + Eb);
    const bool sureIn = rect && alpha < 1.0f - Ea && beta < 1.0f - Eb && fabsf(det) > 1.1e-5f;
    if (sureOut)
      ok = false;
    else if (!sureIn)
    {
      const float4 c3 = q4[3]; // a2 b2Pu b2Pn a2Qv
      const float a2Qn = Q.a2Qn;
      const float Ppu = dn * c3.y, Ppn = du * c3.z;
      const float detp = c3.x * Ppu;
      const float Tpu = ou - c1.x, Tpv = ov - c1.y, Tpn = on - c1.z;
      const float inv_detp = 1.0f / detp;
      const float alphap = (Tpu * Ppu + Tpn * Ppn) * inv_detp;
      const float betap = (dv * (Tpn * c3.w) + dn * (Tpv * a2Qn)) * inv_detp;
      ok = !(fabsf(detp) < 1e-5f) && !(alphap < 0.0f) && !(betap < 0.0f);
    }
  }
  return ok;
}

// (u,v,n) component selection for class c (B2AAQuad::cls & 7); c is warp-uniform.
__device__ __forceinline__ void aa_permute(int c, f3 a, float& u, float& v, float& n)
{
  switch (c & 7)
  {
    case 0: u = a.x, v = a.y, n = a.z; break;
    case 1: u = a.y, v = a.z, n = a.x; break;
    case 2: u = a.z, v = a.x, n = a.y; break;
    case 3: u = a.y, v = a.x, n = a.z; break;
    case 4: u = a.x, v = a.z, n = a.y; break;
    default: u = a.z, v = a.y, n = a.x; break;
  }
}

// ---- phase 1 of the small-scene trace: candidate filter (B2FiltPair).  All 32 lanes run the same
// straight-line code per pair of quads (no divergence), on packed FP32 pairs (FFMA2 / FADD2: two quads per
// instruction); the output per lane is the candidate bit mask (bit nVisit-1-v for visit index v), the smallest
// LOWER BOUND of a candidate's hit distance -- with that candidate's visit index in its low mantissa bits (FiltState) --
// and the second-smallest lower bound.
#ifndef B2PT_FILT_UNROLL
#define B2PT_FILT_UNROLL 1
#endif
constexpr int kFiltUnroll = B2PT_FILT_UNROLL;
struct FiltState
{
  uint32_t mask; // candidates in visit order, shifted in from the right
  // Smallest and second smallest KEY over the candidates.  A key is a lower bound of the candidate's hit distance with
  // the candidate's visit index in its five lowest mantissa bits (kFiltKeyBits): the running minimum then carries the
  // index of the nearest candidate along, and the loop needs no compare-and-select for it.  Replacing the low bits
  // moves the value by less than 32 ulp (3.7e-6 relative); the bound is lowered by 8e-6 relative beforehand (cLo in
  // filt_axis), so a key is still a lower bound.  Non-candidates get kFiltNoKey, a finite value above every distance.
  float tbl;
  float t2;
};
constexpr uint32_t kFiltKeyBits = 31u;          // B2PT_MAX_FILT = 32 visit indices
constexpr uint32_t kFiltNoKey = 0x7f7fffe0u;    // 3.4028e38, low bits free for the index
__device__ __forceinline__ float filt_key(float lowerBound, int visit)
{
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, 0xea;" : "=r"(r) : "r"(__float_as_uint(lowerBound)), "r"(~kFiltKeyBits), "r"((uint32_t)visit));
  return __uint_as_float(r); // (a & b) | c
}
__device__ __forceinline__ float rcp_fast(float x)
{
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// packed pairs of floats in one 64-bit register (sm_100 FFMA2 / FADD2)
typedef unsigned long long f2x;
__device__ __forceinline__ f2x pk2(float lo, float hi)
{
  f2x r;
  asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(f2x v, float& lo, float& hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2x fma2(f2x a, f2x b, f2x c)
{
  f2x r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f2x add2(f2x a, f2x b)
{
  f2x r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f2x sub2(f2x a, f2x b)
{
  f2x r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// One axis group: pairs [pBegin,pEnd) hold quads normal to the frame axis whose ray components are (on,dn);
// (ou,du),(ov,dv) are the components on the two other axes.  Error model (u = 2^-24, S = coordinate scale,
// D = |d|_1/|dn| >= 1): the filter's t' = c*rcp(dn) - on*rcp(dn) and the exact test's t both lie within
// t*(4e-6*D) + 4e-6*S/|dn|  of the true plane distance (>= 20x the forward error of either evaluation, incl. the
// rotation into the frame), and the hit point within  S*(2e-5 + 2e-5*D)  of the true one plus the exact test's
// own edge tolerance (static part folded into hu/hv on the host).  A quad the exact test could accept therefore
// always passes.  The absolute part 4e-6*S/|dn| is dominated by the rotation into a frame and by quads whose plane
// offsets differ by up to 1e-6*S; for a world-frame group of exactly planar quads it is eaCoef = 4e-7 (B2Frame): with
// E01_n = E03_n = 0 and v00_n = c the exact test's t = (T_n A)/(d_n A') carries only relative rounding (<= 10 u), and
// t' = fma(c, r, -(on r)) with r = rcp.approx(dn) (1 ulp) differs from the true distance by at most 3 u |t| +
// u |on| |r| <= 1.8e-7 |t| + 6e-8 S/|dn|.
__device__ __forceinline__ void filt_axis(const B2SmallScene& S, uint32_t byteBegin, uint32_t byteEnd, float on, float dn,
                                          float ou, float du, float ov, float dv, float dabs, float Sr, float eaCoef,
                                          float tmin, FiltState& F)
{
  if (byteEnd == byteBegin)
    return;
  const float inf = __int_as_float(0x7f800000);
  const bool axisOk = fabsf(dn) > 1e-30f; // below that the exact test rejects on |det| < 1e-5
  const float rdn = rcp_fast(dn);
  const float odn = on * rdn;
  const float D = dabs * fabsf(rdn);
  const float marg = Sr * __fmaf_rn(2e-5f, D, 2e-5f);
  const float er = 4e-6f * D;               // relative error bound of t' (and of the exact t)
  const float ea = eaCoef * Sr * fabsf(rdn); // absolute part (B2Frame::eaCoef: 4e-6, exactly planar world-frame groups 4e-7)
  // candidate iff  t' + |t'|*er + ea > tmin  (upper bound of the true distance beyond tmin); as a threshold on t':
  const float bt = tmin - ea;
  // (bt > 0: t' > bt/(1+er), bounded below by bt*(1-2er); bt <= 0: t' > bt/(1-er), bounded below by bt*(1+2er) while
  // er < 0.5 -- one branch-free form, bt - 2er*|bt|, covers both signs)
  // (two selects written as PTX: left to itself the compiler wraps the threshold arithmetic in a branch)
  float tlo = __fmaf_rn(-2.0f * er, fabsf(bt), bt);
  asm("{ .reg .pred p; setp.ne.s32 p, %2, 0; selp.f32 %0, %0, %1, p; }" : "+f"(tlo) : "f"(-inf), "r"((int)(er < 0.5f)));
  asm("{ .reg .pred p; setp.ne.s32 p, %2, 0; selp.f32 %0, %0, %1, p; }" : "+f"(tlo) : "f"(inf), "r"((int)axisOk));
  // lower bound of the true distance used for ordering / pruning:  t'*(1-er) - 3*ea  (valid for either sign of t'
  // that passes the threshold); extreme grazing (er >= 0.5) gets -inf, i.e. is never pruned
  // (8e-6: room for the visit index in the low bits of the bound, FiltState; 3e38 instead of infinity keeps the key finite)
  const float cLo = er < 0.5f ? 0.999992f - er : 0.f;
  const float off = er < 0.5f ? 3.0f * ea : 3e38f;
  const f2x rdn2 = pk2(rdn, rdn), modn2 = pk2(-odn, -odn), du2 = pk2(du, du), ou2 = pk2(ou, ou), dv2 = pk2(dv, dv),
            ov2 = pk2(ov, ov), marg2 = pk2(marg, marg), cLo2 = pk2(cLo, cLo), moff2 = pk2(-off, -off);
  const char* const pairs0 = reinterpret_cast<const char*>(S.pairs);
  const ulonglong2* P = reinterpret_cast<const ulonglong2*>(pairs0 + byteBegin);
  const ulonglong2* const Pend = reinterpret_cast<const ulonglong2*>(pairs0 + byteEnd);
#pragma unroll kFiltUnroll
  for (; P != Pend; P += 3)
  {
    const ulonglong2 a = P[0];  // (c0,c1) (uc0,uc1)
    const ulonglong2 b = P[1];  // (hu0,hu1) (vc0,vc1)
    const ulonglong2 cc = P[2]; // (hv0,hv1) (vis0,vis1)
    const f2x hv2 = cc.x;
    const f2x tp2 = fma2(a.x, rdn2, modn2);
    const f2x eu2 = sub2(fma2(tp2, du2, ou2), a.y), ev2 = sub2(fma2(tp2, dv2, ov2), b.y);
    const f2x hu2 = add2(b.x, marg2), hw2 = add2(hv2, marg2);
    const f2x tl2 = fma2(tp2, cLo2, moff2);
    float tp0, tp1, eu0, eu1, ev0, ev1, hu0, hu1, hw0, hw1, tl0, tl1;
    upk2(tp2, tp0, tp1), upk2(eu2, eu0, eu1), upk2(ev2, ev0, ev1), upk2(hu2, hu0, hu1), upk2(hw2, hw0, hw1);
    upk2(tl2, tl0, tl1);
    const bool pass0 = (tp0 > tlo) & (fabsf(eu0) <= hu0) & (fabsf(ev0) <= hw0); // no short circuit
    const bool pass1 = (tp1 > tlo) & (fabsf(eu1) <= hu1) & (fabsf(ev1) <= hw1);
    const float noKey = __uint_as_float(kFiltNoKey);
    const float l0 = filt_key(pass0 ? tl0 : noKey, (int)(uint32_t)cc.y), l1 = filt_key(pass1 ? tl1 : noKey, (int)(uint32_t)(cc.y >> 32));
    F.t2 = fminf(F.t2, fmaxf(F.tbl, l0));
    F.tbl = fminf(F.tbl, l0);
    F.t2 = fminf(F.t2, fmaxf(F.tbl, l1));
    F.tbl = fminf(F.tbl, l1);
    // (mask = mask*4 + 2*pass0 + pass1 as one shift and two predicated ORs; the compiler's own form is two selects,
    // a multiply-add and an add)
    uint32_t m;
    asm("{ .reg .pred p0, p1; setp.ne.s32 p0, %2, 0; setp.ne.s32 p1, %3, 0; shl.b32 %0, %1, 2; @p0 or.b32 %0, %0, 2; "
        "@p1 or.b32 %0, %0, 1; }"
        : "=&r"(m)
        : "r"(F.mask), "r"((int)pass0), "r"((int)pass1));
    F.mask = m;
  }
}
__device__ __forceinline__ void filt_frame(const B2SmallScene& S, int f, int& pBegin, f3 o, f3 d, float Sr, float tmin,
                                           FiltState& F)
{
  const B2Frame& Fr = S.frames[f];
  f3 ol = o, dl = d;
  float Sf = Sr;
  if (!Fr.identity)
  {
    const f3 r = mk3(o.x - Fr.org[0], o.y - Fr.org[1], o.z - Fr.org[2]);
    ol = mk3(__fmaf_rn(Fr.R[0], r.x, __fmaf_rn(Fr.R[1], r.y, Fr.R[2] * r.z)),
             __fmaf_rn(Fr.R[3], r.x, __fmaf_rn(Fr.R[4], r.y, Fr.R[5] * r.z)),
             __fmaf_rn(Fr.R[6], r.x, __fmaf_rn(Fr.R[7], r.y, Fr.R[8] * r.z)));
    dl = mk3(__fmaf_rn(Fr.R[0], d.x, __fmaf_rn(Fr.R[1], d.y, Fr.R[2] * d.z)),
             __fmaf_rn(Fr.R[3], d.x, __fmaf_rn(Fr.R[4], d.y, Fr.R[5] * d.z)),
             __fmaf_rn(Fr.R[6], d.x, __fmaf_rn(Fr.R[7], d.y, Fr.R[8] * d.z)));
    Sf = 4.0f * Sr; // frame coordinates are relative to org: |.| <= 2*sqrt(3)*Sr
  }
  const float dabs = fabsf(dl.x) + fabsf(dl.y) + fabsf(dl.z);
  filt_axis(S, Fr.grpBegin[0], Fr.grpEnd[0], ol.x, dl.x, ol.y, dl.y, ol.z, dl.z, dabs, Sf, Fr.eaCoef[0], tmin, F);
  filt_axis(S, Fr.grpBegin[1], Fr.grpEnd[1], ol.y, dl.y, ol.z, dl.z, ol.x, dl.x, dabs, Sf, Fr.eaCoef[1], tmin, F);
  filt_axis(S, Fr.grpBegin[2], Fr.grpEnd[2], ol.z, dl.z, ol.x, dl.x, ol.y, dl.y, dabs, Sf, Fr.eaCoef[2], tmin, F);
  pBegin = max(pBegin, Fr.axisEnd[2]);
}

// Closest hit over a kernel-parameter-resident scene.  MapperPathTracer.cxx:410-435: quads first
// (QuadIntersector.cxx:59-71), then spheres continuing from the quads' closest distance
// (SphereIntersector.cxx:88-100).  The reference's strict t<tmax keeps the first-tested primitive on an
// exact-t tie; quads are tested here in a different order (filter candidates nearest first, then boxed quads),
// so a tie is resolved explicitly in favour of the lower original index -- the same winner as index order.
#define B2PT_MISS 0x7fffffff
#ifdef B2PT_DEBUG_HIST
// experiment builds only (scripts/build_variant.sh hist -DB2PT_DEBUG_HIST): per-ray counts of the two-phase filter
__device__ unsigned long long g_debugHist[256];
#endif
__device__ __forceinline__ int closest_small(const B2SmallScene& S, f3 o, f3 d, float tmin, float tmax, float& tHit,
                                             bool withSpheres = true)
{
  float closest = tmax;
  int slot = -1;
  int bestPrim = 0x7fffffff;
  auto test_quad = [&](int q) {
    const B2Quad& Q = S.quads[q];
    float t;
    if (quad_hit(Q, o, d, t) && t > tmin && (t < closest || (t == closest && Q.prim < bestPrim)))
    {
      closest = t;
      slot = q;
      bestPrim = Q.prim;
    }
  };
  // ---- phase 1: candidate filter over the frame-aligned planar quads (uniform control flow)
  if (S.nFilt > 0)
  {
    FiltState F;
    F.mask = 0u;
    F.tbl = F.t2 = __int_as_float(0x7f800000);
    const float Sr = fmaxf(S.sceneAbs, fmaxf(fabsf(o.x), fmaxf(fabsf(o.y), fabsf(o.z))));
    int pBegin = 0;
    for (int f = 0; f < S.nFrames; ++f)
      filt_frame(S, f, pBegin, o, d, Sr, tmin, F);
    // ---- phase 2: the reference's exact test on the candidates, nearest lower bound first.  Every other
    // candidate's exact t is >= its lower bound >= t2, so once the nearest one is accepted with closest < t2
    // none of them can win or tie.  Visit index v sits at mask bit nVisit-1-v.
    uint32_t rest = F.mask;
    const int top = S.nVisit - 1;
    int v = (int)(__float_as_uint(F.tbl) & kFiltKeyBits); // nearest candidate (meaningful when rest != 0)
#ifdef B2PT_DEBUG_HIST
    int iters = 0;
    atomicAdd(&g_debugHist[__popc(rest) < 15 ? __popc(rest) : 15], 1ull); // [0..15]: candidates per ray
#endif
    while (rest)
    {
      rest &= ~(1u << (top - v));
#ifdef B2PT_DEBUG_HIST
      const int slotBefore = slot;
      // [64+v]: first exact test on visit index v; [96+v]: ... that failed; [128+v]: later tests on v; [160+v]: ... that
      // won; [192+v]: first test on v hit, but another candidate's lower bound kept the loop going
      atomicAdd(&g_debugHist[(iters == 0 ? 64 : 128) + v], 1ull);
#endif
      test_quad(S.visitSlot[v]);
#ifdef B2PT_DEBUG_HIST
      if (iters == 0 && slot < 0)
        atomicAdd(&g_debugHist[96 + v], 1ull);
      if (iters > 0 && slot != slotBefore)
        atomicAdd(&g_debugHist[160 + v], 1ull);
      if (iters == 0 && slot >= 0 && rest && !(F.t2 > closest))
        atomicAdd(&g_debugHist[192 + v], 1ull);
      ++iters;
#endif
      if (slot >= 0 && F.t2 > closest) // valid from the first iteration on: the nearest candidate is tested first
        break;
      v = top - (__ffs((int)rest) - 1);
    }
#ifdef B2PT_DEBUG_HIST
    atomicAdd(&g_debugHist[16 + (iters < 15 ? iters : 15)], 1ull); // [16..31]: exact tests per ray
    atomicAdd(&g_debugHist[32 + (slot >= 0 ? 1 : 0)], 1ull);       // [32],[33]: filtered quads gave no hit / a hit
#endif
  }
  // ---- remaining quads behind the slab test of their own leaf box (BVHTraverser.h:35-79, 143-157), then the
  // spheres behind theirs (sphere_gate)
  const int nSph = withSpheres ? S.nSph : 0;
  if (S.firstBoxed < S.nQuads || nSph > 0)
  {
    const f3 inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
    const f3 od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
    for (int q = S.firstBoxed; q < S.nQuads; ++q)
    {
      const B2Quad& Q = S.quads[q];
      float tn, t;
      if (!slab_hit(S.gate[Q.gate - 1].bmin, S.gate[Q.gate - 1].bmax, inv, od, tmin, closest, tn))
        continue;
      // non-planar quads (pad[0] != 0) come last and only win with a strictly smaller t, like the oracle
      if (quad_hit(Q, o, d, t) && t > tmin &&
          (t < closest || (t == closest && Q.pad[0] == 0 && Q.prim < bestPrim)))
      {
        closest = t;
        slot = q;
        bestPrim = Q.prim;
      }
    }
    for (int s = 0; s < nSph; ++s)
    {
      float tn, t;
      if (slab_hit(S.sphGate[s].bmin, S.sphGate[s].bmax, inv, od, tmin, tmax, tn) &&
          sphere_accept(ld3(S.sph[s].c), S.sph[s].r, o, d, tmin, closest, t))
      {
        closest = t;
        slot = S.nQuads + s;
      }
    }
  }
  tHit = closest;
  return slot < 0 ? B2PT_MISS : slot;
}
// ---- primary rays: quad_hit with the origin-dependent terms read from B2PrimQuad (same operations in the same order
// as quad_hit, so the outcome and t are bit-identical), and the closest hit over a tile's candidate mask.
__device__ __forceinline__ bool quad_hit_primary(const B2Quad& Q, const B2PrimQuad& C, f3 o, f3 d, float& t)
{
  const float4* q4 = reinterpret_cast<const float4*>(&Q);
  const float4 c0 = q4[0], c1 = q4[1], c2 = q4[2]; // v00 e01 | e01 e03 | e03 v11
  const float4 k0 = reinterpret_cast<const float4*>(&C)[0], k1 = reinterpret_cast<const float4*>(&C)[1];
  const f3 E03 = mk3(c1.z, c1.w, c2.x);
  f3 P = cross3(d, E03);
  const f3 E01 = mk3(c0.w, c1.x, c1.y);
  float det = dot3(E01, P);
  if (fabsf(det) < 1e-5f)
    return false;
  float inv_det = 1.0f / det;
  const f3 T = mk3(k0.x, k0.y, k0.z);
  float alpha = dot3(T, P) * inv_det;
  if (alpha < 0.0f)
    return false;
  const f3 Qv = mk3(k1.x, k1.y, k1.z);
  float beta = dot3(d, Qv) * inv_det;
  if (beta < 0.0f)
    return false;
  if ((alpha + beta) > 1.0f)
  {
    const float need = k1.w * ((fabsf(d.x) + fabsf(d.y)) + fabsf(d.z)) * Q.secC2;
    if (!((1.0f - fmaxf(alpha, beta)) * fabsf(det) > need && fabsf(det) >= 2e-5f))
    { // near an edge / general quad: the reference's second-triangle arithmetic as written (see quad_hit)
      const float4 c3 = q4[3], c4 = q4[4];
      const f3 E23 = mk3(c3.w, c4.x, c4.y);
      const f3 E21 = mk3(c3.x, c3.y, c3.z);
      f3 Pp = cross3(d, E21);
      float detp = dot3(E23, Pp);
      if (fabsf(detp) < 1e-5f)
        return false;
      float inv_detp = 1.0f / detp;
      f3 Tp = o - mk3(c2.y, c2.z, c2.w);
      float alphap = dot3(Tp, Pp) * inv_detp;
      if (alphap < 0.0f)
        return false;
      f3 Qp = cross3(Tp, E23);
      float betap = dot3(d, Qp) * inv_detp;
      if (betap < 0.0f)
        return false;
    }
  }
  t = k0.w * inv_det;
  if (t < 0.0f)
    return false;
  return true;
}
// Closest hit of a primary ray over the candidates of its tile.  The exact tests run on a SUPERSET of the quads the
// per-ray filter of closest_small would keep, the winner is "smallest t, exact ties to the lowest original index"
// either way, boxed quads and spheres follow with the same rules, so the result equals closest_small's bit for bit.
__device__ __forceinline__ int closest_small_masked(const B2SmallScene& S, const B2PrimQuad* __restrict__ pq, uint2 mask,
                                                    f3 o, f3 d, float tmin, float tmax, float& tHit)
{
  float closest = tmax;
  int slot = -1;
  int bestPrim = 0x7fffffff;
  for (uint32_t m = mask.x; m; m &= m - 1u) // warp-uniform loop: the mask belongs to the tile
  {
    const int q = S.visitSlot[__ffs((int)m) - 1];
    const B2Quad& Q = S.quads[q];
    const B2PrimQuad C = pq[q];
    float t;
    if (quad_hit_primary(Q, C, o, d, t) && t > tmin && (t < closest || (t == closest && Q.prim < bestPrim)))
    {
      closest = t;
      slot = q;
      bestPrim = Q.prim;
    }
  }
  if (mask.y)
  {
    const f3 inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
    const f3 od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
    for (int q = S.firstBoxed; q < S.nQuads; ++q)
    {
      const B2Quad& Q = S.quads[q];
      if (!((mask.y >> (Q.gate - 1)) & 1u))
        continue;
      float tn, t;
      if (!slab_hit(S.gate[Q.gate - 1].bmin, S.gate[Q.gate - 1].bmax, inv, od, tmin, closest, tn))
        continue;
      if (quad_hit(Q, o, d, t) && t > tmin && (t < closest || (t == closest && Q.pad[0] == 0 && Q.prim < bestPrim)))
      {
        closest = t;
        slot = q;
        bestPrim = Q.prim;
      }
    }
    for (int s = 0; s < S.nSph; ++s)
    {
      if (!((mask.y >> (B2PT_PRIM_SPH_SHIFT + s)) & 1u))
        continue;
      float tn, t;
      if (slab_hit(S.sphGate[s].bmin, S.sphGate[s].bmax, inv, od, tmin, tmax, tn) &&
          sphere_accept(ld3(S.sph[s].c), S.sph[s].r, o, d, tmin, closest, t))
      {
        closest = t;
        slot = S.nQuads + s;
      }
    }
  }
  tHit = closest;
  return slot < 0 ? B2PT_MISS : slot;
}
// Hit record of the winning primitive (Surface.h:180-192, :334-345): point, normal, material.
__device__ __forceinline__ void fill_small(const B2SmallScene& S, int slot, f3 o, f3 d, float closest, Hit& h)
{
  h.t = closest;
  h.p = o + d * closest; // Surface.h:187, :334
  if (slot < S.nQuads)
  {
    const B2Quad& Q = S.quads[slot];
    h.n = quad_normal(Q, d);
    h.alb = ld3(Q.alb);
    h.kind = Q.kind;
    h.prim = Q.prim;
    h.mat = Q.mat;
    h.texi = Q.texi;
  }
  else
  {
    const B2Sphere& SP = S.sph[slot - S.nQuads];
    f3 c = ld3(SP.c);
    h.n = mk3((h.p.x - c.x) / SP.r, (h.p.y - c.y) / SP.r, (h.p.z - c.z) / SP.r); // Surface.h:340
    h.alb = ld3(SP.alb);
    h.kind = SP.kind;
    h.prim = SP.prim;
    h.mat = SP.mat;
    h.texi = SP.texi;
  }
}

// Closest hit by stack traversal of the 32-byte-node BVH (one tree for quads and spheres).  A stack entry
// packs (leaf count << 24 | first child / first slot), so a node's own 32 bytes are never re-read: an inner
// visit is one 64-byte fetch of the adjacent child pair (4 x LDG.128).  Leaves test primitives in ascending
// original index, so exact-t ties resolve like brute force within a leaf; across leaves the nearer child is
// visited first (BVHTraverser.h:189-201).
__device__ __forceinline__ uint32_t bvh_pack(float leftBits, float countBits)
{
  return ((uint32_t)__float_as_int(countBits) << 24) | (uint32_t)__float_as_int(leftBits);
}
// withSpheres = false skips the sphere entries of the leaves (the -direct G-buffers see quads only).
// tiesToLowestIndex = true: an exact-t tie between quads of different leaves goes to the lower quad index, as in
// closest_small and the oracle, instead of to the leaf visited first -- the hit no longer depends on the tree's shape
// (quads only: use with withSpheres = false).
__device__ __forceinline__ int closest_bvh(const B2BvhScene& S, f3 o, f3 d, float tmin, float tmax, float& tHit,
                                           bool withSpheres = true, bool tiesToLowestIndex = false)
{
  f3 inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
  f3 od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
  float closest = tmax;
  int best = 0;
  bool found = false;
  uint32_t stack[64];
  int sp = 0;
  const float4* root = reinterpret_cast<const float4*>(S.nodes);
  uint32_t cur = S.nNodes > 0 ? bvh_pack(__ldg(root).w, __ldg(root + 1).w) : 0u;
  while (S.nNodes > 0)
  {
    const uint32_t count = cur >> 24;
    const uint32_t left = cur & 0xffffffu;
    if (count)
    {
      for (uint32_t k = 0; k < count; ++k)
      {
        const int enc = __ldg(S.primSlots + left + k);
        float t;
        if (enc >= 0)
        {
          const bool accept = tiesToLowestIndex
            ? quad_hit(S.quads[enc], o, d, t) && t > tmin && (t < closest || (t == closest && enc < best))
            : quad_accept(S.quads[enc], o, d, tmin, closest, t);
          if (accept)
          {
            closest = t;
            best = enc;
            found = true;
          }
        }
        else if (withSpheres)
        {
          const float4 cr = __ldg(reinterpret_cast<const float4*>(S.sph + (~enc)));
          if (sphere_may_hit(mk3(cr.x, cr.y, cr.z), cr.w, o, d) &&
              sphere_gate(mk3(cr.x, cr.y, cr.z), cr.w, inv, od, tmin, tmax) &&
              sphere_accept(mk3(cr.x, cr.y, cr.z), cr.w, o, d, tmin, closest, t))
          {
            closest = t;
            best = enc;
            found = true;
          }
        }
      }
      if (sp == 0)
        break;
      cur = stack[--sp];
    }
    else
    {
      const float4* lp = reinterpret_cast<const float4*>(S.nodes + left);
      const float4 l0 = __ldg(lp), l1 = __ldg(lp + 1), r0 = __ldg(lp + 2), r1 = __ldg(lp + 3);
      float tl, tr;
      const float lmin[3] = { l0.x, l0.y, l0.z }, lmax[3] = { l1.x, l1.y, l1.z };
      const float rmin[3] = { r0.x, r0.y, r0.z }, rmax[3] = { r1.x, r1.y, r1.z };
      const bool hl = slab_hit(lmin, lmax, inv, od, tmin, closest, tl);
      const bool hr = slab_hit(rmin, rmax, inv, od, tmin, closest, tr);
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
      else
      {
        if (sp == 0)
          break;
        cur = stack[--sp];
      }
    }
  }
  // Non-planar quads are kept out of the tree and tested last, each behind the slab test of its own leaf box
  // with the closest distance of everything else: the acceptance rule of the reference's near-first
  // traversal, independent of tree topology (DESIGN.md "leaf-box gate").
  for (int g = 0; g < S.nGate; ++g)
  {
    float tn, t;
    if (!slab_hit(S.gate[g].bmin, S.gate[g].bmax, inv, od, tmin, closest, tn))
      continue;
    const int q = S.gate[g].quad;
    if (quad_accept(S.quads[q], o, d, tmin, closest, t))
    {
      closest = t;
      best = q;
      found = true;
    }
  }
  tHit = closest;
  return found ? best : B2PT_MISS;
}
__device__ __forceinline__ void fill_bvh(const B2BvhScene& S, int best, f3 o, f3 d, float closest, Hit& h)
{
  h.t = closest;
  h.p = o + d * closest;
  if (best >= 0)
  {
    const B2Quad& Q = S.quads[best];
    h.n = quad_normal(Q, d);
    h.alb = ld3(Q.alb);
    h.kind = Q.kind;
    h.prim = Q.prim;
    h.mat = Q.mat;
    h.texi = Q.texi;
  }
  else
  {
    const B2Sphere& SP = S.sph[~best];
    f3 c = ld3(SP.c);
    h.n = mk3((h.p.x - c.x) / SP.r, (h.p.y - c.y) / SP.r, (h.p.z - c.z) / SP.r);
    h.alb = ld3(SP.alb);
    h.kind = SP.kind;
    h.prim = SP.prim;
    h.mat = SP.mat;
    h.texi = SP.texi;
  }
}

// ------------------------------------------------------------------------------ 8-wide compressed BVH (b2pt_wide.h)
// Traversal state of one ray over the wide tree.  A GROUP is a set of children of one node that still have to be
// visited: x = base index (childBase: inner children; primBase: primitive children), y = hit bits in visiting order
// (bit b = slot b XOR octant, ascending b = approximately front to back) | the node's inner / primitive slot mask << 8
// | kWidePrimGroup for a primitive group.  The stack holds groups of either kind.
constexpr uint32_t kWidePrimGroup = 0x10000u;
constexpr int kWideStack = B2PT_WIDE_STACK; // groups: at most one per level (build_trace_structures checks the depth)
struct WideTrav
{
  uint32_t nx, ny; // current node group (ny & 0xff == 0: none)
  uint32_t px, py; // current primitive group
  int sp;
};
// bit index b = s ^ oct within each byte of the low 16 bits
__device__ __forceinline__ uint32_t wide_perm(uint32_t m, uint32_t oct)
{
  if (oct & 1u)
    m = ((m & 0x5555u) << 1) | ((m >> 1) & 0x5555u);
  if (oct & 2u)
    m = ((m & 0x3333u) << 2) | ((m >> 2) & 0x3333u);
  if (oct & 4u)
    m = ((m & 0x0f0fu) << 4) | ((m >> 4) & 0x0f0fu);
  return m;
}
// Slab test of a node's eight quantised child boxes against the ray (culling arithmetic: FMA, conservative boxes).
// Dequantisation: PRMT drops byte q into the mantissa of 2^23, giving the float 2^23 + q exactly, and one FMA evaluates
// (2^23 + q) * (scale * inv) + (b - 2^23 * scale * inv): the constant's rounding error is at most half a quantisation
// step in t, which the builder's extra step of widening covers (b2pt_wide.h).  Returns the hit bits by SLOT.
__device__ __forceinline__ uint32_t wide_node_hits(const uint4* __restrict__ node, f3 inv, f3 od, float tmin, float closest,
                                                   uint32_t& childBase, uint32_t& primBase, uint32_t& innerMask,
                                                   uint32_t& primMask)
{
  const uint4 h0 = __ldg(node), h1 = __ldg(node + 1), qa = __ldg(node + 2), qb = __ldg(node + 3), qc = __ldg(node + 4);
  const uint32_t e = h0.w;
  childBase = h1.x;
  primBase = h1.y;
  innerMask = e >> 24;
  primMask = h1.z & 0xffu;
  const float six = __uint_as_float((e & 0xffu) << 23) * inv.x, siy = __uint_as_float(((e >> 8) & 0xffu) << 23) * inv.y,
              siz = __uint_as_float(((e >> 16) & 0xffu) << 23) * inv.z;
  const float bx = __fmaf_rn(-8388608.f, six, __fmaf_rn(__uint_as_float(h0.x), inv.x, -od.x));
  const float by = __fmaf_rn(-8388608.f, siy, __fmaf_rn(__uint_as_float(h0.y), inv.y, -od.y));
  const float bz = __fmaf_rn(-8388608.f, siz, __fmaf_rn(__uint_as_float(h0.z), inv.z, -od.z));
  // near / far plane bytes by the direction's sign: qlo = (qa.x qa.y | qa.z qa.w | qb.x qb.y), qhi = (qb.z qb.w | qc.x
  // qc.y | qc.z qc.w) for x | y | z
  const bool ngx = inv.x < 0.f, ngy = inv.y < 0.f, ngz = inv.z < 0.f;
  const uint32_t nx[2] = { ngx ? qb.z : qa.x, ngx ? qb.w : qa.y }, fx[2] = { ngx ? qa.x : qb.z, ngx ? qa.y : qb.w };
  const uint32_t ny[2] = { ngy ? qc.x : qa.z, ngy ? qc.y : qa.w }, fy[2] = { ngy ? qa.z : qc.x, ngy ? qa.w : qc.y };
  const uint32_t nz[2] = { ngz ? qc.z : qb.x, ngz ? qc.w : qb.y }, fz[2] = { ngz ? qb.x : qc.z, ngz ? qb.y : qc.w };
  uint32_t hits = 0u;
#pragma unroll
  for (int s = 0; s < 8; ++s)
  {
    const int w = s >> 2;
    const uint32_t sel = 0x7540u | (uint32_t)(s & 3);
    const float tnx = __fmaf_rn(__uint_as_float(__byte_perm(nx[w], 0x4B000000u, sel)), six, bx);
    const float tny = __fmaf_rn(__uint_as_float(__byte_perm(ny[w], 0x4B000000u, sel)), siy, by);
    const float tnz = __fmaf_rn(__uint_as_float(__byte_perm(nz[w], 0x4B000000u, sel)), siz, bz);
    const float tfx = __fmaf_rn(__uint_as_float(__byte_perm(fx[w], 0x4B000000u, sel)), six, bx);
    const float tfy = __fmaf_rn(__uint_as_float(__byte_perm(fy[w], 0x4B000000u, sel)), siy, by);
    const float tfz = __fmaf_rn(__uint_as_float(__byte_perm(fz[w], 0x4B000000u, sel)), siz, bz);
    const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmin));
    const float tf = fminf(fminf(tfx, tfy), fminf(tfz, closest));
    if (tn <= tf)
      hits |= 1u << s;
  }
  return hits;
}
// Exact test of the primitive in leaf-order slot `slot` (the reference's arithmetic; spheres behind their own leaf box,
// sphere_gate).  Winner rule = brute force in index order: smallest t, an exact tie to the lower primitive id -- so the
// result does not depend on the order in which the tree presents the primitives.
__device__ __forceinline__ void wide_test_prim(const B2BvhScene& S, uint32_t slot, f3 o, f3 d, f3 inv, f3 od, float tmin,
                                               float tmax, float& closest, int& best, int& bestId)
{
  const int enc = __ldg(S.primSlots + slot);
  float t = 0.f;
  bool h = false;
  if (enc >= 0)
    h = quad_hit(S.quads[enc], o, d, t) && t > tmin && t <= closest;
  else
  {
    const float4 g = __ldg(S.leafSph + slot);
    const f3 c = mk3(g.x, g.y, g.z);
    if (sphere_may_hit(c, g.w, o, d) && sphere_gate(c, g.w, inv, od, tmin, tmax))
    { // Surface.h:319-367 with the upper bound made inclusive (the tie rule below decides equality)
      const f3 oc = o - c;
      const float a = dot3(d, d), b = dot3(oc, d), cc = dot3(oc, oc) - g.w * g.w;
      const float disc = b * b - a * cc;
      if (disc > 0.f)
      {
        const float sq = sqrtf(b * b - a * cc);
        float temp = (-b - sq) / a;
        if (temp <= closest && temp > tmin)
          t = temp, h = true;
        else
        {
          temp = (-b + sq) / a;
          if (temp <= closest && temp > tmin)
            t = temp, h = true;
        }
      }
    }
  }
  const int id = enc >= 0 ? enc : S.nQuads + (~enc);
  if (h && (t < closest || id < bestId))
  {
    closest = t;
    best = enc;
    bestId = id;
  }
}
// One traversal step of a lane: if it holds a node group, visit that group's next child node (A); the caller then runs
// wide_step_prim for lanes holding a primitive group (B).  Returns false when the ray has nothing left.
__device__ __forceinline__ void wide_push(uint32_t* stackX, uint32_t* stackY, int& sp, uint32_t x, uint32_t y)
{
  if (sp < kWideStack)
  {
    stackX[sp] = x;
    stackY[sp] = y;
    ++sp;
  }
}
__device__ __forceinline__ void wide_start(WideTrav& R, uint32_t oct, bool any)
{
  // the root is "inner child 0 of a virtual node": one hit bit at the position slot 0 has for this octant
  R.nx = 0u;
  R.ny = any ? ((1u << 8) | (1u << oct)) : 0u;
  R.px = R.py = 0u;
  R.sp = 0;
}
// (A) visit the next child of the node group; new groups replace / are stacked as described in WideTrav
__device__ __forceinline__ void wide_step_node(const B2BvhScene& S, WideTrav& R, uint32_t* stackX, uint32_t* stackY, f3 inv,
                                               f3 od, uint32_t oct, float tmin, float closest)
{
  const uint32_t hb = R.ny & 0xffu;
  const uint32_t b = (uint32_t)__ffs((int)hb) - 1u;
  const uint32_t s = b ^ oct;
  const uint32_t child = R.nx + (uint32_t)__popc((R.ny >> 8) & 0xffu & ((1u << s) - 1u));
  R.ny &= ~(1u << b);
  if (R.ny & 0xffu)
    wide_push(stackX, stackY, R.sp, R.nx, R.ny);
  uint32_t childBase, primBase, innerMask, primMask;
  const uint32_t hits = wide_node_hits(S.wide + 5 * (size_t)child, inv, od, tmin, closest, childBase, primBase, innerMask,
                                       primMask);
  const uint32_t pm = wide_perm((hits & innerMask) | ((hits & primMask) << 8), oct);
  R.nx = childBase;
  R.ny = (innerMask << 8) | (pm & 0xffu);
  const uint32_t ph = pm >> 8;
  if (ph)
  {
    if (R.py & 0xffu) // (cannot happen: a lane holding a primitive group does not take step A)
      wide_push(stackX, stackY, R.sp, R.px, R.py);
    R.px = primBase;
    R.py = kWidePrimGroup | (primMask << 8) | ph;
  }
}
// (B) exact test of the next primitive of the primitive group
__device__ __forceinline__ void wide_step_prim(const B2BvhScene& S, WideTrav& R, f3 o, f3 d, f3 inv, f3 od, uint32_t oct,
                                               float tmin, float tmax, float& closest, int& best, int& bestId)
{
  const uint32_t hb = R.py & 0xffu;
  const uint32_t b = (uint32_t)__ffs((int)hb) - 1u;
  const uint32_t s = b ^ oct;
  const uint32_t slot = R.px + (uint32_t)__popc((R.py >> 8) & 0xffu & ((1u << s) - 1u));
  R.py &= ~(1u << b);
  wide_test_prim(S, slot, o, d, inv, od, tmin, tmax, closest, best, bestId);
}
// both groups empty: take the next group from the stack; returns false when the traversal is over
__device__ __forceinline__ bool wide_next(WideTrav& R, const uint32_t* stackX, const uint32_t* stackY)
{
  if ((R.ny & 0xffu) || (R.py & 0xffu))
    return true;
  if (R.sp == 0)
    return false;
  --R.sp;
  const uint32_t x = stackX[R.sp], y = stackY[R.sp];
  if (y & kWidePrimGroup)
    R.px = x, R.py = y;
  else
    R.nx = x, R.ny = y;
  return true;
}
__device__ __forceinline__ uint32_t wide_octant(f3 inv)
{
  return (inv.x < 0.f ? 1u : 0u) | (inv.y < 0.f ? 2u : 0u) | (inv.z < 0.f ? 4u : 0u);
}
// Closest hit of one ray (stage-level kernels; the bounce kernels use the persistent-lane form, trace_body_wide)
__device__ __forceinline__ int closest_wide(const B2BvhScene& S, f3 o, f3 d, float tmin, float tmax, float& tHit)
{
  const f3 inv = mk3(rcp_safe(d.x), rcp_safe(d.y), rcp_safe(d.z));
  const f3 od = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
  const uint32_t oct = wide_octant(inv);
  float closest = tmax;
  int best = 0, bestId = 0x7fffffff;
  uint32_t stackX[kWideStack], stackY[kWideStack];
  WideTrav R;
  wide_start(R, oct, S.nWide > 0);
  while (wide_next(R, stackX, stackY))
  {
    if (R.py & 0xffu)
      wide_step_prim(S, R, o, d, inv, od, oct, tmin, tmax, closest, best, bestId);
    else
      wide_step_node(S, R, stackX, stackY, inv, od, oct, tmin, closest);
  }
  bool found = bestId != 0x7fffffff;
  for (int g = 0; g < S.nGate; ++g)
  { // non-planar quads: after the traversal, each behind its own leaf box (DESIGN.md "leaf-box gate")
    float tn, t;
    if (!slab_hit(S.gate[g].bmin, S.gate[g].bmax, inv, od, tmin, closest, tn))
      continue;
    const int q = S.gate[g].quad;
    if (quad_accept(S.quads[q], o, d, tmin, closest, t))
    {
      closest = t;
      best = q;
      found = true;
    }
  }
  tHit = closest;
  return found ? best : B2PT_MISS;
}
__device__ __forceinline__ int closest_hit(const B2WideScene& S, f3 o, f3 d, float tmin, float tmax, float& t)
{
  return closest_wide(S, o, d, tmin, tmax, t);
}

__device__ __forceinline__ int closest_hit(const B2SmallScene& S, f3 o, f3 d, float tmin, float tmax, float& t)
{
  return closest_small(S, o, d, tmin, tmax, t);
}
__device__ __forceinline__ int closest_hit(const B2BvhScene& S, f3 o, f3 d, float tmin, float tmax, float& t)
{
  return closest_bvh(S, o, d, tmin, tmax, t);
}
__device__ __forceinline__ void fill_hit(const B2SmallScene& S, int code, f3 o, f3 d, float t, Hit& h)
{
  fill_small(S, code, o, d, t, h);
}
__device__ __forceinline__ void fill_hit(const B2BvhScene& S, int code, f3 o, f3 d, float t, Hit& h)
{
  fill_bvh(S, code, o, d, t, h);
}
// material kind (matType) of the primitive behind a closest-hit code
__device__ __forceinline__ int hit_kind(const B2SmallScene& S, int slot)
{
  return slot < S.nQuads ? S.quads[slot].kind : S.sph[slot - S.nQuads].kind;
}
__device__ __forceinline__ int hit_kind(const B2BvhScene& S, int code)
{
  return code >= 0 ? S.quads[code].kind : S.sph[~code].kind;
}
// closest hit + hit record in one call (stage-level kernels)
template <class SceneT>
__device__ __forceinline__ bool trace(const SceneT& S, f3 o, f3 d, float tmin, float tmax, Hit& h)
{
  float t;
  const int code = closest_hit(S, o, d, tmin, tmax, t);
  if (code == B2PT_MISS)
  {
    h.prim = -1;
    h.t = t;
    return false;
  }
  fill_hit(S, code, o, d, t, h);
  return true;
}

// ------------------------------------------------------------------------------------------ shading
struct Onb
{
  f3 u, v, w;
};
// onb.h:34-45
__device__ __forceinline__ Onb onb_from_w(f3 n)
{
  Onb o;
  o.w = unit3(n);
  f3 a = (fabsf(o.w.x) > 0.9f) ? mk3(0.f, 1.f, 0.f) : mk3(1.f, 0.f, 0.f);
  o.v = unit3(cross3(o.w, a));
  o.u = cross3(o.w, o.v);
  return o;
}
// onb.h:30-31
__device__ __forceinline__ f3 onb_local(const Onb& o, f3 a) { return (o.u * a.x + o.v * a.y) + o.w * a.z; }

#define B2PT_TWO_PI_D 6.283185307179586476925286766559
#define B2PT_INV_PI_F 0.31830988618379067154f

// PdfWorklet.h:47-53: z=sqrt(1-r2), phi=2*Pi()*r1 (Float64 product narrowed), x,y carry the reference's 2*sqrt(r2)
__device__ __forceinline__ f3 random_cosine_direction(float r1, float r2)
{
  float z = sqrtf(1.f - r2);
  float phi = (float)(B2PT_TWO_PI_D * (double)r1);
  float sp, cp;
  sincosf(phi, &sp, &cp);
  float s2 = sqrtf(r2);
  return mk3(cp * 2.f * s2, sp * 2.f * s2, z);
}
// PdfWorklet.h:157-165
__device__ __forceinline__ f3 random_to_sphere(float radius, float dist2, float r1, float r2)
{
  float z = 1.f + r2 * (sqrtf(1.f - radius * radius / dist2) - 1.f);
  float phi = (float)(B2PT_TWO_PI_D * (double)r1);
  float sp, cp;
  sincosf(phi, &sp, &cp);
  float s = sqrtf(1.f - z * z);
  return mk3(cp * s, sp * s, z);
}

// PdfWorklet.h:230-248 (QuadPDFWorklet::pdf_value) against one light quad.
__device__ __forceinline__ float quad_pdf_value(const B2LightQuad& L, f3 o, f3 v)
{
  float t;
  bool h;
  if (L.aa.cls >= 0)
  { // axis-aligned light quad: bit-identical specialised test (warp-uniform branch)
    float du, dv, dn, ou, ov, on;
    aa_permute(L.aa.cls, v, du, dv, dn);
    aa_permute(L.aa.cls, o, ou, ov, on);
    h = aa_quad_hit(L.aa, du, dv, dn, ou, ov, on, t);
  }
  else
    h = quad_hit(L.geo, o, v, t);
  if (!(h && t < FLT_MAX && t > 0.001f))
    return 0.f;
  f3 n = quad_normal(L.geo, v);
  float dist2 = t * t * dot3(v, v);
  float cosine = fabsf(dot3(v, n) * rmag3_fast(v));
  return div_fast(dist2, cosine * L.area);
}
// PdfWorklet.h:333-347 (SpherePDFWorklet::pdf_value)
__device__ __forceinline__ float sphere_pdf_value(const B2LightSphere& L, f3 o, f3 v)
{
  float t;
  f3 c = ld3(L.c);
  if (!sphere_accept(c, L.r, o, v, 0.001f, FLT_MAX, t))
    return 0.f;
  f3 co = c - o;
  float cos_theta_max = sqrtf(1.f - div_fast(L.r * L.r, dot3(co, co)));
  float solid_angle = 6.28318530717958647692f * (1.f - cos_theta_max);
  return div_fast(1.f, solid_angle);
}

// EmitWorklet.h:152-226 (DielectricWorklet): returns the specular direction (reflect or refract).
__device__ __noinline__ f3 dielectric_scatter(f3 dir, f3 n, float refIdx, float rnd)
{
  float dn = dot3(dir, n);
  f3 reflected = dir - n * (2.f * dn);
  f3 outward;
  float ni_over_nt, cosine;
  if (dn > 0.f)
  {
    outward = -n;
    ni_over_nt = refIdx;
    cosine = refIdx * dn * rmag3(dir);
  }
  else
  {
    outward = n;
    ni_over_nt = (float)(1.0 / (double)refIdx);
    cosine = -dn * rmag3(dir);
  }
  f3 uv = unit3(dir);
  float dt = dot3(uv, outward);
  float disc = (float)(1.0 - (double)(ni_over_nt * ni_over_nt * (1.f - dt * dt)));
  float reflect_prob = 1.0f;
  f3 refracted = mk3(0.f, 0.f, 0.f);
  if (disc > 0.f)
  {
    refracted = (uv - outward * dt) * ni_over_nt - outward * sqrtf(disc);
    float r0 = (1.f - refIdx) / (1.f + refIdx);
    r0 = r0 * r0;
    double x = (double)(1.f - cosine);
    double x2 = x * x;
    reflect_prob = (float)((double)r0 + (double)(1.f - r0) * (x2 * x2 * x)); // schlick, pow(x,5)
  }
  return (rnd < reflect_prob) ? reflected : refracted;
}

enum BounceResult
{
  BOUNCE_CONTINUE = 0,
  BOUNCE_DONE = 1
};

// Lambertian bounce: strategy choice, direction generator, light pdfs, mixture pdf, throughput, next ray
// (PdfWorklet.h:19-21, 63-79, 112-137, 193-213, 274-316, 374-399; ScatterWorklet.h:67-117).
// `which` is re-drawn here from the path's RNG state; when the caller binned rays by strategy (k_trace) it is
// the same for the whole warp and the three generator branches do not diverge.
__device__ __forceinline__ BounceResult shade_lambert(const B2Lights& lights, const Hit& hit, f3& o, f3& d, f3& T,
                                                      uint32_t& rng, uint32_t flags, f3& L)
{
  const int which = draw_which(rng);
  // The generators overwrite `generated` once per light (PdfWorklet.h:112-137, 193-213), so only the LAST light's
  // direction survives; the earlier lights only consume their draws.  The cosine and the sphere generator share one
  // copy of the frame construction and the sincos: local = (cos(phi)*m*s, sin(phi)*m*s, z) around w, with
  // (m, s, z, w) = (2, sqrt(r2), sqrt(1-r2), n) resp. (1, sqrt(1-z*z), 1+r2*(sqrt(1-R*R/d2)-1), c-p); m = 1 multiplies
  // exactly, so both evaluate the reference's operation sequence (PdfWorklet.h:47-53, 157-165).
  f3 g = mk3(0.f, 0.f, 0.f);
  if (which == 2)
  {
    if (lights.nLightQuads > 0)
    {
      for (int k = 0; k < 3 * (lights.nLightQuads - 1); ++k)
        wang32(rng);
      const B2LightQuad& LQ = lights.lq[lights.nLightQuads - 1];
      float r1 = randf(rng);
      float r2 = randf(rng);
      float r3 = randf(rng);
      float y0 = LQ.pt1[1];
      f3 rp = mk3(LQ.pt1[0] + r1 * (LQ.pt2[0] - LQ.pt1[0]), y0 + r2 * (y0 - y0), LQ.pt1[2] + r3 * (LQ.pt2[2] - LQ.pt1[2]));
      g = rp - hit.p;
    }
  }
  else if (which <= 1 || lights.nLightSph > 0)
  {
    float r1, r2, z, s, m;
    f3 w;
    if (which <= 1)
    {
      r1 = randf(rng);
      r2 = randf(rng);
      w = hit.n;
      z = sqrtf(1.f - r2);
      s = sqrtf(r2);
      m = 2.f;
    }
    else
    {
      for (int k = 0; k < 2 * (lights.nLightSph - 1); ++k)
        wang32(rng);
      // PdfWorklet.h:210: argument evaluation order of GCC x86-64 (right to left): r2 is drawn first
      r2 = randf(rng);
      r1 = randf(rng);
      const B2LightSphere& LS = lights.ls[lights.nLightSph - 1];
      w = ld3(LS.c) - hit.p;
      const float d2 = dot3(w, w);
      z = 1.f + r2 * (sqrtf(1.f - LS.r * LS.r / d2) - 1.f);
      s = sqrtf(1.f - z * z);
      m = 1.f;
    }
    const float phi = (float)(B2PT_TWO_PI_D * (double)r1);
    float sp, cp;
    sincosf(phi, &sp, &cp);
    const Onb uvw = onb_from_w(w);
    g = denan3(onb_local(uvw, mk3(cp * m * s, sp * m * s, z)));
  }
  wang32(rng); // SpherePDFWorklet's unused index draw (PdfWorklet.h:393)
  // light pdfs: sum = weight*quad + weight*sphere (no occlusion test in either)
  float sum = 0.f;
#pragma unroll
  for (int l = 0; l < B2PT_MAX_LIGHT_QUADS; ++l)
    if (l < lights.nLightQuads)
      sum += lights.weight * quad_pdf_value(lights.lq[l], hit.p, g);
#pragma unroll
  for (int l = 0; l < B2PT_MAX_LIGHT_SPH; ++l)
    if (l < lights.nLightSph)
      sum += lights.weight * sphere_pdf_value(lights.ls[l], hit.p, g);
  // ScatterWorklet.h:20-28, 52-58, 95-110
  f3 ug = unit3_fast(g);
  float cosw = dot3(ug, unit3_fast(hit.n));
  float value = (cosw > 0.f) ? cosw * B2PT_INV_PI_F : 0.f;
  float pdf_val = 0.5f * sum + 0.5f * value;
  float c2 = dot3(hit.n, ug);
  float spdf = (c2 < 0.f) ? 0.f : c2 * B2PT_INV_PI_F;
  float sctr = div_fast(spdf, pdf_val);
  T = mk3(T.x * (hit.alb.x * sctr), T.y * (hit.alb.y * sctr), T.z * (hit.alb.z * sctr));
  o = hit.p;
  d = g;
  if ((flags & B2PT_FLAG_KILL_ZERO_THROUGHPUT_DEV) && T.x == 0.f && T.y == 0.f && T.z == 0.f)
  {
    L = mk3(0.f, 0.f, 0.f);
    return BOUNCE_DONE;
  }
  return BOUNCE_CONTINUE;
}

// Specular (dielectric) bounce: DielectricWorklet (EmitWorklet.h:244-272): one draw, specular ray, attenuation 1.
// The direction generators and the sphere-pdf worklet still run for such a pixel and consume their draws (which 1,
// generator 2 / 3 per light quad / 2 per light sphere, pdf index 1); their outputs are unused.  Draw order while
// alive is the reference's (SURVEY A.3).  k_trace finishes misses and emitter hits itself, so k_shade only ever
// sees this case (bin 0) and the lambertian one (bins 1..3, shade_lambert).
__device__ __forceinline__ BounceResult shade_specular(const B2Lights& lights, const Hit& hit, f3& o, f3& d, uint32_t& rng)
{
  const float r = randf(rng);
  const f3 sdir = dielectric_scatter(d, hit.n, lights.refIdx, r);
  const int which = draw_which(rng);
  const int burn = (which <= 1) ? 2 : (which == 2 ? 3 * lights.nLightQuads : 2 * lights.nLightSph);
  for (int k = 0; k < burn + 1; ++k)
    wang32(rng);
  o = hit.p;
  d = sdir;
  return BOUNCE_CONTINUE;
}

} // namespace b2pt
#endif
