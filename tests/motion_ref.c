/*
 * motion_ref.c -- the motion vectors of b2pt_render_views_motion (include/b2pt.h, DESIGN.md 8i) restated on top of the
 * CPU oracle.  TEST INFRASTRUCTURE: built by tests/motion_ref.py, loaded only by tests.
 *
 * lens_ref.c (which compiles the oracle source unchanged) gives the primary ray of a sample, pinhole or lens, and the
 * oracle its camera basis and closest hit.  This file adds only the projection, the visibility ray and the sums:
 *   X = o + d*t;  proj(C, X): D = X - pos, w = D.nlook, x = (D.dx) / (w * (dx.dx)) + W*0.5, y likewise with dy, H;
 *   valid = w > 0 && w' > 0;  m = (x' - x, y' - y);
 *   visible = (x', y') on the canvas && the closest hit from pos' along (X - pos') nudged and normalised, L its
 *   magnitude, is absent or has t' >= L * (1 - 2^-12).
 */
#include "lens_ref.c"

/* proj(C, X) of the header; returns w */
static float project(const cam_basis* b, v3 X, float* x, float* y)
{
  const v3 D = vsub(X, b->pos);
  const float w = vdot(D, b->nlook);
  *x = vdot(D, b->dx) / (w * vdot(b->dx, b->dx)) + 0.5f * (float)b->W;
  *y = vdot(D, b->dy) / (w * vdot(b->dy, b->dy)) + 0.5f * (float)b->H;
  return w;
}

/* One sample of pixel idx from stream state seed.  out[0..7] = (x, y, x', y', w, w', visible, hit), out[8] = t;
 * returns 1 when the sample is valid (a hit in front of both cameras). */
int motion_sample(const orc_scene* sc, const orc_camera* cam, const orc_camera* prev, float aperture, float focus,
                  int64_t idx, uint32_t seed, float* out)
{
  const cam_basis b = make_basis(cam), bp = make_basis(prev);
  float o3[3], d3[3];
  lens_raygen(cam, aperture, focus, idx, &seed, o3, d3);
  for (int k = 0; k < 9; ++k)
    out[k] = 0.f;
  float rec[9];
  int hid[2];
  rec[HR_T] = FLT_MAX;
  if (closest_hit(sc, ld3(o3), ld3(d3), 0.001f, FLT_MAX, 0, rec, hid) < 0)
    return 0;
  const v3 o = ld3(o3), d = ld3(d3);
  const v3 X = vadd(o, vscale(d, rec[HR_T]));
  out[7] = 1.f;
  out[8] = rec[HR_T];
  out[4] = project(&b, X, &out[0], &out[1]);
  out[5] = project(&bp, X, &out[2], &out[3]);
  if (!(out[4] > 0.f && out[5] > 0.f))
    return 0;
  const float xp = out[2], yp = out[3];
  if (xp >= 0.f && xp < (float)b.W && yp >= 0.f && yp < (float)b.H)
  {
    v3 e = vsub(X, bp.pos);
    if (e.x == 0.f)
      e.x += 0.0000001f;
    if (e.y == 0.f)
      e.y += 0.0000001f;
    if (e.z == 0.f)
      e.z += 0.0000001f;
    const float L = sqrtf(vdot(e, e));
    e = V(e.x / L, e.y / L, e.z / L);
    rec[HR_T] = FLT_MAX;
    if (closest_hit(sc, bp.pos, e, 0.001f, FLT_MAX, 0, rec, hid) < 0 || rec[HR_T] >= L * 0.999755859375f)
      out[6] = 1.f;
  }
  return 1;
}

/* The sums of b2pt_render_views_motion for one view: out[k][j*W+i] float4 = (sum m.x, sum m.y, sum visible,
 * sum valid) over the valid samples s < checkpoints[k], in sample order from +0.0. */
int motion_sums(const orc_scene* sc, const orc_camera* cam, const orc_camera* prev, float aperture, float focus,
                uint32_t seedOffset, int nCheckpoints, const int* checkpoints, float* out)
{
  if (nCheckpoints < 1 || cam->W != prev->W || cam->H != prev->H)
    return -1;
  const int64_t N = (int64_t)cam->W * cam->H;
  const int last = checkpoints[nCheckpoints - 1];
#pragma omp parallel for schedule(dynamic, 64)
  for (int64_t i = 0; i < N; i++)
  {
    float sum[4] = { 0.f, 0.f, 0.f, 0.f };
    int k = 0;
    for (int s = 0; s < last; s++)
    {
      float r[9];
      if (motion_sample(sc, cam, prev, aperture, focus, i, (uint32_t)i + seedOffset + (uint32_t)s * ORC_GOLDEN, r))
      {
        sum[0] += r[2] - r[0];
        sum[1] += r[3] - r[1];
        sum[2] += r[6];
        sum[3] += 1.f;
      }
      if (s + 1 == checkpoints[k])
      {
        float* dst = out + 4 * ((int64_t)k * N + i);
        dst[0] = sum[0], dst[1] = sum[1], dst[2] = sum[2], dst[3] = sum[3];
        ++k;
      }
    }
  }
  return 0;
}
