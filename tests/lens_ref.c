/*
 * lens_ref.c -- the thin lens of b2pt_set_lens (include/b2pt.h, DESIGN.md 8h) restated on top of the CPU oracle.
 * TEST INFRASTRUCTURE: built by tests/lens_ref.py, loaded only by tests.
 *
 * The oracle source is compiled into this unit unchanged, so the lens reuses its own camera basis, pinhole raygen,
 * closest hit and forward path sampler (mode 3, the production stream).  Per primary ray, with aperture > 0:
 *   1. d0 = raygen(basis, p, rng): the two jitter draws;
 *   2. up to 16 pairs a = 2 randf - 1, b = 2 randf - 1, the first with a*a + b*b < 1; (0, 0) after 16 rejections;
 *   3. per camera u = dx/|dx|, v = dy/|dy|, r = aperture/2, f = focus > 0 ? focus : |lookAt - pos|;
 *   4. o = (pos + u*(r*a)) + v*(r*b);
 *   5. F = pos + d0*(f / (d0 . nlook));
 *   6. d = F - o, nudged and normalised as raygen does;
 *   7. the path continues from (o, d) with the stream after the 2 + 2k draws.
 * Step 6 is raygen itself: the ray is traced from a synthetic basis with pos = o, nlook = F - o and dx = dy = 0, for
 * which raygen's sum nlook + dx*sx + dy*sy is F - o exactly and its nudge and division are the ones step 6 names.
 * raygen draws twice, so the synthetic ray starts from the stream after 2k draws, and leaves it after 2 + 2k.
 */
#include "../oracle/b2pt_oracle.c"

typedef struct
{
  v3 u, v;
  float r, f;
} lens_rec;

static lens_rec make_lens(const cam_basis* b, const orc_camera* cam, float aperture, float focus)
{
  lens_rec L;
  const float lu = sqrtf(vdot(b->dx, b->dx)), lv = sqrtf(vdot(b->dy, b->dy));
  L.u = V(b->dx.x / lu, b->dx.y / lu, b->dx.z / lu);
  L.v = V(b->dy.x / lv, b->dy.y / lv, b->dy.z / lv);
  L.r = aperture / 2.f;
  if (focus > 0.f)
    L.f = focus;
  else
  {
    const v3 e = vsub(ld3(cam->lookAt), b->pos);
    L.f = sqrtf(vdot(e, e));
  }
  return L;
}

/* Steps 1-5 for pixel idx from stream state seed0: the synthetic basis of the lens ray in *ray and the number of draws
 * in *draws; returns the stream state from which raygen(ray, idx, .) takes the lens ray (seed0 after 2k draws). */
static uint32_t lens_ray(const cam_basis* b, const lens_rec* L, int64_t idx, uint32_t seed0, cam_basis* ray, int* draws)
{
  uint32_t s = seed0;
  const v3 d0 = raygen(b, idx, &s);
  float a = 0.f, c = 0.f;
  int pairs = 0;
  while (pairs < 16)
  {
    const float x = 2.f * orc_randf(&s) - 1.f;
    const float y = 2.f * orc_randf(&s) - 1.f;
    ++pairs;
    if (x * x + y * y < 1.f)
    {
      a = x, c = y;
      break;
    }
  }
  const float ra = L->r * a, rb = L->r * c;
  const v3 o = vadd(vadd(b->pos, vscale(L->u, ra)), vscale(L->v, rb));
  const float k = L->f / vdot(d0, b->nlook);
  const v3 F = vadd(b->pos, vscale(d0, k));
  *ray = *b;
  ray->pos = o;
  ray->nlook = vsub(F, o);
  ray->dx = V(0.f, 0.f, 0.f);
  ray->dy = V(0.f, 0.f, 0.f);
  *draws = 2 + 2 * pairs;
  uint32_t j = seed0;
  for (int n = 0; n < 2 * pairs; ++n)
    orc_wang32(&j);
  return j;
}

/* The primary ray of pixel idx from *seed (left after the ray's draws): origin o3, direction dir3; returns the draws
 * (2 for the pinhole, aperture <= 0). */
int lens_raygen(const orc_camera* cam, float aperture, float focus, int64_t idx, uint32_t* seed, float* o3,
                float* dir3)
{
  const cam_basis b = make_basis(cam);
  if (!(aperture > 0.f))
  {
    st3(dir3, raygen(&b, idx, seed));
    st3(o3, b.pos);
    return 2;
  }
  const lens_rec L = make_lens(&b, cam, aperture, focus);
  cam_basis ray;
  int draws;
  uint32_t s = lens_ray(&b, &L, idx, *seed, &ray, &draws);
  st3(dir3, raygen(&ray, idx, &s));
  st3(o3, ray.pos);
  *seed = s;
  return draws;
}

/* orc_primary_hits through the lens: sample 0 (seed i + seedOffset), t measured from the lens origin. */
int lens_primary_hits(const orc_scene* sc, const orc_camera* cam, float aperture, float focus, uint32_t seedOffset,
                      int flags, int32_t* primId, float* t)
{
  const int64_t N = (int64_t)cam->W * cam->H;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < N; i++)
  {
    uint32_t seed = (uint32_t)i + seedOffset;
    float o[3], d[3];
    lens_raygen(cam, aperture, focus, i, &seed, o, d);
    float rec[9];
    int hid[2];
    rec[HR_T] = FLT_MAX;
    const int64_t prim = closest_hit(sc, ld3(o), ld3(d), 0.001f, FLT_MAX, flags, rec, hid);
    primId[i] = (int32_t)prim;
    if (t)
      t[i] = prim >= 0 ? rec[HR_T] : FLT_MAX;
  }
  return 0;
}

/* orc_render mode 3 (FORWARD_FAST, the production stream) through the lens: samples [sampleBegin, sampleBegin+spp),
 * rgba = the un-normalised sums, W*H*4 floats; stats count the lens draws too. */
int lens_render(const orc_scene* sc, const orc_camera* cam, float aperture, float focus, int spp, int sampleBegin,
                int maxDepth, uint32_t seedOffset, int flags, int nThreads, float* rgba, orc_stats* stats)
{
  if (spp < 0 || maxDepth < 1 || cam->W <= 0 || cam->H <= 0)
    return -1;
  const int64_t N = (int64_t)cam->W * cam->H;
  const cam_basis cb = make_basis(cam);
  const int lens = aperture > 0.f;
  const lens_rec L = make_lens(&cb, cam, lens ? aperture : 0.f, focus);
  orc_stats total;
  memset(&total, 0, sizeof(total));
  total.paths = N * (int64_t)spp;
  memset(rgba, 0, sizeof(float) * 4 * (size_t)N);
  omp_set_num_threads(nThreads > 0 ? nThreads : omp_get_num_procs());
#pragma omp parallel
  {
    LStats ls;
    memset(&ls, 0, sizeof(ls));
#pragma omp for schedule(dynamic, 256)
    for (int64_t i = 0; i < N; i++)
    {
      float* px = rgba + 4 * i;
      for (int s = 0; s < spp; s++)
      {
        uint32_t seed = (uint32_t)i + seedOffset + (uint32_t)(sampleBegin + s) * ORC_GOLDEN;
        float Lr[3];
        if (lens)
        {
          cam_basis ray;
          int draws;
          uint32_t s2 = lens_ray(&cb, &L, i, seed, &ray, &draws);
          ls.draws += draws - 2; /* forward_sample counts raygen's two */
          forward_sample(sc, &ray, i, &s2, maxDepth, 0, flags, Lr, &ls, NULL);
        }
        else
          forward_sample(sc, &cb, i, &seed, maxDepth, 0, flags, Lr, &ls, NULL);
        px[0] += Lr[0], px[1] += Lr[1], px[2] += Lr[2];
      }
    }
#pragma omp critical
    merge_stats(&total, &ls);
  }
  if (stats)
    *stats = total;
  return 0;
}
