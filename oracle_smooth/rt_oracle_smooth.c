/* TEST INFRASTRUCTURE — the oracle's smooth-shading mode (include/b200rt.h, B200RT_SAMPLING_SMOOTH_NORMALS).  NOT part
 * of the product: only tests/ and tools/ may load this library.
 *
 * oracle/rt_oracle.c is compiled into this library unchanged, so the sampling, BSDF, traversal and generator code it
 * restates is the code the oracle's own tests pin bit for bit to the reference's kernels.  Its closest_hit, path_sample
 * and orc_render are compiled under other names (the #defines below).  This file then defines:
 *   - closest_hit: the oracle's closest hit, whose normal is replaced by smooth_normal at x = o + unit(d) * k (the point
 *     the path continues from, Raytracing.cl:79) when sampling bit 32 is set;
 *   - path_sample: rt_oracle.c's path_sample statement for statement, so that its bounce and light rays go through this
 *     closest_hit (tests/test_smooth_oracle.py holds this library to oracle/, oracle_jitter/ and oracle_adaptive/ bit for
 *     bit when bit 32 is clear);
 *   - orc_render_smooth: orc_render's per-pixel loop, with orc_render_jitter's camera ray per sample when sampling bit 8 is
 *     set and orc_render_adaptive's stopping rule when `ad` is given;
 *   - orc_smooth_normal: the rule on its own.
 * Same arithmetic conventions as rt_oracle.c.
 */
#define closest_hit closest_hit_flat
#define path_sample path_sample_flat
#define orc_render orc_render_flat
#include "../oracle/rt_oracle.c"
#undef closest_hit
#undef path_sample
#undef orc_render

/* the shading normal of a hit on triangle t at point x (include/b200rt.h): n0 for a flat triangle (n0, n1, n2 equal bit
 * for bit), else the normalised barycentric interpolation of the three vertex normals, or n0 when that is not a usable
 * direction.  NOT in the reference, which shades with n0 (MathLib.cl:151). */
static v3 smooth_normal(const scene_t *sc, int t, v3 x) {
  const int *f = sc->face + 10 * t;
  const float *a = sc->vn + 3 * f[4], *b = sc->vn + 3 * f[5], *c = sc->vn + 3 * f[6];
  v3 n0 = V(a[0], a[1], a[2]);
  if (memcmp(a, b, 3 * sizeof(float)) == 0 && memcmp(a, c, 3 * sizeof(float)) == 0) return n0;
  const float *pa = sc->vp + 3 * f[7], *pb = sc->vp + 3 * f[8], *pc = sc->vp + 3 * f[9];
  v3 A = V(pa[0], pa[1], pa[2]);
  v3 e1 = sub3(V(pb[0], pb[1], pb[2]), A);
  v3 e2 = sub3(V(pc[0], pc[1], pc[2]), A);
  v3 p = sub3(x, A);
  float d00 = dot3(e1, e1), d01 = dot3(e1, e2), d11 = dot3(e2, e2);
  float d20 = dot3(p, e1), d21 = dot3(p, e2);
  float den = d00 * d11 - d01 * d01;
  float b1 = (d11 * d20 - d01 * d21) / den;
  float b2 = (d00 * d21 - d01 * d20) / den;
  float b0 = (1.0f - b1) - b2;
  v3 m = add3(add3(scale3(n0, b0), scale3(V(b[0], b[1], b[2]), b1)), scale3(V(c[0], c[1], c[2]), b2));
  v3 n = unit3(m);
  if (!isfinite(n.x) || !isfinite(n.y) || !isfinite(n.z) || !(dot3(n, n) > 0.0f)) return n0;
  return n;
}

static hit_t closest_hit(const scene_t *sc, const ray_t *r) {
  hit_t best = closest_hit_flat(sc, r);
  if (best.hit && (sc->sampling & 32)) best.n = smooth_normal(sc, best.tri, add3(r->o, scale3(unit3(r->d), best.k)));
  return best;
}

/* rt_oracle.c's path_sample (Raytracing.cl:39-153), unchanged but for the closest_hit above */
static v3 path_sample(const scene_t *sc, int max_bounce, hit_t H, ray_t R, mat_t M, rng_t *g,
                      uint32_t pixel, uint32_t sample) {
  v3 acc = V(1.0f, 1.0f, 1.0f);
  v3 rad = V(0.0f, 0.0f, 0.0f);      /* direct light gathered along the path (light sampling only) */
  const int nee = (sc->sampling & 2) && sc->n_light > 0;
  for (int j = 0; j <= max_bounce; ++j) {
    rng_set_bounce(g, pixel, sample, (uint32_t)j);
    if (!H.hit) { /* :146-150 */
      acc = scale3(mul3(acc, ibl_lookup(sc, R.d)), sc->env[4]);
      break;
    }
    if (M.type == 0) { /* :140-144 */
      acc = scale3(acc, M.roughness);
      break;
    }
    if (nee && M.type != 3) {   /* emitters are sampled at every surface that scatters (not at pass-through glass) */
      float u[3];
      rng_light3(g, pixel, sample, (uint32_t)j, u);
      ray_t sh;
      int target;
      v3 x = add3(R.o, scale3(unit3(R.d), H.k));
      v3 direct = sample_light(sc, &M, H.n, x, R.d, acc, u, &sh, &target);
      hit_t Hl = closest_hit(sc, &sh);
      if (Hl.hit && Hl.tri == target) rad = add3(rad, direct);
    }
    ray_t nb;
    v3 brdf = V(0, 0, 0);
    float inv_pdf = 0.0f;
    nb.d = V(0, 0, 0);
    const v3 d_in = R.d;
    switch (M.type) { /* :58-78 (case 0 is unreachable here) */
      case 1:
        nb.d = sample_cosine(H.n, g, &inv_pdf);
        brdf = scale3(M.color, 1.0f / 3.14f);
        break;
      case 2:
        if (sc->sampling & 1) nb.d = sample_glossy_importance(M.roughness, H.n, R.d, g, &inv_pdf);
        else nb.d = sample_uniform(H.n, g, &inv_pdf);
        brdf = bsdf_ggx(&M, V(-R.d.x, -R.d.y, -R.d.z), nb.d, H.n);
        break;
      case 3:
        nb.d = R.d;
        brdf = M.color;
        inv_pdf = 1.0f / fabsf(dot3(nb.d, unit3(H.n)));
        break;
    }
    nb.o = add3(R.o, scale3(unit3(R.d), H.k)); /* :79, no epsilon offset */
    hit_t Hb = closest_hit(sc, &nb);
    mat_t Mb = material_at(sc, Hb.mat);
    float att = inv_pdf * fabsf(dot3(nb.d, unit3(H.n)));
    acc = scale3(mul3(acc, brdf), att);
    if (Hb.hit) {
      int from_type = M.type;
      mat_t Mfrom = M;
      v3 nfrom = H.n;
      R = nb; H = Hb; M = Mb;
      if (Mb.type != 0) {
        if (j == max_bounce) { acc = V(0, 0, 0); break; }
      } else {
        acc = scale3(acc, Mb.roughness);
        if (nee && from_type != 3) {
          /* the light sample at the surface this ray left could have produced the same connection: balance heuristic */
          v3 wi = unit3(nb.d);
          float pb_ = bsdf_pdf(sc, &Mfrom, nfrom, d_in, wi);
          float pl = light_pdf(sc, Hb.tri, wi, (Hb.k * Hb.k) * dot3(nb.d, nb.d));
          float den = pb_ + pl;
          acc = scale3(acc, den > 0.0f ? pb_ / den : 0.0f);
        }
        break;
      }
    } else { /* escaped: sun shadow ray + environment, :111-138 */
      ray_t sr;
      sr.o = nb.o;
      sr.d = sun_direction(sc);
      hit_t Hs = closest_hit(sc, &sr);
      mat_t Ms = material_at(sc, Hs.mat);
      v3 sun = V(0, 0, 0);
      if (!Hs.hit && M.type != 3) sun = V(sc->env[3], sc->env[3], sc->env[3]);
      if (Hs.hit && Ms.type == 3) sun = scale3(Ms.color, sc->env[3]);
      v3 envl = scale3(ibl_lookup(sc, nb.d), sc->env[4]);
      acc = mul3(acc, add3(sun, envl));
      break;
    }
  }
  return nee ? add3(rad, acc) : acc;
}

/* oracle_jitter/rt_oracle_jitter.c's jitter draw and camera ray, unchanged (that file compiles rt_oracle.c in as well,
 * so it cannot be included here) */
/* (ux, uy) of sample s of pixel i: the generator's next two values in reference mode, words 0 and 1 of the Philox
 * block (i, s, 0, 2) otherwise */
static void rng_jitter2(rng_t *g, uint32_t pixel, uint32_t sample, float *ux, float *uy) {
  if (g->mode == 0) {
    *ux = rng_next(g);
    *uy = rng_next(g);
    return;
  }
  uint32_t ctr[4] = {pixel, sample, 0u, 2u}, out[4];
  philox4x32_10(ctr, g->key0, g->key1, out);
  tl_cnt.rand_calls += 2;
  *ux = bits_to_unit(out[0]);
  *uy = bits_to_unit(out[1]);
}

/* camera_ray's statements (Raytracing.cl:18-37) through image-plane point (col + ux - 0.5, row + uy - 0.5) */
static ray_t camera_ray_jittered(const scene_t *sc, int i, float ux, float uy) {
  const float *cam = sc->cam;
  int w = (int)cam[6];
  int col = (i + 1) % w;
  int row = (i - col) / w;
  v3 pos = V(cam[0], cam[1], cam[2]);
  v3 focal = V(cam[0], cam[1] - (1.0f / (2.0f * cr_tan(cam[9] / 2.0f))), cam[2]);
  float step = (float)(1.0 / (double)cam[6]);
  float fx = (float)col + (ux - 0.5f);
  float fz = (float)row + (uy - 0.5f);
  v3 pix = V(fx * step - 0.5f, 0.0f, 0.5f - fz * step);
  ray_t r;
  r.o = pos;
  r.d = unit3(sub3(add3(pos, pix), focal));
  r.d = rotate_about(cam[3] * DEG2RAD, V(1, 0, 0), r.d);
  r.d = rotate_about(cam[4] * DEG2RAD, V(0, 1, 0), r.d);
  r.d = rotate_about(cam[5] * DEG2RAD, V(0, 0, 1), r.d);
  return r;
}

typedef struct {
  int min_spp, check_every;
  float rel_error, floor;
} orc_adaptive;

/* orc_render's signature and loop (work-items [i0,i1), sample range, raw sums, threads).  Sampling bit 8: every sample
 * traces its own jittered camera ray (orc_render_jitter).  ad != NULL: orc_render_adaptive's stopping rule over [0, spp)
 * (opts->s0 / s1 / raw_sums not read), with samples taken and standard error in spp_out / err_out. */
void orc_render_smooth(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
                       const float *mat, const float *bvh, const float *cam, const float *env, int tri_count,
                       int img_size, int spp, int max_bounce, const unsigned char *ibl, int ibl_w, int ibl_h,
                       int i0, int i1, const orc_opts *opts, const orc_adaptive *ad, int *spp_out, float *err_out,
                       unsigned long long *counters_out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, mat, bvh, cam, env, tri_count, ibl, ibl_w, ibl_h, opts->stack_cap);
  sc.sampling = opts->sampling;
  sc.n_light = opts->light ? opts->n_light : 0;
  sc.light = opts->light;
  const int jitter = (opts->sampling & 8) != 0;
  int s0 = opts->s0, s1 = opts->s1;
  if (s1 <= 0 || ad) { s0 = 0; s1 = spp; }
  unsigned long long c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#ifdef _OPENMP
  if (opts->nthreads > 0) omp_set_num_threads(opts->nthreads);
#endif
#pragma omp parallel reduction(+ : c0, c1, c2, c3)
  {
    memset(&tl_cnt, 0, sizeof tl_cnt);
#pragma omp for schedule(dynamic, 64)
    for (int i = i0; i < i1; ++i) {
      rng_t g;
      memset(&g, 0, sizeof g);
      g.mode = opts->rng_mode;
      g.a = (uint32_t)(i % img_size);
      g.b = (uint32_t)(i / img_size);
      g.key0 = opts->seed_lo;
      g.key1 = opts->seed_hi;
      ray_t r = {{0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}};
      hit_t H0 = {0};
      mat_t M0 = {0};
      if (!jitter) {
        r = camera_ray(&sc, i);
        H0 = closest_hit(&sc, &r);
        M0 = material_at(&sc, H0.mat);
      }
      /* adaptive: a primary miss or an emitter is ray-free and not subject to the rule */
      const int rule = ad && H0.hit && M0.type != 0;
      v3 sum = V(0.0f, 0.0f, 0.0f);
      float mean = 0.0f, m2 = 0.0f;
      int n = spp;
      for (int s = s0; s < s1; ++s) {
        if (jitter) {
          float ux, uy;
          rng_jitter2(&g, (uint32_t)i, (uint32_t)s, &ux, &uy);
          r = camera_ray_jittered(&sc, i, ux, uy);
          H0 = closest_hit(&sc, &r);
          M0 = material_at(&sc, H0.mat);
        }
        v3 c = path_sample(&sc, max_bounce, H0, r, M0, &g, (uint32_t)i, (uint32_t)s);
        sum = add3(sum, c);
        if (!rule) continue;
        const int k = s + 1;
        const float y = (0.2126f * c.x + 0.7152f * c.y) + 0.0722f * c.z;
        const float delta = y - mean;
        mean = mean + delta / (float)k;
        m2 = m2 + delta * (y - mean);
        if (k >= ad->min_spp && (k - ad->min_spp) % ad->check_every == 0 && k < spp) {
          const float v = (m2 / (float)(k - 1)) / (float)k;
          const float e = ad->rel_error * fmaxf(fminf(mean, 1.0f), ad->floor);
          if (v <= e * e) {
            n = k;
            break;
          }
        }
      }
      if (opts->raw_sums && !ad) {
        out[3 * (size_t)i + 0] = sum.x; out[3 * (size_t)i + 1] = sum.y; out[3 * (size_t)i + 2] = sum.z;
      } else {
        sum = div3s(sum, (float)(ad ? n : spp));
        if (i < img_size) {
          out[3 * (size_t)i + 0] = fmaxf(fminf(sum.x, 1.0f), 0.0f);
          out[3 * (size_t)i + 1] = fmaxf(fminf(sum.y, 1.0f), 0.0f);
          out[3 * (size_t)i + 2] = fmaxf(fminf(sum.z, 1.0f), 0.0f);
          if (ad) {
            spp_out[i] = n;
            err_out[i] = rule ? sqrtf((m2 / (float)(n - 1)) / (float)n) : 0.0f;
          }
        }
      }
    }
    c0 += tl_cnt.rays; c1 += tl_cnt.box_tests; c2 += tl_cnt.tri_tests; c3 += tl_cnt.rand_calls;
  }
  if (counters_out) { counters_out[0] = c0; counters_out[1] = c1; counters_out[2] = c2; counters_out[3] = c3; }
}

/* smooth_normal of n hits: triangle tri[i] at point x[3i .. 3i+2] */
void orc_smooth_normal(const float *vp, const float *vn, const int *face, int n, const int *tri, const float *x,
                       float *out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, NULL, face, NULL, NULL, NULL, NULL, 0, NULL, 0, 0, 0);
  for (int i = 0; i < n; ++i) {
    v3 r = smooth_normal(&sc, tri[i], V(x[3 * i], x[3 * i + 1], x[3 * i + 2]));
    out[3 * i] = r.x; out[3 * i + 1] = r.y; out[3 * i + 2] = r.z;
  }
}
