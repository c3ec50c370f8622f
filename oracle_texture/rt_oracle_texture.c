/* TEST INFRASTRUCTURE — the oracle's albedo-texture mode (include/b200rt.h, B200RT_SAMPLING_TEXTURES).  NOT part of the
 * product: only tests/ and tools/ may load this library.
 *
 * oracle_glass/rt_oracle_glass.c is compiled into this library unchanged, and with it oracle_smooth/rt_oracle_smooth.c
 * and oracle/rt_oracle.c, so the sampling, BSDF, traversal, generator, smooth-shading and glass code the other oracles'
 * tests pin bit for bit is the code used here.  Its path_sample_glass and orc_render_glass are simply not called.  This
 * file defines:
 *   - texel_factor: the texel rule of the header (repeat wrap, bilinear as lerps) for one texture and one (u, v);
 *   - tex_albedo: the albedo of a type-1 or type-2 hit, from the barycentrics of the smooth-shading rule and the UVs;
 *   - path_sample_tex: rt_oracle_glass.c's path_sample_glass statement for statement, but with the albedo in place of the
 *     material colour of every type-1 or type-2 hit when sampling bit 512 is set (tests/test_texture_oracle.py holds this
 *     library to oracle_glass/ bit for bit, counters included, when nothing is bound);
 *   - orc_render_tex: orc_render_glass's per-pixel loop (plain, pixel-jitter bit 8, adaptive, smooth bit 32, glass bit
 *     128) calling path_sample_tex;
 *   - orc_gbuffer_albedo_tex: the G-buffer albedo of given primary hits;
 *   - orc_texel: texel_factor on its own.
 * Same arithmetic conventions as rt_oracle.c.
 */
#include "../oracle_glass/rt_oracle_glass.c"

#define TEX_BIT 512

/* the bound textures: texels back to back (RGBA8, row-major, top row first), per texture (w, h) and its first texel,
 * per material its texture or -1 */
typedef struct {
  const unsigned char *texels;
  const int *dims;
  long long *first;
  const int *mat_tex;
  int n_mat;
} tex_t;

static inline float lerpf(float a, float b, float t) { return a + (b - a) * t; }

static inline int wrap_index(int i, int n) {
  const int r = i % n;
  return r < 0 ? r + n : r;
}

static void texel_value(const unsigned char *rgba, int w, int x, int y, float c[3]) {
  const unsigned char *p = rgba + 4 * ((size_t)y * (size_t)w + (size_t)x);
  for (int k = 0; k < 3; ++k) c[k] = (float)p[k] / 255.0f;
}

/* the texture factor of the header at (u, v) for one w x h texture */
static v3 texel_factor(const unsigned char *rgba, int w, int h, float u, float v) {
  if (!isfinite(u) || !isfinite(v)) return V(1.0f, 1.0f, 1.0f);
  const float fu = u - floorf(u), fv = v - floorf(v);
  const float tx = fu * (float)w - 0.5f, ty = (1.0f - fv) * (float)h - 0.5f;
  const int x0 = (int)floorf(tx), y0 = (int)floorf(ty);
  const float ax = tx - (float)x0, ay = ty - (float)y0;
  const int xa = wrap_index(x0, w), xb = wrap_index(x0 + 1, w), ya = wrap_index(y0, h), yb = wrap_index(y0 + 1, h);
  float c00[3], c10[3], c01[3], c11[3], f[3];
  texel_value(rgba, w, xa, ya, c00);
  texel_value(rgba, w, xb, ya, c10);
  texel_value(rgba, w, xa, yb, c01);
  texel_value(rgba, w, xb, yb, c11);
  for (int k = 0; k < 3; ++k) f[k] = lerpf(lerpf(c00[k], c10[k], ax), lerpf(c01[k], c11[k], ax), ay);
  return V(f[0], f[1], f[2]);
}

/* the albedo of a type-1 or type-2 hit on triangle t of material M at point x: M's colour times the texture factor at
 * the interpolated UV, or the colour itself when the material has no texture.  NOT in the reference, which fetches the
 * UVs and never reads them (MathLib.cl:203-228). */
static v3 tex_albedo(const scene_t *sc, const tex_t *T, int t, const mat_t *M, v3 x) {
  const int *f = sc->face + 10 * t;
  if (!T || f[0] >= T->n_mat || T->mat_tex[f[0]] < 0) return M->color;
  const int k = T->mat_tex[f[0]];
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
  const float *q0 = sc->vuv + 2 * f[1], *q1 = sc->vuv + 2 * f[2], *q2 = sc->vuv + 2 * f[3];
  const float u = (q0[0] * b0 + q1[0] * b1) + q2[0] * b2;
  const float v = (q0[1] * b0 + q1[1] * b1) + q2[1] * b2;
  return mul3(M->color, texel_factor(T->texels + 4 * T->first[k], T->dims[2 * k], T->dims[2 * k + 1], u, v));
}

/* rt_oracle_glass.c's path_sample_glass (Raytracing.cl:39-153), unchanged but for the albedo of type-1 / type-2 hits */
static v3 path_sample_tex(const scene_t *sc, const tex_t *T, int max_bounce, hit_t H, ray_t R, mat_t M, rng_t *g,
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
    if ((sc->sampling & TEX_BIT) && (M.type == 1 || M.type == 2))   /* the albedo (include/b200rt.h) */
      M.color = tex_albedo(sc, T, H.tri, &M, add3(R.o, scale3(unit3(R.d), H.k)));
    if (nee && M.type != 3) {   /* emitters are sampled at every surface that scatters (not at glass) */
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
    int interface = 0, reflected = 0;
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
        if ((sc->sampling & GLASS_BIT) && M.ior != 1.0f) {   /* the interface (include/b200rt.h) */
          float F;
          const float u = rng_next(g);   /* reference: the next value; Philox: word 0 of block (i, s, j, 0) */
          nb.d = dielectric(R.d, unit3(H.n), glass_ior(M.ior), u, &reflected, &F);
          interface = 1;
        } else {                                               /* the reference's pass-through */
          nb.d = R.d;
          brdf = M.color;
          inv_pdf = 1.0f / fabsf(dot3(nb.d, unit3(H.n)));
        }
        break;
    }
    nb.o = add3(R.o, scale3(unit3(R.d), H.k)); /* :79, no epsilon offset */
    hit_t Hb = closest_hit(sc, &nb);
    mat_t Mb = material_at(sc, Hb.mat);
    if (interface) {   /* weight 1: a reflection keeps the throughput, a refraction is tinted by the colour */
      if (!reflected) acc = mul3(acc, M.color);
    } else {
      float att = inv_pdf * fabsf(dot3(nb.d, unit3(H.n)));
      acc = scale3(mul3(acc, brdf), att);
    }
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
    } else { /* escaped: sun shadow ray + environment, :111-138 (a glass segment, either outcome, gets no sun) */
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

/* the texture table: first texel of every texture (prefix sums of w * h); NULL when nothing is bound */
static tex_t *make_tex(tex_t *T, const unsigned char *texels, const int *dims, int n_tex, const int *mat_tex, int n_mat) {
  if (n_tex <= 0 || n_mat <= 0) return NULL;
  T->texels = texels;
  T->dims = dims;
  T->mat_tex = mat_tex;
  T->n_mat = n_mat;
  T->first = (long long *)malloc(sizeof(long long) * (size_t)n_tex);
  long long s = 0;
  for (int k = 0; k < n_tex; ++k) {
    T->first[k] = s;
    s += (long long)dims[2 * k] * dims[2 * k + 1];
  }
  return T;
}

/* orc_render_glass's signature and loop, calling path_sample_tex, plus the bound textures (texels, dims, n_tex, mat_tex,
 * n_mat as b200rt_set_textures takes them; n_tex 0: nothing bound) */
void orc_render_tex(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
                    const float *mat, const float *bvh, const float *cam, const float *env, int tri_count,
                    int img_size, int spp, int max_bounce, const unsigned char *ibl, int ibl_w, int ibl_h,
                    int i0, int i1, const orc_opts *opts, const orc_adaptive *ad, int *spp_out, float *err_out,
                    unsigned long long *counters_out, const unsigned char *texels, const int *dims, int n_tex,
                    const int *mat_tex, int n_mat) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, mat, bvh, cam, env, tri_count, ibl, ibl_w, ibl_h, opts->stack_cap);
  sc.sampling = opts->sampling;
  sc.n_light = opts->light ? opts->n_light : 0;
  sc.light = opts->light;
  tex_t tex;
  const tex_t *T = make_tex(&tex, texels, dims, n_tex, mat_tex, n_mat);
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
        v3 c = path_sample_tex(&sc, T, max_bounce, H0, r, M0, &g, (uint32_t)i, (uint32_t)s);
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
  if (T) free(tex.first);
}

/* The G-buffer albedo (3 floats per pixel) of the primary hits tri / k of work-items [0, n): (1, 1, 1) for a miss or an
 * emitter, the material colour for glass, tex_albedo at cam_pos + unit(d) * k for a type-1 or type-2 hit. */
void orc_gbuffer_albedo_tex(float *albedo, const float *vp, const float *vuv, const int *face, const float *mat,
                            const float *cam, int n, const int *tri, const float *k, const unsigned char *texels,
                            const int *dims, int n_tex, const int *mat_tex, int n_mat) {
  scene_t sc;
  memset(&sc, 0, sizeof sc);
  sc.vp = vp; sc.vuv = vuv; sc.face = face; sc.mat = mat; sc.cam = cam;
  tex_t tex;
  const tex_t *T = make_tex(&tex, texels, dims, n_tex, mat_tex, n_mat);
  for (int i = 0; i < n; ++i) {
    v3 a = V(1.0f, 1.0f, 1.0f);
    if (tri[i] >= 0) {
      const mat_t M = material_at(&sc, sc.face[10 * tri[i]]);
      if (M.type == 1 || M.type == 2) {
        const ray_t r = camera_ray(&sc, i);
        a = tex_albedo(&sc, T, tri[i], &M, add3(r.o, scale3(unit3(r.d), k[i])));
      } else if (M.type == 3) {
        a = M.color;
      }
    }
    albedo[3 * (size_t)i] = a.x; albedo[3 * (size_t)i + 1] = a.y; albedo[3 * (size_t)i + 2] = a.z;
  }
  if (T) free(tex.first);
}

/* texel_factor of one w x h texture for n points (u[i], v[i]) -> out[3i ..] */
void orc_texel(const unsigned char *rgba, int w, int h, int n, const float *u, const float *v, float *out) {
  for (int i = 0; i < n; ++i) {
    const v3 f = texel_factor(rgba, w, h, u[i], v[i]);
    out[3 * i] = f.x; out[3 * i + 1] = f.y; out[3 * i + 2] = f.z;
  }
}
