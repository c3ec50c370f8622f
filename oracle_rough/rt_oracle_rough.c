/* TEST INFRASTRUCTURE — the oracle's rough-glass mode (include/b200rt.h, B200RT_SAMPLING_ROUGH_GLASS).  NOT part of the
 * product: only tests/ and tools/ may load this library.
 *
 * oracle_texture/rt_oracle_texture.c is compiled into this library unchanged, and with it oracle_glass/, oracle_smooth/
 * and oracle/rt_oracle.c, so the sampling, BSDF, traversal, generator, smooth-shading, glass and texture code the other
 * oracles' tests pin bit for bit is the code used here.  Its path_sample_tex and orc_render_tex are simply not called.
 * This file defines:
 *   - rough_dielectric: the rough interface rule of the header for one (w, n, ior, roughness, uf, u1, u2);
 *   - path_sample_rough: rt_oracle_texture.c's path_sample_tex statement for statement, but for case 3, which follows the
 *     rule when sampling bits 128 and 2048 are set, the ior slot is not 1 and the roughness is > 0 (tests/
 *     test_rough_glass_oracle.py holds this library to oracle_texture/ bit for bit, counters included, when every glass
 *     roughness is 0);
 *   - orc_render_rough: orc_render_tex's signature and per-pixel loop calling path_sample_rough;
 *   - orc_rough_dielectric: the rule on its own.
 * Same arithmetic conventions as rt_oracle.c.
 */
#include "../oracle_texture/rt_oracle_texture.c"

#define ROUGH_BIT 2048

/* the GGX visible normal [Heitz 2018] of roughness al around the unit N seen from the unit Vw, drawn with (u1, u2):
 * csrc/rt_shade.cuh's basis_duff and ggx_visible_normal statement for statement (rt_oracle.c's
 * sample_glossy_importance holds the same statements for glossy surfaces) */
static v3 ggx_visible_normal(float al, v3 N, v3 Vw, float u1, float u2) {
  const float kTwoPi = 6.2831853f;
  float sg = copysignf(1.0f, N.z);
  float a = -1.0f / (sg + N.z);
  float b = N.x * N.y * a;
  v3 T = V(1.0f + sg * N.x * N.x * a, sg * b, -sg * N.x);
  v3 B = V(b, sg + N.y * N.y * a, -N.y);
  float phi = kTwoPi * u2;
  float sp = cr_sin(phi), cp = cr_cos(phi);
  float r = sqrtf(u1);
  v3 Vh = unit3(V(al * dot3(Vw, T), al * dot3(Vw, B), dot3(N, Vw)));
  float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
  v3 T1 = V(1.0f, 0.0f, 0.0f);
  if (lensq > 0.0f) {
    float inv = 1.0f / sqrtf(lensq);
    T1 = V(-Vh.y * inv, Vh.x * inv, 0.0f);
  }
  v3 T2 = cross3(Vh, T1);
  float t1 = r * cp;
  float t2 = r * sp;
  float s = 0.5f * (1.0f + Vh.z);
  t2 = (1.0f - s) * sqrtf(fmaxf(0.0f, 1.0f - t1 * t1)) + s * t2;
  float t3 = sqrtf(fmaxf(0.0f, 1.0f - t1 * t1 - t2 * t2));
  v3 Nh = add3(add3(scale3(T1, t1), scale3(T2, t2)), scale3(Vh, t3));
  v3 hl = unit3(V(al * Nh.x, al * Nh.y, fmaxf(0.0f, Nh.z)));
  return add3(add3(scale3(T, hl.x), scale3(B, hl.y)), scale3(N, hl.z));
}

/* the next direction at a rough dielectric interface of index ior and roughness al > 0 met along d, un the unit normal,
 * uf u1 u2 the three uniforms: a GGX microfacet normal h seen from the incident side, then Fresnel's choice at h
 * [Walter et al. 2007].  *weight is Smith's G1 of the outgoing direction, 0 on the wrong side of the surface; c == 0, a
 * non-finite c or a non-finite h take dielectric() with uf and weight 1.  NOT in the reference, whose glass passes the
 * ray through (MathLib.cl:391-395). */
static v3 rough_dielectric(v3 d, v3 un, float ior, float al, float uf, float u1, float u2, int *reflected,
                           float *weight) {
  const v3 w = unit3(d);
  const float c = dot3(w, un);
  float eta;
  v3 m;
  if (c < 0.0f) {
    eta = 1.0f / ior; m = un;
  } else {
    eta = ior; m = V(-un.x, -un.y, -un.z);
  }
  const v3 Vw = V(-w.x, -w.y, -w.z);
  const v3 h = ggx_visible_normal(al, m, Vw, u1, u2);
  *weight = 1.0f;
  if (c == 0.0f || !isfinite(c) || !isfinite(h.x) || !isfinite(h.y) || !isfinite(h.z)) {
    float F;
    return dielectric(d, un, ior, uf, reflected, &F);
  }
  const float ch = dot3(Vw, h);
  const float k = 1.0f - (eta * eta) * (1.0f - ch * ch);
  float ct = 0.0f;
  int refl = 1;
  if (k >= 0.0f) {
    ct = sqrtf(k);
    const float rs = (eta * ch - ct) / (eta * ch + ct);
    const float rp = (ch - eta * ct) / (ch + eta * ct);
    const float F = 0.5f * (rs * rs + rp * rp);
    refl = !(uf >= F);
  }
  *reflected = refl;
  const v3 nd = refl ? add3(w, scale3(h, 2.0f * ch)) : add3(scale3(w, eta), scale3(h, eta * ch - ct));
  const float co = dot3(nd, m);
  if (refl ? co > 0.0f : co < 0.0f) {
    const float a = fabsf(co), a2 = al * al;
    *weight = (2.0f * a) / (a + sqrtf(a2 + (1.0f - a2) * a * a));
  } else {
    *weight = 0.0f;
  }
  return nd;
}

/* rt_oracle_texture.c's path_sample_tex (Raytracing.cl:39-153), unchanged but for case 3 with bits 128 and 2048 and the
 * weight of a rough-glass scatter */
static v3 path_sample_rough(const scene_t *sc, const tex_t *T, int max_bounce, hit_t H, ray_t R, mat_t M, rng_t *g,
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
    float weight = 1.0f;   /* rough glass: G1 of the outgoing direction, 0 on the wrong side */
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
        if ((sc->sampling & GLASS_BIT) && (sc->sampling & ROUGH_BIT) && M.ior != 1.0f && M.roughness > 0.0f) {
          /* the rough interface (include/b200rt.h): reference, the next three values; Philox, words 0-2 of (i, s, j, 0) */
          const float uf = rng_next(g);
          const float u1 = rng_next(g);
          const float u2 = rng_next(g);
          nb.d = rough_dielectric(R.d, unit3(H.n), glass_ior(M.ior), M.roughness, uf, u1, u2, &reflected, &weight);
          interface = 1;
        } else if ((sc->sampling & GLASS_BIT) && M.ior != 1.0f) {   /* the smooth interface (include/b200rt.h) */
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
    if (interface) {   /* a reflection keeps the throughput, a refraction is tinted by the colour; then the weight */
      if (!reflected) acc = mul3(acc, M.color);
      acc = weight == 0.0f ? V(0.0f, 0.0f, 0.0f) : scale3(acc, weight);
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

/* orc_render_tex's signature and loop, calling path_sample_rough */
void orc_render_rough(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
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
        v3 c = path_sample_rough(&sc, T, max_bounce, H0, r, M0, &g, (uint32_t)i, (uint32_t)s);
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

/* rough_dielectric for n cases: incoming direction w[3i..], unit normal nrm[3i..], ior slot v[i] (not 1; 0 resolves to
 * the default), roughness r[i] > 0, uniforms uf[i], u1[i], u2[i] -> direction d_out[3i..], reflected refl_out[i] (1 / 0),
 * weight_out[i] */
void orc_rough_dielectric(int n, const float *w, const float *nrm, const float *v, const float *r, const float *uf,
                          const float *u1, const float *u2, float *d_out, int *refl_out, float *weight_out) {
  for (int i = 0; i < n; ++i) {
    int refl;
    float wt;
    const v3 o = rough_dielectric(V(w[3 * i], w[3 * i + 1], w[3 * i + 2]), V(nrm[3 * i], nrm[3 * i + 1], nrm[3 * i + 2]),
                                  glass_ior(v[i]), r[i], uf[i], u1[i], u2[i], &refl, &wt);
    d_out[3 * i] = o.x; d_out[3 * i + 1] = o.y; d_out[3 * i + 2] = o.z;
    refl_out[i] = refl;
    weight_out[i] = wt;
  }
}
