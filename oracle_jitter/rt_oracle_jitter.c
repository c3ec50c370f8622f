/* TEST INFRASTRUCTURE — the oracle's pixel-jitter mode (include/b200rt.h, B200RT_SAMPLING_PIXEL_JITTER).  NOT part of
 * the product: only tests/ and tools/ may load this library.
 *
 * oracle/rt_oracle.c is compiled into this library unchanged, so everything it restates is the same code the
 * oracle's own tests pin bit for bit to the reference's kernels; this file adds one entry point, orc_render_jitter:
 * orc_render's per-pixel loop in which every sample traces its own camera ray through a jittered point of its pixel
 * and then runs the oracle's path_sample from that ray's hit.  path_sample tests sampling bits 0 and 1 only, so the
 * jitter bit in opts->sampling does not reach it.  Same arithmetic conventions as rt_oracle.c.
 */
#include "../oracle/rt_oracle.c"

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

/* orc_render's signature and loop (work-items [i0,i1), sample range, raw sums, threads), one camera ray per sample */
void orc_render_jitter(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
                       const float *mat, const float *bvh, const float *cam, const float *env, int tri_count,
                       int img_size, int spp, int max_bounce, const unsigned char *ibl, int ibl_w, int ibl_h,
                       int i0, int i1, const orc_opts *opts, unsigned long long *counters_out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, mat, bvh, cam, env, tri_count, ibl, ibl_w, ibl_h, opts->stack_cap);
  sc.sampling = opts->sampling;
  sc.n_light = opts->light ? opts->n_light : 0;
  sc.light = opts->light;
  int s0 = opts->s0, s1 = opts->s1;
  if (s1 <= 0) { s0 = 0; s1 = spp; }
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
      v3 sum = V(0.0f, 0.0f, 0.0f);
      for (int s = s0; s < s1; ++s) {
        float ux, uy;
        rng_jitter2(&g, (uint32_t)i, (uint32_t)s, &ux, &uy);
        ray_t r = camera_ray_jittered(&sc, i, ux, uy);
        hit_t H0 = closest_hit(&sc, &r);
        mat_t M0 = material_at(&sc, H0.mat);
        v3 c = path_sample(&sc, max_bounce, H0, r, M0, &g, (uint32_t)i, (uint32_t)s);
        sum = add3(sum, c);
      }
      if (opts->raw_sums) {
        out[3 * (size_t)i + 0] = sum.x; out[3 * (size_t)i + 1] = sum.y; out[3 * (size_t)i + 2] = sum.z;
      } else {
        sum = div3s(sum, (float)spp);
        if (i < img_size) {
          out[3 * (size_t)i + 0] = fmaxf(fminf(sum.x, 1.0f), 0.0f);
          out[3 * (size_t)i + 1] = fmaxf(fminf(sum.y, 1.0f), 0.0f);
          out[3 * (size_t)i + 2] = fmaxf(fminf(sum.z, 1.0f), 0.0f);
        }
      }
    }
    c0 += tl_cnt.rays; c1 += tl_cnt.box_tests; c2 += tl_cnt.tri_tests; c3 += tl_cnt.rand_calls;
  }
  if (counters_out) { counters_out[0] = c0; counters_out[1] = c1; counters_out[2] = c2; counters_out[3] = c3; }
}
