/* TEST INFRASTRUCTURE — the oracle's adaptive-sampling mode (include/b200rt.h, b200rt_adaptive).  NOT part of the
 * product: only tests/ may load this library.
 *
 * oracle/rt_oracle.c is compiled into this library unchanged, so everything it restates is the same code the
 * oracle's own tests pin bit for bit to the reference's kernels; this file adds one entry point,
 * orc_render_adaptive: orc_render's per-pixel loop over [0, spp) with the stopping rule of b200rt.h applied after
 * every sample.  Same arithmetic conventions as rt_oracle.c (binary32, -ffp-contract=off, true division, sqrtf).
 */
#include "../oracle/rt_oracle.c"

typedef struct {
  int min_spp, check_every;
  float rel_error, floor;
} orc_adaptive;

/* Work-items [i0,i1) of an img_size-item launch with at most spp samples each.  opts->s0 / s1 / raw_sums are not
 * read (an adaptive frame is the whole sample range, finalised).  out: img_size*3 floats, spp_out / err_out:
 * img_size entries (only [i0,i1) written): samples taken and standard error of the mean luminance. */
void orc_render_adaptive(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
                         const float *mat, const float *bvh, const float *cam, const float *env, int tri_count,
                         int img_size, int spp, int max_bounce, const unsigned char *ibl, int ibl_w, int ibl_h,
                         int i0, int i1, const orc_opts *opts, const orc_adaptive *ad, int *spp_out, float *err_out,
                         unsigned long long *counters_out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, mat, bvh, cam, env, tri_count, ibl, ibl_w, ibl_h, opts->stack_cap);
  sc.sampling = opts->sampling;
  sc.n_light = opts->light ? opts->n_light : 0;
  sc.light = opts->light;
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
      ray_t r = camera_ray(&sc, i);
      hit_t H0 = closest_hit(&sc, &r);
      mat_t M0 = material_at(&sc, H0.mat);
      /* a primary miss or an emitter: every sample is the same ray-free value, and the rule does not apply (the GPU's
         primary-hit kernel finishes such pixels itself) */
      const int rule = H0.hit && M0.type != 0;
      v3 sum = V(0.0f, 0.0f, 0.0f);
      float mean = 0.0f, m2 = 0.0f;
      int n = spp;
      for (int s = 0; s < spp; ++s) {
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
      sum = div3s(sum, (float)n);
      if (i < img_size) {
        out[3 * (size_t)i + 0] = fmaxf(fminf(sum.x, 1.0f), 0.0f);
        out[3 * (size_t)i + 1] = fmaxf(fminf(sum.y, 1.0f), 0.0f);
        out[3 * (size_t)i + 2] = fmaxf(fminf(sum.z, 1.0f), 0.0f);
        spp_out[i] = n;
        err_out[i] = rule ? sqrtf((m2 / (float)(n - 1)) / (float)n) : 0.0f;
      }
    }
    c0 += tl_cnt.rays; c1 += tl_cnt.box_tests; c2 += tl_cnt.tri_tests; c3 += tl_cnt.rand_calls;
  }
  if (counters_out) { counters_out[0] = c0; counters_out[1] = c1; counters_out[2] = c2; counters_out[3] = c3; }
}
