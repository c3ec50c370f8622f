/* TEST INFRASTRUCTURE — the oracle's per-hit shading rules one record at a time, in the record layout of
 * include/b200rt.h's b200rt_rule_probe, so that tests can compare the device's rules with the oracle's value by value.
 * NOT part of the product: only tests/ and tools/ may load this library.
 *
 * oracle_rough/rt_oracle_rough.c is compiled in unchanged; it brings in oracle_texture/, oracle_glass/, oracle_smooth/
 * and oracle/rt_oracle.c.  Every rule calls the static function those files define for it (sample_cosine,
 * sample_uniform, sample_glossy_importance, bsdf_ggx, sample_light, light_pdf, bsdf_pdf, dielectric, rough_dielectric,
 * smooth_normal, tex_albedo, texel_factor); nothing is restated.  The samplers draw their uniforms from an rng_t in
 * Philox mode whose block holds the record's words 12-15: rng_next then returns bits_to_unit(word) in order, the
 * device's conversion.  Same arithmetic conventions as rt_oracle.c.
 *
 * Where the device takes a value, this side takes it too and two rules read the scene differently:
 *   - rule 8 picks its emitter with u[0] from a light list of n_light entries that all name the record's emitter;
 *   - rules 9 and 10 read the triangle's vertex normals / UVs and its material from faceData (the device reads the
 *     repacked records of the same data); rule 10 takes the triangle's own material, so i10 must be that material,
 *     and rule 9's curved flag is "the three vertex normals are not equal bit for bit", the test smooth_normal makes.
 */
#include "../oracle_rough/rt_oracle_rough.c"

static inline int word_i(const float *a) { int32_t v; memcpy(&v, a, 4); return v; }
static inline uint32_t word_u(const float *a) { uint32_t v; memcpy(&v, a, 4); return v; }

/* n records in[16 i ..] -> out[8 i ..] of rule `rule` (b200rt.h b200rt_rule_probe).  Scene arrays as orc_render takes
 * them (NULL when no rule of the call reads them); textures as b200rt_set_textures takes them (n_tex 0: none bound). */
void orc_rule_probe(int rule, const float *in, int n, float *out, const float *vp, const float *vn, const float *vuv,
                    const int *face, const float *mat, int tri_count, const unsigned char *texels, const int *dims,
                    int n_tex, const int *mat_tex, int n_mat) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, mat, NULL, NULL, NULL, tri_count, NULL, 0, 0, 0);
  tex_t tex;
  const tex_t *T = make_tex(&tex, texels, dims, n_tex, mat_tex, n_mat);
  int *light = NULL;
  int light_cap = 0;
  for (int i = 0; i < n; ++i) {
    const float *a = in + 16 * (size_t)i;
    float *o = out + 8 * (size_t)i;
    const v3 d = V(a[0], a[1], a[2]), nr = V(a[3], a[4], a[5]), x = V(a[6], a[7], a[8]);
    const int i9 = word_i(a + 9), i10 = word_i(a + 10), i11 = word_i(a + 11);
    rng_t g;
    memset(&g, 0, sizeof g);
    g.mode = 1;
    for (int k = 0; k < 4; ++k) g.blk[k] = word_u(a + 12 + k);
    g.blk_pos = 0;
    const float u0 = bits_to_unit(g.blk[0]), u1 = bits_to_unit(g.blk[1]), u2 = bits_to_unit(g.blk[2]);
    float r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    v3 v = V(0.0f, 0.0f, 0.0f);
    int flag = 0;
    switch (rule) {
      case 0: {
        float F;
        v = dielectric(d, nr, a[6], u0, &flag, &F);
        r[3] = flag ? 1.0f : 0.0f;
        break;
      }
      case 1:
        v = rough_dielectric(d, nr, a[6], a[7], u0, u1, u2, &flag, &r[4]);
        r[3] = flag ? 1.0f : 0.0f;
        break;
      case 2: case 3: v = sample_cosine(nr, &g, &r[3]); break;
      case 4: case 5: v = sample_uniform(nr, &g, &r[3]); break;
      case 6: {
        mat_t M = {2, V(1.0f, 1.0f, 1.0f), a[6], 0.0f};
        sc.sampling = 1;
        v = sample_glossy_importance(M.roughness, nr, d, &g, &r[3]);
        r[4] = bsdf_pdf(&sc, &M, nr, d, unit3(v));
        break;
      }
      case 7: {
        mat_t M = {2, V(a[9], a[10], a[11]), a[12], 0.0f};
        v = bsdf_ggx(&M, d, x, nr);
        break;
      }
      case 8: {
        if (i11 > light_cap) {
          free(light);
          light_cap = i11;
          light = (int *)malloc(sizeof(int) * (size_t)light_cap);
        }
        for (int k = 0; k < i11; ++k) light[k] = i9;
        sc.n_light = i11;
        sc.light = light;
        sc.sampling = word_i(a + 15);
        const mat_t M = material_at(&sc, i10);
        const float u[3] = {u0, u1, u2};
        ray_t sh;
        int target;
        v = sample_light(&sc, &M, nr, x, d, V(1.0f, 1.0f, 1.0f), u, &sh, &target);
        const float dist2 = dot3(sh.d, sh.d);
        const v3 wi = div3s(sh.d, sqrtf(dist2));
        r[3] = sh.d.x; r[4] = sh.d.y; r[5] = sh.d.z;
        r[6] = light_pdf(&sc, target, wi, dist2);
        r[7] = bsdf_pdf(&sc, &M, nr, d, wi);
        break;
      }
      case 9: {
        const int *f = face + 10 * (size_t)i9;
        const float *n0 = vn + 3 * f[4], *n1 = vn + 3 * f[5], *n2 = vn + 3 * f[6];
        v = smooth_normal(&sc, i9, x);
        r[3] = (memcmp(n0, n1, 3 * sizeof(float)) == 0 && memcmp(n0, n2, 3 * sizeof(float)) == 0) ? 0.0f : 1.0f;
        break;
      }
      case 10: {
        mat_t M = material_at(&sc, i10);
        M.color = d;
        v = tex_albedo(&sc, T, i9, &M, x);
        break;
      }
      case 11:
        if (T) v = texel_factor(T->texels + 4 * T->first[i9], dims[2 * i9], dims[2 * i9 + 1], a[6], a[7]);
        break;
    }
    r[0] = v.x; r[1] = v.y; r[2] = v.z;
    for (int k = 0; k < 8; ++k) o[k] = r[k];
  }
  free(light);
  if (T) free(tex.first);
}
