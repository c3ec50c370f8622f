/* TEST INFRASTRUCTURE — CPU restatement of the reference hot path.  NOT part of the
 * product: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may
 * load this library, and only as the checker.
 *
 * What it restates (file:line relative to the reference repository):
 *   Kernels/Raytracing.cl   extractMaterial :5-15, genCameraRay :18-37, naiveGI :39-153,
 *                           __kernel Raytracing :161-221
 *   Kernels/MathLib.cl      quaternion_mult/rotateVec :51-65, SampleSphericalMap/sampleIBL
 *                           :72-90, intersect :117-160, intersectBox/interNode :167-199,
 *                           makeTri :203-228, rayTrace :234-288, rand :294-310,
 *                           rand_hemi_cosine :313-339, rand_hemi_uniform :342-366,
 *                           rand_sample_Glass :391-395, BRDF_GGX :461-500,
 *                           BRDF_Lambert :503-506, BRDF_Glass :509-512
 *   Kernels/stack.cl        Stack/push/pop :1-34
 *   Kernels/ImgProcessing.cl :1-9
 *
 * How it is pinned: tests/test_oracle_vs_ref.py requires this file to reproduce
 * oracle/_ref/libclref.so (the reference's own .cl text compiled by g++, see
 * oracle/build_ref.py) BIT FOR BIT — full renders, primary hits, the RNG stream and
 * the tonemap — on every shipped scene; tests/golden/ holds outputs of that library so
 * the same check runs where /root/reference is absent.
 *
 * Arithmetic conventions (identical to oracle/ref_shim/cl_shim.h): IEEE binary32, no
 * contraction (-ffp-contract=off), dot products summed left to right, normalize by true
 * division, transcendental built-ins correctly rounded (binary64 libm rounded once).
 *
 * Two additions beyond the reference, both opt-in through orc_opts:
 *   - rng_mode 1: counter-based Philox4x32-10 keyed by (pixel, sample, bounce) instead of
 *     the reference's sequential per-pixel generator (north_star asks for it; the
 *     reference generator cannot split a pixel's samples across GPUs);
 *   - sample range [s0,s1) with raw per-pixel sums as output (multi-GPU partial sums).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "cr_tie.h"
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { float x, y, z; } v3;
typedef struct { float w, x, y, z; } quat;

/* ---- correctly-rounded binary32 transcendentals ------------------------------------ */
/* glibc's binary64 value rounded once; where it lies within CR_TIE_GUARD binary64 ulps of a binary32 rounding boundary
 * (cr_tie.h) it is evaluated again in x87 extended precision and that is rounded instead.  Done on the domains on which
 * the kernels are correctly rounded (every float with |a| <= 8 for sin / cos, all of acos / asin, pow with the exponent
 * 2.2f; tests/test_cr_hard_cases.py checks every input the guard catches against mpmath); elsewhere the once-rounded
 * binary64 value, as on the GPU.  ref_shim/cl_shim.h states the same rule. */
static inline float cr_cos(float a) {
  const double r = cos((double)a);
  return (fabsf(a) <= 8.0f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)cosl((long double)a) : (float)r;
}
static inline float cr_sin(float a) {
  const double r = sin((double)a);
  return (fabsf(a) <= 8.0f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)sinl((long double)a) : (float)r;
}
static inline float cr_tan(float a) { return (float)tan((double)a); }
static inline float cr_acos(float a) {
  const double r = acos((double)a);
  return cr_tie_dist(r) <= CR_TIE_GUARD ? (float)acosl((long double)a) : (float)r;
}
static inline float cr_asin(float a) {
  const double r = asin((double)a);
  return cr_tie_dist(r) <= CR_TIE_GUARD ? (float)asinl((long double)a) : (float)r;
}
static inline float cr_atan2(float y, float x) { return (float)atan2((double)y, (double)x); }
static inline float cr_pow(float a, float b) {
  const double r = pow((double)a, (double)b);
  return (b == 2.2f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)powl((long double)a, (long double)b) : (float)r;
}

/* ---- small vector algebra (every product and sum rounded separately) ---------------- */
static inline v3 V(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline v3 add3(v3 a, v3 b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 sub3(v3 a, v3 b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 mul3(v3 a, v3 b) { return V(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 scale3(v3 a, float s) { return V(a.x * s, a.y * s, a.z * s); }
static inline v3 div3s(v3 a, float s) { return V(a.x / s, a.y / s, a.z / s); }
static inline float dot3(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline v3 cross3(v3 a, v3 b) {
  return V(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static inline v3 unit3(v3 a) { return div3s(a, sqrtf(dot3(a, a))); }

/* ---- counters ------------------------------------------------------------------------ */
typedef struct { unsigned long long rays, box_tests, tri_tests, rand_calls; } orc_counters;
static _Thread_local orc_counters tl_cnt;

/* ---- options -------------------------------------------------------------------------- */
typedef struct {
  int rng_mode;        /* 0 = reference generator (MathLib.cl:294-310), 1 = Philox4x32-10 */
  uint32_t seed_lo;    /* Philox key */
  uint32_t seed_hi;
  int stack_cap;       /* traversal stack capacity; the reference has 20 (MathLib.cl:248) */
  int s0, s1;          /* sample range [s0,s1); s1 <= 0 means [0, spp) */
  int raw_sums;        /* 1: write the un-normalised, un-clamped sum over [s0,s1) */
  int nthreads;        /* 0 = OpenMP default */
  int sampling;        /* bit 0: importance sampling of glossy surfaces; bit 1: direct sampling of the emitters listed in
                          `light` (opt-in, SURVEY 8f-4); 0 = the reference's estimator */
  int n_light;         /* lightData as FileManager builds it (FileManager.py:235-240): triangles whose material is emissive */
  const int *light;
} orc_opts;

typedef struct {
  const float *vp, *vn, *vuv, *mat, *bvh;
  const int *face;
  int tri_count;
  const unsigned char *ibl;
  int ibl_w, ibl_h;
  const float *cam, *env;
  int stack_cap;
  int sampling;
  int n_light;
  const int *light;
} scene_t;

/* =========================================================================================
 * Random numbers
 * ======================================================================================= */

/* MathLib.cl:294-310 as the kernel actually wires it.  Raytracing.cl:205-206 hands
 * (&seed0,&seed1) to naiveGI, naiveGI hands (seed1,seed0) to the samplers (:61-69) and
 * the samplers call rand(seed0,seed1) (MathLib.cl:316).  Net effect on the kernel's own
 * two words A = seed0, B = seed1:  B <- 36969*(A&65535)+(A>>16);  A <- 18000*(B&65535)+(B>>16);
 * bits = (B<<16)+A.  The incoming B is never read. */
typedef struct {
  int mode;
  uint32_t a, b;            /* reference generator words (kernel's seed0, seed1) */
  uint32_t key0, key1;      /* Philox key */
  uint32_t ctr[4];          /* Philox counter: pixel, sample, bounce, 0 */
  uint32_t blk[4];
  int blk_pos;
} rng_t;

static inline float bits_to_unit(uint32_t bits) {
  union { float f; uint32_t u; } c;
  c.u = (bits & 0x007fffffu) | 0x40000000u;
  return (c.f - 2.0f) / 2.0f;
}

static void philox4x32_10(const uint32_t ctr_in[4], uint32_t k0, uint32_t k1, uint32_t out[4]) {
  uint32_t c0 = ctr_in[0], c1 = ctr_in[1], c2 = ctr_in[2], c3 = ctr_in[3];
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* called at the top of every bounce iteration j of sample s of pixel i */
static inline void rng_set_bounce(rng_t *g, uint32_t pixel, uint32_t sample, uint32_t bounce) {
  if (g->mode == 1) {
    g->ctr[0] = pixel; g->ctr[1] = sample; g->ctr[2] = bounce; g->ctr[3] = 0;
    g->blk_pos = 4; /* lazily generated */
  }
}

static float rng_next(rng_t *g) {
  tl_cnt.rand_calls++;
  if (g->mode == 0) {
    g->b = 36969u * (g->a & 65535u) + (g->a >> 16);
    g->a = 18000u * (g->b & 65535u) + (g->b >> 16);
    return bits_to_unit((g->b << 16) + g->a);
  }
  if (g->blk_pos >= 4) {
    philox4x32_10(g->ctr, g->key0, g->key1, g->blk);
    g->ctr[3]++;
    g->blk_pos = 0;
  }
  return bits_to_unit(g->blk[g->blk_pos++]);
}

/* =========================================================================================
 * Rotation by quaternion — MathLib.cl:51-65
 * ======================================================================================= */
static inline quat qmul(quat q, quat p) {
  v3 qv = V(q.x, q.y, q.z), pv = V(p.x, p.y, p.z);
  quat r;
  r.w = q.w * p.w - dot3(qv, pv);
  v3 t = add3(add3(scale3(qv, p.w), scale3(pv, q.w)), cross3(qv, pv));
  r.x = t.x; r.y = t.y; r.z = t.z;
  return r;
}

static v3 rotate_about(float angle, v3 axis, v3 vec) {
  float half = angle * 0.5f;
  float c = cr_cos(half);
  v3 sv = scale3(unit3(axis), cr_sin(half));
  quat q = {c, sv.x, sv.y, sv.z};
  quat p = {0.0f, vec.x, vec.y, vec.z};
  /* conjugate scaled by |q|^2, then normalised as a 4-vector (MathLib.cl:62) */
  float n2 = q.w * q.w + dot3(sv, sv);
  v3 neg = scale3(sv, -1.0f);
  quat u = {q.w * n2, neg.x * n2, neg.y * n2, neg.z * n2};
  float len = sqrtf(u.w * u.w + u.x * u.x + u.y * u.y + u.z * u.z);
  quat qi = {u.w / len, u.x / len, u.y / len, u.z / len};
  quat r = qmul(qmul(q, p), qi);
  return V(r.x, r.y, r.z);
}

#define DEG2RAD (3.14f / 180.0f)

/* =========================================================================================
 * Environment lookup — MathLib.cl:72-90
 * ======================================================================================= */
static v3 ibl_lookup(const scene_t *sc, v3 dir) {
  dir = rotate_about(90 * DEG2RAD, V(1, 0, 0), dir);
  dir = rotate_about(90 * DEG2RAD, V(0, 1, 0), dir);
  float u = cr_atan2(dir.z, dir.x) * 0.1591f + 0.5f;
  float v = cr_asin(dir.y) * 0.3183f + 0.5f;
  int px = (int)(u * (float)sc->ibl_w);
  int py = (int)(v * (float)sc->ibl_h);
  /* integer-coordinate read with a clamp-to-edge sampler (Raytracing.cl:179) */
  if (px < 0) px = 0;
  if (px > sc->ibl_w - 1) px = sc->ibl_w - 1;
  if (py < 0) py = 0;
  if (py > sc->ibl_h - 1) py = sc->ibl_h - 1;
  const unsigned char *t = sc->ibl + 4 * ((size_t)py * (size_t)sc->ibl_w + (size_t)px);
  return scale3(V(t[0] / 255.0f, t[1] / 255.0f, t[2] / 255.0f), 1.0f);
}

/* =========================================================================================
 * Geometry
 * ======================================================================================= */
typedef struct { v3 o, d; } ray_t;
typedef struct { int hit; float k; int mat; v3 n; int tri; } hit_t;
typedef struct { int type; v3 color; float roughness, ior; } mat_t;

static inline mat_t material_at(const scene_t *sc, int idx) { /* Raytracing.cl:5-15 */
  const float *m = sc->mat + 6 * idx;
  mat_t r;
  r.type = (int)m[0];
  r.color = V(m[1], m[2], m[3]);
  r.roughness = m[4];
  r.ior = m[5];
  return r;
}

/* slab test with true divisions, no interval clipping — MathLib.cl:167-199 */
static inline int line_meets_box(const ray_t *r, const float *node) {
  tl_cnt.box_tests++;
  float a, b, lo, hi;
  a = (node[2] - r->o.x) / r->d.x;
  b = (node[5] - r->o.x) / r->d.x;
  lo = fminf(a, b);
  hi = fmaxf(a, b);
  a = (node[3] - r->o.y) / r->d.y;
  b = (node[6] - r->o.y) / r->d.y;
  lo = fmaxf(lo, fminf(a, b));
  hi = fminf(hi, fmaxf(a, b));
  a = (node[4] - r->o.z) / r->d.z;
  b = (node[7] - r->o.z) / r->d.z;
  lo = fmaxf(lo, fminf(a, b));
  hi = fminf(hi, fmaxf(a, b));
  return hi >= lo;
}

/* Möller–Trumbore on triangle `t` — makeTri MathLib.cl:203-228 + intersect :117-160.
 * Only the three positions, the first vertex normal and the material are consumed. */
static inline int tri_hit(const scene_t *sc, int t, const ray_t *r, float *k_out) {
  tl_cnt.tri_tests++;
  const int *f = sc->face + 10 * t;
  const float *pa = sc->vp + 3 * f[7], *pb = sc->vp + 3 * f[8], *pc = sc->vp + 3 * f[9];
  v3 A = V(pa[0], pa[1], pa[2]);
  v3 e1 = sub3(V(pb[0], pb[1], pb[2]), A);
  v3 e2 = sub3(V(pc[0], pc[1], pc[2]), A);
  const float eps = 0.0000001;
  v3 h = cross3(r->d, e2);
  float a = dot3(e1, h);
  if (a > -eps && a < eps) return 0;
  float f_ = (float)(1.0 / (double)a);
  v3 s = sub3(r->o, A);
  float u = f_ * dot3(s, h);
  if ((double)u < 0.0 || (double)u > 1.0) return 0;
  v3 q = cross3(s, e1);
  float v = f_ * dot3(r->d, q);
  if ((double)v < 0.0 || (double)(u + v) > 1.0) return 0;
  float k = f_ * dot3(e2, q);
  if (k > eps) { *k_out = k; return 1; }
  return 0;
}

/* closest hit in the reference's visiting order — MathLib.cl:234-288, stack.cl:21-34 */
static hit_t closest_hit(const scene_t *sc, const ray_t *r) {
  tl_cnt.rays++;
  hit_t best;
  best.hit = 0; best.k = 1000.0f; best.mat = 0; best.n = V(0, 0, 0); best.tri = -1;
  int stack[64];
  const int cap = sc->stack_cap;
  int top = -1;
  stack[++top] = 0;
  while (top != -1) {
    int cur = stack[top--];
    const float *node = sc->bvh + 9 * cur;
    if (!line_meets_box(r, node)) continue;
    int t = (int)node[8];
    if (t != -1) {
      float k;
      if (tri_hit(sc, t, r, &k) && k < best.k && k > 0.0001f) {
        const int *f = sc->face + 10 * t;
        const float *n0 = sc->vn + 3 * f[4];
        best.hit = 1; best.k = k; best.mat = f[0]; best.n = V(n0[0], n0[1], n0[2]); best.tri = t;
      }
    }
    int l = (int)node[0], rr = (int)node[1];
    if (l != -1 && top != cap - 1) stack[++top] = l;   /* push drops silently when full */
    if (rr != -1 && top != cap - 1) stack[++top] = rr;
  }
  if (best.k <= 0.0001f) { best.hit = 0; best.k = 0.0f; }
  return best;
}

/* Raytracing.cl:18-37 */
static ray_t camera_ray(const scene_t *sc, int i) {
  const float *cam = sc->cam;
  int w = (int)cam[6];
  int col = (i + 1) % w;
  int row = (i - col) / w;
  v3 pos = V(cam[0], cam[1], cam[2]);
  v3 focal = V(cam[0], cam[1] - (1.0f / (2.0f * cr_tan(cam[9] / 2.0f))), cam[2]);
  float step = (float)(1.0 / (double)cam[6]);
  v3 pix = V((float)col * step - 0.5f, 0.0f, 0.5f - (float)row * step);
  ray_t r;
  r.o = pos;
  r.d = unit3(sub3(add3(pos, pix), focal));
  r.d = rotate_about(cam[3] * DEG2RAD, V(1, 0, 0), r.d);
  r.d = rotate_about(cam[4] * DEG2RAD, V(0, 1, 0), r.d);
  r.d = rotate_about(cam[5] * DEG2RAD, V(0, 0, 1), r.d);
  return r;
}

/* =========================================================================================
 * Direction sampling — MathLib.cl:313-366
 * ======================================================================================= */
static const v3 ZUP = {0.0f, 0.0f, 1.0f};

static v3 sample_cosine(v3 n, rng_t *g, float *inv_pdf) {
  float u = rng_next(g);
  float theta = rng_next(g) * 2.0f * 3.14f;
  float rad = sqrtf(u);
  v3 local = V(rad * cr_cos(theta), rad * cr_sin(theta), sqrtf(fmaxf(0.0f, 1.0f - u)));
  v3 l;
  if (fabsf(dot3(unit3(n), ZUP)) == 1.0f) {
    l = scale3(local, n.z);
  } else {
    v3 axis = cross3(ZUP, n);
    float ang = cr_acos(dot3(n, ZUP));
    l = unit3(rotate_about(ang, axis, local));
  }
  *inv_pdf = 3.14f / fmaxf(dot3(l, n), 0.0f);
  return l;
}

static v3 sample_uniform(v3 n, rng_t *g, float *inv_pdf) {
  float phi = 2.0f * 3.14f * rng_next(g);
  float theta = cr_acos(1.0f - rng_next(g));
  float st = cr_sin(theta);
  v3 local = V(cr_cos(phi) * st, st * cr_sin(phi), cr_cos(theta));
  v3 w;
  if (fabsf(dot3(unit3(n), ZUP)) == 1.0f) {
    w = scale3(local, n.z);
  } else {
    v3 axis = unit3(cross3(ZUP, n));
    float ang = cr_acos(dot3(n, ZUP));
    w = rotate_about(ang, axis, local);
  }
  *inv_pdf = 2.0f * 3.14f;
  return w;
}

/* Opt-in (orc_opts.sampling = 1; NOT the reference's estimator — the reference draws glossy directions uniformly,
 * MathLib.cl:342-366): one-sample mixture of GGX visible-normal sampling [Heitz 2018] with alpha = roughness (the normal
 * distribution of BRDF_GGX, MathLib.cl:470-472; the lobe the author's dead rand_sample_GGX aims at, :369-387) and a
 * cosine lobe for the BRDF's diffuse term; returns the direction and 1 / pdf of the mixture.  Restated statement by
 * statement from csrc/rt_shade.cuh::sample_glossy_importance so that the two agree bit for bit. */
/* density (per solid angle) with which sample_glossy_importance draws direction l: half GGX visible normals reflected,
 * half cosine lobe; the cosine lobe alone when the viewer is below the surface.  N, Vw unit vectors. */
static float glossy_mix_pdf(float al, v3 N, v3 Vw, v3 l) {
  const float kPi = 3.14159265f;
  float ndv = dot3(N, Vw);
  float ndl = dot3(N, l);
  float pdf_cos = fmaxf(ndl, 0.0f) / kPi;
  float pdf_spec = 0.0f;
  if (ndv > 0.0f && ndl > 0.0f) {
    v3 h = unit3(add3(l, Vw));
    float ndh = dot3(N, h);
    float a2 = al * al;
    float dden = ndh * ndh * (a2 - 1.0f) + 1.0f;
    float D = a2 / (kPi * dden * dden);
    float G1 = (2.0f * ndv) / (ndv + sqrtf(a2 + (1.0f - a2) * ndv * ndv));
    pdf_spec = (G1 * D) / (4.0f * ndv);
  }
  float ps = ndv > 0.0f ? 0.5f : 0.0f;
  return ps * pdf_spec + (1.0f - ps) * pdf_cos;
}

static v3 sample_glossy_importance(float roughness, v3 n, v3 d_in, rng_t *g, float *inv_pdf) {
  const float kPi = 3.14159265f, kTwoPi = 6.2831853f;
  float u0 = rng_next(g);
  float u1 = rng_next(g);
  v3 N = unit3(n);
  v3 Vw = unit3(V(-d_in.x, -d_in.y, -d_in.z));
  float ndv = dot3(N, Vw);
  float sg = copysignf(1.0f, N.z);
  float a = -1.0f / (sg + N.z);
  float b = N.x * N.y * a;
  v3 T = V(1.0f + sg * N.x * N.x * a, sg * b, -sg * N.x);
  v3 B = V(b, sg + N.y * N.y * a, -N.y);
  int spec = ndv > 0.0f && u0 < 0.5f;
  float u0r = u0 < 0.5f ? u0 * 2.0f : u0 * 2.0f - 1.0f;
  float al = roughness;
  float phi = kTwoPi * u1;
  float sp = cr_sin(phi), cp = cr_cos(phi);
  float r = sqrtf(u0r);
  v3 l;
  if (spec) {
    v3 Vh = unit3(V(al * dot3(Vw, T), al * dot3(Vw, B), ndv));
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
    v3 h = add3(add3(scale3(T, hl.x), scale3(B, hl.y)), scale3(N, hl.z));
    l = sub3(scale3(h, 2.0f * dot3(Vw, h)), Vw);
  } else {
    l = add3(add3(scale3(T, r * cp), scale3(B, r * sp)), scale3(N, sqrtf(fmaxf(0.0f, 1.0f - u0r))));
  }
  float pdf = glossy_mix_pdf(al, N, Vw, l);
  /* the reference's uniform sampler weighs with 2 * 3.14 where the true density is 1 / (2 pi): its expectation is
   * 3.14 / pi times the integral.  Kept, so that both samplers converge to the same image. */
  *inv_pdf = pdf > 0.0f ? (3.14f / kPi) / pdf : 0.0f;
  return l;
}

/* =========================================================================================
 * BSDFs — MathLib.cl:461-512
 * ======================================================================================= */
static inline float ipow(float x, int n) { float r = 1.0f; for (int i = 0; i < n; ++i) r = r * x; return r; }

static v3 bsdf_ggx(const mat_t *m, v3 v, v3 l, v3 n) {
  v3 h = unit3(add3(l, v));
  float a2 = ipow(m->roughness, 2);
  float D = a2 / (3.14f * ipow(ipow(fmaxf(dot3(n, h), 0.0f), 2) * (a2 - 1.0f) + 1.0f, 2));
  float ndv = fmaxf(dot3(n, v), 0.0f);
  float kk = m->roughness * sqrtf(2.0f / 3.14f);
  float g1 = ndv / (ndv * (1.0f - kk) + kk);
  float ndl = fmaxf(dot3(n, l), 0.0f);
  float g2 = ndl / (ndl * (1.0f - kk) + kk);
  float G = g1 * g2;
  float F = 0.04f + (1 - 0.04f) * ipow(1.0f - fmaxf(dot3(h, v), 0.0f), 5);
  float spec = (F * G * D) * (1.0f / fmaxf(4.0f * fmaxf(dot3(v, n), 0.0f) * fmaxf(dot3(l, n), 0.0f), 0.001f));
  float kd = (1.0f - F) * (1.0f - 0.5f);
  v3 diffuse = div3s(scale3(m->color, kd), 3.14f);
  /* kd * color is commutative per component, so scale3(color,kd) rounds identically */
  return V(diffuse.x + spec, diffuse.y + spec, diffuse.z + spec);
}

/* ---- opt-in light sampling (orc_opts.sampling bit 1) -----------------------------------------------------------------
 * NOT in the reference, whose kernel receives lightData and never reads it (Raytracing.cl:163); the author's intent is
 * the dead sampleLight, MathLib.cl:404-454.  At every surface that scatters (types 1, 2) one emitter triangle is chosen
 * uniformly from lightData and one point uniformly on it; a shadow ray decides visibility.  The emitter is then reachable
 * two ways — by this light sample and by the surface's own direction sample happening to hit it — and both are kept with
 * balance-heuristic weights p / (p_light + p_bsdf) (densities per solid angle), which keeps the estimate bounded next to a
 * large emitter where light sampling alone has unbounded variance.  Same expectation as the reference's estimator:
 * emission is the material's power (roughness slot, Raytracing.cl:105-109) from both faces, the diffuse factor is
 * color / pi and the glossy one 3.14 / pi x BRDF_GGX, which is what the reference's samplers converge to.
 * Mirrors csrc/rt_shade.cuh statement by statement. */

/* density per solid angle with which the light sampler reaches the point at squared distance dist2 along unit direction
 * wi on emitter triangle t; 0 when the triangle is seen edge-on */
static float light_pdf(const scene_t *sc, int t, v3 wi, float dist2) {
  const int *f = sc->face + 10 * t;
  const float *pa = sc->vp + 3 * f[7], *pb = sc->vp + 3 * f[8], *pc = sc->vp + 3 * f[9];
  v3 A = V(pa[0], pa[1], pa[2]);
  v3 e1 = sub3(V(pb[0], pb[1], pb[2]), A);
  v3 e2 = sub3(V(pc[0], pc[1], pc[2]), A);
  v3 NL = cross3(e1, e2);
  float area2 = sqrtf(dot3(NL, NL));
  float cosL = fabsf(dot3(NL, wi)) / area2;
  if (!(cosL > 0.0f) || !(area2 > 0.0f)) return 0.0f;
  return dist2 / ((cosL * ((float)sc->n_light * 0.5f)) * area2);
}

/* density per solid angle with which the surface's own sampler draws unit direction l (M.type 1 or 2) */
static float bsdf_pdf(const scene_t *sc, const mat_t *M, v3 n, v3 d_in, v3 l) {
  const float kPi = 3.14159265f;
  v3 N = unit3(n);
  float ndl = dot3(N, l);
  if (M->type == 1) return fmaxf(ndl, 0.0f) / kPi;
  if (sc->sampling & 1) return glossy_mix_pdf(M->roughness, N, unit3(V(-d_in.x, -d_in.y, -d_in.z)), l);
  return ndl > 0.0f ? 1.0f / (2.0f * kPi) : 0.0f;
}

static v3 sample_light(const scene_t *sc, const mat_t *M, v3 n, v3 x, v3 d_in, v3 acc, const float u[3], ray_t *shadow,
                       int *target) {
  const float kPi = 3.14159265f;
  int idx = (int)(u[0] * (float)sc->n_light);
  if (idx > sc->n_light - 1) idx = sc->n_light - 1;
  int t = sc->light[idx];
  const int *f = sc->face + 10 * t;
  const float *pa = sc->vp + 3 * f[7], *pb = sc->vp + 3 * f[8], *pc = sc->vp + 3 * f[9];
  v3 A = V(pa[0], pa[1], pa[2]);
  v3 e1 = sub3(V(pb[0], pb[1], pb[2]), A);
  v3 e2 = sub3(V(pc[0], pc[1], pc[2]), A);
  mat_t ML = material_at(sc, f[0]);
  float Le = ML.type == 0 ? ML.roughness : 0.0f;
  float ua = u[1], ub = u[2];
  if (ua + ub > 1.0f) { ua = 1.0f - ua; ub = 1.0f - ub; }
  v3 y = add3(add3(A, scale3(e1, ua)), scale3(e2, ub));
  v3 w = sub3(y, x);
  float dist2 = dot3(w, w);
  float dist = sqrtf(dist2);
  v3 wi = div3s(w, dist);
  float cosS = dot3(wi, unit3(n));
  v3 fr;
  if (M->type == 1) {
    fr = scale3(M->color, 1.0f / kPi);
  } else {
    fr = scale3(bsdf_ggx(M, V(-d_in.x, -d_in.y, -d_in.z), wi, n), 3.14f / kPi);
  }
  shadow->o = x;
  shadow->d = w;
  *target = t;
  if (!(cosS > 0.0f) || !(dist2 > 0.0f)) return V(0.0f, 0.0f, 0.0f);
  float pl = light_pdf(sc, t, wi, dist2);
  if (!(pl > 0.0f)) return V(0.0f, 0.0f, 0.0f);
  float pb_ = bsdf_pdf(sc, M, n, d_in, wi);
  return scale3(mul3(acc, fr), (cosS * Le) / (pl + pb_));
}

/* three uniforms for the light sample of bounce j: the generator's next three values in reference mode, the second
 * Philox block of (pixel, sample, bounce) otherwise (the first block feeds the direction sampling) */
static void rng_light3(rng_t *g, uint32_t pixel, uint32_t sample, uint32_t bounce, float u[3]) {
  if (g->mode == 0) {
    u[0] = rng_next(g); u[1] = rng_next(g); u[2] = rng_next(g);
    return;
  }
  uint32_t ctr[4] = {pixel, sample, bounce, 1u}, out[4];
  philox4x32_10(ctr, g->key0, g->key1, out);
  tl_cnt.rand_calls += 3;
  u[0] = bits_to_unit(out[0]); u[1] = bits_to_unit(out[1]); u[2] = bits_to_unit(out[2]);
}

/* =========================================================================================
 * One sample — Raytracing.cl:39-153
 * ======================================================================================= */
static v3 sun_direction(const scene_t *sc) { /* Raytracing.cl:115-118 */
  v3 s = V(1, 1, 1);
  s = rotate_about(sc->env[0] * DEG2RAD, V(1, 0, 0), s);
  s = rotate_about(sc->env[1] * DEG2RAD, V(0, 1, 0), s);
  s = rotate_about(sc->env[2] * DEG2RAD, V(0, 0, 1), s);
  return s;
}

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

/* =========================================================================================
 * Entry points
 * ======================================================================================= */
static void fill_scene(scene_t *sc, const float *vp, const float *vn, const float *vuv, const int *face,
                       const float *mat, const float *bvh, const float *cam, const float *env,
                       int tri_count, const unsigned char *ibl, int ibl_w, int ibl_h, int stack_cap) {
  sc->sampling = 0;
  sc->n_light = 0;
  sc->light = NULL;
  sc->vp = vp; sc->vn = vn; sc->vuv = vuv; sc->face = face; sc->mat = mat; sc->bvh = bvh;
  sc->cam = cam; sc->env = env; sc->tri_count = tri_count;
  sc->ibl = ibl; sc->ibl_w = ibl_w; sc->ibl_h = ibl_h;
  sc->stack_cap = (stack_cap <= 0) ? 20 : (stack_cap > 64 ? 64 : stack_cap);
}

/* `Raytracing` work-items [i0,i1) of an img_size-item launch — Raytracing.cl:161-221.
 * out: img_size*3 floats (only [i0,i1) written). */
void orc_render(float *out, const float *vp, const float *vn, const float *vuv, const int *face,
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
      g.a = (uint32_t)(i % img_size); /* Raytracing.cl:171-172; imgSize receives imgDim */
      g.b = (uint32_t)(i / img_size);
      g.key0 = opts->seed_lo;
      g.key1 = opts->seed_hi;
      ray_t r = camera_ray(&sc, i);
      hit_t H0 = closest_hit(&sc, &r);
      mat_t M0 = material_at(&sc, H0.mat);
      v3 sum = V(0.0f, 0.0f, 0.0f);
      for (int s = s0; s < s1; ++s) {
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

/* primary ray of work-items [i0,i1): direction, kept triangle (-1 = miss), distance, material */
void orc_primary(const float *vp, const float *vn, const float *vuv, const int *face, const float *bvh,
                 const float *cam, int tri_count, int stack_cap, int i0, int i1, float *dir_out,
                 int *tri_out, float *k_out, int *mat_out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, NULL, bvh, cam, NULL, tri_count, NULL, 0, 0, stack_cap);
#pragma omp parallel for schedule(dynamic, 256)
  for (int i = i0; i < i1; ++i) {
    ray_t r = camera_ray(&sc, i);
    hit_t h = closest_hit(&sc, &r);
    size_t o = (size_t)(i - i0);
    dir_out[3 * o] = r.d.x; dir_out[3 * o + 1] = r.d.y; dir_out[3 * o + 2] = r.d.z;
    tri_out[o] = h.hit ? h.tri : -1;
    k_out[o] = h.k;
    mat_out[o] = h.mat;
  }
}

/* closest hit of n arbitrary rays (o,d packed 6 floats each) — used to check traversal alone */
void orc_trace_rays(const float *vp, const float *vn, const float *vuv, const int *face, const float *bvh,
                    int tri_count, int stack_cap, const float *rays, int n, int *tri_out, float *k_out,
                    unsigned long long *counters_out) {
  scene_t sc;
  fill_scene(&sc, vp, vn, vuv, face, NULL, bvh, NULL, NULL, tri_count, NULL, 0, 0, stack_cap);
  unsigned long long c1 = 0, c2 = 0;
#pragma omp parallel reduction(+ : c1, c2)
  {
    memset(&tl_cnt, 0, sizeof tl_cnt);
#pragma omp for schedule(dynamic, 256)
    for (int i = 0; i < n; ++i) {
      ray_t r;
      r.o = V(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]);
      r.d = V(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
      hit_t h = closest_hit(&sc, &r);
      tri_out[i] = h.hit ? h.tri : -1;
      k_out[i] = h.k;
    }
    c1 += tl_cnt.box_tests; c2 += tl_cnt.tri_tests;
  }
  if (counters_out) { counters_out[0] = (unsigned long long)n; counters_out[1] = c1; counters_out[2] = c2; counters_out[3] = 0; }
}

/* ImgProcessing.cl:1-9 over work-items [0,global) */
void orc_img_processing(const float *in, float *out, int n, int global) {
  for (int i = 0; i < global; ++i) {
    if (i < n) {
      float p = in[i];
      p = (1.0f < p) ? 1.0f : p; /* OpenCL min(x,y) = y < x ? y : x */
      out[i] = cr_pow(p, 2.2f);
    }
  }
}

/* n draws of the per-pixel stream (mode 0) or of one (pixel,sample,bounce) Philox block sequence */
void orc_rand_stream(int mode, uint32_t pixel, uint32_t img_size, uint32_t seed_lo, uint32_t seed_hi,
                     uint32_t sample, uint32_t bounce, int n, float *out) {
  rng_t g;
  memset(&g, 0, sizeof g);
  g.mode = mode;
  g.a = pixel % img_size; g.b = pixel / img_size;
  g.key0 = seed_lo; g.key1 = seed_hi;
  rng_set_bounce(&g, pixel, sample, bounce);
  for (int i = 0; i < n; ++i) out[i] = rng_next(&g);
}

void orc_philox(const uint32_t ctr[4], uint32_t k0, uint32_t k1, uint32_t out[4]) {
  philox4x32_10(ctr, k0, k1, out);
}

/* single-function probes so the GPU's device math can be compared value by value */
void orc_math_probe(int fn, const float *a, const float *b, int n, float *out) {
  for (int i = 0; i < n; ++i) {
    switch (fn) {
      case 0: out[i] = cr_sin(a[i]); break;
      case 1: out[i] = cr_cos(a[i]); break;
      case 2: out[i] = cr_acos(a[i]); break;
      case 3: out[i] = cr_asin(a[i]); break;
      case 4: out[i] = cr_atan2(a[i], b[i]); break;
      case 5: out[i] = cr_tan(a[i]); break;
      case 6: out[i] = cr_pow(a[i], b[i]); break;
      case 7: out[i] = a[i] / b[i]; break;
      case 8: out[i] = sqrtf(a[i]); break;
      default: out[i] = 0.0f;
    }
  }
}

void orc_rotate(float angle, const float *axis, const float *vec, float *out) {
  v3 r = rotate_about(angle, V(axis[0], axis[1], axis[2]), V(vec[0], vec[1], vec[2]));
  out[0] = r.x; out[1] = r.y; out[2] = r.z;
}
