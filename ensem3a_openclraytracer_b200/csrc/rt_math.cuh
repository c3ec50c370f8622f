// Device arithmetic of the b200rt kernels.
//
// Numerical contract (DESIGN.md "Arithmetic"): every + - * / sqrt is IEEE binary32
// round-to-nearest and is never contracted (this translation unit is compiled with
// -fmad=false; FMAs appear only where written as __fmaf_rn), dot products are summed
// left to right, normalize divides, and the transcendental built-ins of the reference
// kernels (cos sin acos asin atan2 powr; MathLib.cl) are CORRECTLY ROUNDED binary32,
// obtained by evaluating in binary64 and rounding once.  B200 runs binary64 at half the
// binary32 rate, so this costs a few percent of a path and buys results that are
// independent of any vendor's float libm.
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

namespace b200rt {

struct v3 {
  float x, y, z;
};
struct quat {
  float w, x, y, z;
};

#define RT_DEV __device__ __forceinline__
#define RT_HD __host__ __device__ __forceinline__

RT_HD v3 mk3(float x, float y, float z) {
  v3 r;
  r.x = x; r.y = y; r.z = z;
  return r;
}
RT_HD v3 operator+(v3 a, v3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_HD v3 operator-(v3 a, v3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_HD v3 operator*(v3 a, v3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
RT_HD v3 operator*(v3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_HD v3 operator/(v3 a, float s) { return mk3(a.x / s, a.y / s, a.z / s); }
RT_HD v3 neg3(v3 a) { return mk3(-a.x, -a.y, -a.z); }
RT_HD float dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
RT_HD v3 cross(v3 a, v3 b) {
  return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
RT_HD v3 unit(v3 a) { return a / sqrtf(dot(a, a)); }

// fmax(fmin(x, 1), 0) with OpenCL/IEEE minNum semantics (Raytracing.cl:217-219): a NaN becomes 1, not 0.
// nvcc fuses the plain fmaxf(fminf(x,1),0) into FADD.SAT, whose NaN result is +0, so NaN is handled
// explicitly (tests/test_gpu_parity.py::test_nan_and_inf_semantics_survive).
RT_DEV float clamp01(float x) {
  float t = fmaxf(fminf(x, 1.0f), 0.0f);
  return (x != x) ? 1.0f : t;
}

// ---- correctly-rounded binary32 transcendentals (binary64 evaluation, one rounding) ----
// A binary64 value within e ulps of the true value, rounded once, is the correctly rounded binary32 unless the true value
// lies within e binary64 ulps of a binary32 rounding boundary.  CUDA's binary64 acos / asin / pow are within 2 ulp, and on
// the domains the kernels reach (every float with |x| <= 1 for acos / asin, 0 < p <= 1 for pow(p, 2.2f)) every input
// where that matters is known: tests/golden/make_cr_hard_cases.py lists each float whose binary64 value lies within 64
// binary64 ulps of a boundary, with its correctly rounded result (cr_hard_cases.inc: 84 acos, 68 asin, 122 pow).  These
// routines take their value from that table whenever their own binary64 result lies within kCrTieGuard ulps of a boundary,
// so they are correctly rounded on all of those domains; without it, acos was wrong on 2 of its 2.13e9 inputs.
// tests/test_gpu_arith_exhaustive.py compares every input of the domains with the oracle.  Elsewhere (exponents other
// than 2.2f, tan, atan2, the probes' cr_sin / cr_cos, cr_sincos beyond |a| <= 8) the once-rounded binary64 value is
// returned, correctly rounded except within ~2 binary64 ulps of a boundary; those inputs are only sampled.
#include "cr_hard_cases.inc"
constexpr long long kCrTieGuard = 16;  // binary64 ulps; the oracle's CR_TIE_GUARD (oracle/cr_tie.h)

// distance of |r| from the nearer binary32 rounding boundary around it, in binary64 ulps (the boundary is the mean of
// two neighbouring floats, exact in binary64, so the one below a power of two is found at a quarter ulp)
RT_DEV long long cr_tie_dist(double r) {
  const double a = fabs(r);
  if (!(a <= 3.4028234663852886e38)) return LLONG_MAX;
  const float f = __double2float_rn(a);
  const unsigned fb = __float_as_uint(f);
  const long long ab = __double_as_longlong(a);
  long long d = __double_as_longlong(0.5 * ((double)f + (double)__uint_as_float(fb + 1u))) - ab;
  if (fb != 0u) d = min(d, ab - __double_as_longlong(0.5 * ((double)f + (double)__uint_as_float(fb - 1u))));
  return d;
}

// The correctly rounded binary32 value of the binary64 result r of a routine at input x: the once-rounded r, or the table
// entry of x where r lies within kCrTieGuard binary64 ulps of a rounding boundary.  Where |r| is in the normal binary32
// range the boundaries inside its binade are where the 29 low mantissa bits read 2^28 (the one just below the next power
// of two included), so integer operations on the low word filter; the rare rest (and anything below 2^-126) goes out of
// line to cr_tie_dist and the table, sorted by input bits, in which x is looked up (r rounded once if x is not listed).
#define RT_NOINLINE __device__ __noinline__
RT_NOINLINE float cr_hard_case(const uint32_t (*t)[2], int n, float x, double r) {
  if (cr_tie_dist(r) <= kCrTieGuard) {
    const uint32_t k = __float_as_uint(x);
    int lo = 0, hi = n - 1;
    while (lo <= hi) {
      const int m = (lo + hi) >> 1;
      const uint32_t v = t[m][0];
      if (v == k) return __uint_as_float(t[m][1]);
      if (v < k) lo = m + 1;
      else hi = m - 1;
    }
  }
  return __double2float_rn(r);
}
RT_DEV float cr_round(const uint32_t (*t)[2], int n, float x, double r) {
  const unsigned lo = (unsigned)__double2loint(r) & 0x1fffffffu;
  const bool tiny = (__double2hiint(r) & 0x7fffffff) < 0x38100000;  // |r| < 2^-126
  if (tiny || lo - (0x10000000u - (unsigned)kCrTieGuard) <= 2u * (unsigned)kCrTieGuard) return cr_hard_case(t, n, x, r);
  return __double2float_rn(r);
}

// The binary64 routines are large; they are kept out of line so that the shading code holds one copy of each
// and stays resident in the instruction cache next to the traversal loop.
RT_NOINLINE float cr_sin(float a) { return __double2float_rn(sin((double)a)); }
RT_NOINLINE float cr_cos(float a) { return __double2float_rn(cos((double)a)); }
RT_NOINLINE float2 cr_sincos2(float a) {  // (sin, cos), any argument
  double ds, dc;
  sincos((double)a, &ds, &dc);
  return make_float2(__double2float_rn(ds), __double2float_rn(dc));
}
// The samplers only take sines and cosines of angles in [0, 2·3.14] (MathLib.cl:316,344-345).  For |a| <= 8 the
// binary64 evaluation is done here directly: Cody–Waite reduction by pi/2 in two parts (exact for |k| <= 6),
// then the classic minimax kernels on [-pi/4, pi/4] (error < 1 ulp of binary64).  Its arithmetic is fixed, so its
// correct rounding is a fact about these 2.18e9 inputs, not an estimate: tests/test_gpu_arith_exhaustive.py compares
// every one of them with the oracle (0 disagreements; the 120 inputs of the hard-case list are all correctly rounded),
// and it needs no table.  A third of the instructions of the general routine and no branches, which matters in a kernel
// whose lanes are already scattered over material types.
RT_DEV void cr_sincos(float a, float *s, float *c) {
  if (!(fabsf(a) <= 8.0f)) {
    float2 r = cr_sincos2(a);
    *s = r.x;
    *c = r.y;
    return;
  }
  const double x = (double)a;
  const double kd = rint(x * 6.36619772367581382433e-01);            // 2/pi
  double r = fma(-kd, 1.57079632673412561417e+00, x);                // pi/2, first 33 bits
  r = fma(-kd, 6.07710050650619224932e-11, r);                       // pi/2 - the above
  const double z = r * r;
  double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
  ps = fma(z, ps, 2.75573137070700676789e-06);
  ps = fma(z, ps, -1.98412698298579493134e-04);
  ps = fma(z, ps, 8.33333333332248946124e-03);
  ps = fma(z, ps, -1.66666666666666324348e-01);
  const double sn = fma(z * r, ps, r);
  double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
  pc = fma(z, pc, -2.75573143513906633035e-07);
  pc = fma(z, pc, 2.48015872894767294178e-05);
  pc = fma(z, pc, -1.38888888888741095749e-03);
  pc = fma(z, pc, 4.16666666666666019037e-02);
  const double cs = fma(z * z, pc, fma(z, -0.5, 1.0));
  const int n = (int)kd & 3;
  const double sv = (n & 1) ? cs : sn, cv = (n & 1) ? sn : cs;
  const float sf = __double2float_rn((n & 2) ? -sv : sv);
  *s = (a == 0.0f) ? a : sf;  // sin(-0) = -0
  *c = __double2float_rn(((n + 1) & 2) ? -cv : cv);
}
RT_NOINLINE float cr_tan(float a) { return __double2float_rn(tan((double)a)); }
RT_NOINLINE float cr_acos(float a) { return cr_round(cr_hard_acos, CR_HARD_ACOS_N, a, acos((double)a)); }
RT_NOINLINE float cr_asin(float a) { return cr_round(cr_hard_asin, CR_HARD_ASIN_N, a, asin((double)a)); }
RT_NOINLINE float cr_atan2(float y, float x) { return __double2float_rn(atan2((double)y, (double)x)); }
RT_NOINLINE float cr_pow(float a, float b) {  // the table holds the exponent 2.2f (the tonemap's) only
  const double r = pow((double)a, (double)b);
  return b == 2.2f ? cr_round(cr_hard_pow, CR_HARD_POW_N, a, r) : __double2float_rn(r);
}

// ---- quaternion rotation, MathLib.cl:51-65 ------------------------------------------------
RT_HD quat qmul(quat q, quat p) {
  v3 qv = mk3(q.x, q.y, q.z), pv = mk3(p.x, p.y, p.z);
  quat r;
  r.w = q.w * p.w - dot(qv, pv);
  v3 t = ((qv * p.w) + (pv * q.w)) + cross(qv, pv);
  r.x = t.x; r.y = t.y; r.z = t.z;
  return r;
}

// The pair (q, normalised scaled conjugate) the reference builds for one rotateVec call.
struct rotor {
  quat q, qi;
};

RT_HD rotor make_rotor(float c, float s, v3 axis) {  // c = cos(angle/2), s = sin(angle/2), correctly rounded
  v3 sv = unit(axis) * s;
  rotor r;
  r.q.w = c; r.q.x = sv.x; r.q.y = sv.y; r.q.z = sv.z;
  float n2 = c * c + dot(sv, sv);
  v3 ng = sv * (-1.0f);
  float uw = c * n2, ux = ng.x * n2, uy = ng.y * n2, uz = ng.z * n2;
  float len = sqrtf(uw * uw + ux * ux + uy * uy + uz * uz);
  r.qi.w = uw / len; r.qi.x = ux / len; r.qi.y = uy / len; r.qi.z = uz / len;
  return r;
}

RT_HD v3 apply_rotor(const rotor &r, v3 v) {
  quat p;
  p.w = 0.0f; p.x = v.x; p.y = v.y; p.z = v.z;
  quat o = qmul(qmul(r.q, p), r.qi);
  return mk3(o.x, o.y, o.z);
}

// ---- random numbers ---------------------------------------------------------------------------
RT_HD float bits_to_unit(uint32_t bits) {  // MathLib.cl:302-309
#ifdef __CUDA_ARCH__
  float f = __uint_as_float((bits & 0x007fffffu) | 0x40000000u);
#else
  union { float f; uint32_t u; } cvt;
  cvt.u = (bits & 0x007fffffu) | 0x40000000u;
  float f = cvt.f;
#endif
  return (f - 2.0f) / 2.0f;
}

RT_DEV void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                          uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Two uniform draws for bounce `j` of sample `s` of pixel `i`.
struct rng_state {
  // Reference generator (MathLib.cl:294-310) as the kernel wires it: Raytracing.cl:205-206 passes
  // (&seed0,&seed1), naiveGI swaps them for the samplers (:61-69), so on the kernel's own words
  // seed1 <- 36969*(seed0&65535)+(seed0>>16); seed0 <- 18000*(seed1&65535)+(seed1>>16); bits = (seed1<<16)+seed0.
  // The incoming seed1 is never read: the whole state is seed0.
  uint32_t a;
};

template <int RNG>
RT_DEV void draw2(rng_state &g, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t k0, uint32_t k1,
                  float *u0, float *u1) {
  if (RNG == 0) {
    uint32_t b = 36969u * (g.a & 65535u) + (g.a >> 16);
    uint32_t a = 18000u * (b & 65535u) + (b >> 16);
    *u0 = bits_to_unit((b << 16) + a);
    b = 36969u * (a & 65535u) + (a >> 16);
    a = 18000u * (b & 65535u) + (b >> 16);
    *u1 = bits_to_unit((b << 16) + a);
    g.a = a;
  } else {
    uint32_t o[4];
    philox4x32_10(pixel, sample, bounce, 0u, k0, k1, o);
    *u0 = bits_to_unit(o[0]);
    *u1 = bits_to_unit(o[1]);
  }
}

// One uniform draw for bounce `j` (opt-in refractive glass): draw2's first value, i.e. the generator's next value in
// reference mode, word 0 of the Philox block (pixel, sample, bounce, 0) otherwise.
template <int RNG>
RT_DEV float draw1(rng_state &g, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t k0, uint32_t k1) {
  if (RNG == 0) {
    const uint32_t b = 36969u * (g.a & 65535u) + (g.a >> 16);
    const uint32_t a = 18000u * (b & 65535u) + (b >> 16);
    g.a = a;
    return bits_to_unit((b << 16) + a);
  }
  uint32_t o[4];
  philox4x32_10(pixel, sample, bounce, 0u, k0, k1, o);
  return bits_to_unit(o[0]);
}

// Three uniform draws for bounce `j`: the generator's next three values in reference mode, words 0, 1 and 2 of the
// Philox block (pixel, sample, bounce, n) otherwise.  The light sample (opt-in light sampling) uses n = 1, the block
// after the one draw2 reads; rough glass (opt-in) n = 0, the block draw2 reads, which a glass hit never draws from.
template <int RNG>
RT_DEV void draw3(rng_state &g, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t n, uint32_t k0, uint32_t k1,
                  float *u0, float *u1, float *u2) {
  if (RNG == 0) {
    float u[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const uint32_t b = 36969u * (g.a & 65535u) + (g.a >> 16);
      const uint32_t a = 18000u * (b & 65535u) + (b >> 16);
      u[i] = bits_to_unit((b << 16) + a);
      g.a = a;
    }
    *u0 = u[0]; *u1 = u[1]; *u2 = u[2];
  } else {
    uint32_t o[4];
    philox4x32_10(pixel, sample, bounce, n, k0, k1, o);
    *u0 = bits_to_unit(o[0]);
    *u1 = bits_to_unit(o[1]);
    *u2 = bits_to_unit(o[2]);
  }
}

// The two uniforms of a sample's jittered camera ray (opt-in pixel jitter), drawn when the sample starts: the
// generator's next two values in reference mode, words 0 and 1 of the Philox block (pixel, sample, 0, 2) otherwise.
template <int RNG>
RT_DEV void draw2_jitter(rng_state &g, uint32_t pixel, uint32_t sample, uint32_t k0, uint32_t k1, float *ux, float *uy) {
  if (RNG == 0) {
    draw2<0>(g, pixel, sample, 0u, k0, k1, ux, uy);
  } else {
    uint32_t o[4];
    philox4x32_10(pixel, sample, 0u, 2u, k0, k1, o);
    *ux = bits_to_unit(o[0]);
    *uy = bits_to_unit(o[1]);
  }
}

}  // namespace b200rt
