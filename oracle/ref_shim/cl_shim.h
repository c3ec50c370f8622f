// TEST INFRASTRUCTURE — not part of the product path.
//
// OpenCL-C compatibility shim that lets g++ compile the reference's own
// Kernels/*.cl (after the two mechanical regex rewrites done by
// oracle/build_ref.py) as host C++.  Nothing here restates the reference's
// algorithm; it only pins down the arithmetic of the OpenCL *built-ins* the
// reference calls, which no OpenCL driver documents to the last bit
// (SURVEY.md §8c "third-party arithmetic").  The canonical choices:
//
//   + - * /  sqrt          IEEE-754 binary32, round-to-nearest-even, never
//                          contracted (compile with -ffp-contract=off)
//   dot                    x*x + y*y + z*z (+ w*w), left to right
//   normalize(v)           v / sqrt(dot(v,v))   (true divisions)
//   cos sin tan acos asin atan2 powr
//                          CORRECTLY ROUNDED binary32: evaluated by the host
//                          libm in binary64 and rounded once to binary32;
//                          where that value lies within CR_TIE_GUARD binary64
//                          ulps of a binary32 rounding boundary (../cr_tie.h)
//                          cos / sin (|x| <= 8), acos, asin and powr(x, 2.2f)
//                          are evaluated again in x87 extended precision and
//                          that is rounded.  Checked against mpmath on every
//                          float of those domains (tests/test_cr_hard_cases.py;
//                          the once-rounded binary64 value alone was wrong on
//                          2 of 2.13e9 acos inputs, 0 elsewhere).  tan and
//                          atan2 are the once-rounded binary64 value, wrong
//                          only within ~1 binary64 ulp of a boundary; sampled.
//                          Same rule as oracle/rt_oracle.c.
//                          Correct rounding is the one definition every
//                          conforming implementation — CPU or GPU — can meet
//                          independently, which is what makes a bit-exact
//                          CPU/GPU comparison meaningful.
//   pown(x,n)              repeated multiply from 1
//   fmin/fmax              IEEE minNum/maxNum (NaN dropped), as OpenCL says
//   (int2)(float,float)    C truncation
//   read_imagef            integer coords, clamp-to-edge, UNORM_INT8: b/255.0f
//
// -DCLREF_LIBM_FLOAT switches the transcendental set to glibc's binary32
// functions (cosf, sinf, ...) — used only to quantify how much the result
// depends on the last bit of the built-ins.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#include "../cr_tie.h"

namespace clref {

// ---- address-space / kernel qualifiers ------------------------------------
#define __global
#define __constant
#define __kernel
#define __read_only
#define __write_only
#define __private
#define __local

// ---- counters (only in the counting build) --------------------------------
struct Counters {
  unsigned long long rays, box_tests, tri_tests, rand_calls;
};
extern thread_local Counters g_cnt;
#ifdef CLREF_COUNTERS
#define CLREF_COUNT(field) (++::clref::g_cnt.field)
#else
#define CLREF_COUNT(field) ((void)0)
#endif

// ---- work-item id -----------------------------------------------------------
extern thread_local int g_global_id;
static inline int get_global_id(int) { return g_global_id; }

// ---- scalar built-ins ---------------------------------------------------------
#ifdef CLREF_LIBM_FLOAT
static inline float cos(float x) { return ::cosf(x); }
static inline float sin(float x) { return ::sinf(x); }
static inline float tan(float x) { return ::tanf(x); }
static inline float acos(float x) { return ::acosf(x); }
static inline float asin(float x) { return ::asinf(x); }
static inline float atan2(float y, float x) { return ::atan2f(y, x); }
static inline float powr(float x, float y) { return ::powf(x, y); }
#else
static inline float cos(float x) {
  const double r = ::cos((double)x);
  return (::fabsf(x) <= 8.0f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)::cosl((long double)x) : (float)r;
}
static inline float sin(float x) {
  const double r = ::sin((double)x);
  return (::fabsf(x) <= 8.0f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)::sinl((long double)x) : (float)r;
}
static inline float tan(float x) { return (float)::tan((double)x); }
static inline float acos(float x) {
  const double r = ::acos((double)x);
  return cr_tie_dist(r) <= CR_TIE_GUARD ? (float)::acosl((long double)x) : (float)r;
}
static inline float asin(float x) {
  const double r = ::asin((double)x);
  return cr_tie_dist(r) <= CR_TIE_GUARD ? (float)::asinl((long double)x) : (float)r;
}
static inline float atan2(float y, float x) { return (float)::atan2((double)y, (double)x); }
static inline float powr(float x, float y) {
  const double r = ::pow((double)x, (double)y);
  return (y == 2.2f && cr_tie_dist(r) <= CR_TIE_GUARD) ? (float)::powl((long double)x, (long double)y) : (float)r;
}
#endif
static inline float sqrt(float x) { return ::sqrtf(x); }
static inline float fabs(float x) { return ::fabsf(x); }
static inline float fmin(float a, float b) { return ::fminf(a, b); }
static inline float fmax(float a, float b) { return ::fmaxf(a, b); }
static inline float min(float a, float b) { return b < a ? b : a; }
static inline float pown(float x, int n) {
  float r = 1.0f;
  for (int i = 0; i < n; ++i) r = r * x;
  return r;
}
static inline int convert_int_rte(float x) { return (int)::nearbyintf(x); }
// a double argument reaching one of these would silently change precision:
double cos(double) = delete;
double sin(double) = delete;
double tan(double) = delete;
double acos(double) = delete;
double asin(double) = delete;
double sqrt(double) = delete;
double fabs(double) = delete;

// ---- vector types ---------------------------------------------------------------
struct float2 {
  float x, y;
  float2() {}
  float2(float s) : x(s), y(s) {}
  float2(float a, float b) : x(a), y(b) {}
};
struct float3 {
  float x, y, z;
  float3() {}
  float3(float s) : x(s), y(s), z(s) {}
  float3(float a, float b, float c) : x(a), y(b), z(c) {}
};
struct float4 {
  float x, y, z, w;
  float4() {}
  float4(float s) : x(s), y(s), z(s), w(s) {}
  float4(float a, float b, float c, float d) : x(a), y(b), z(c), w(d) {}
  float4(float a, const float3 &v) : x(a), y(v.x), z(v.y), w(v.z) {}
  float3 yzw() const { return float3(y, z, w); }
  float3 xyz() const { return float3(x, y, z); }
};
struct int2 {
  int x, y;
  int2() {}
  int2(float a, float b) : x((int)a), y((int)b) {}
};

#define CLREF_VEC_OP2(op)                                                        \
  static inline float2 operator op(const float2 &a, const float2 &b) {           \
    return float2(a.x op b.x, a.y op b.y);                                       \
  }                                                                              \
  static inline float3 operator op(const float3 &a, const float3 &b) {           \
    return float3(a.x op b.x, a.y op b.y, a.z op b.z);                           \
  }                                                                              \
  static inline float4 operator op(const float4 &a, const float4 &b) {           \
    return float4(a.x op b.x, a.y op b.y, a.z op b.z, a.w op b.w);               \
  }
CLREF_VEC_OP2(+)
CLREF_VEC_OP2(-)
CLREF_VEC_OP2(*)
CLREF_VEC_OP2(/)
#undef CLREF_VEC_OP2
static inline float3 operator-(const float3 &a) { return float3(-a.x, -a.y, -a.z); }
static inline float3 &operator+=(float3 &a, const float3 &b) {
  a = a + b;
  return a;
}

static inline float dot(const float3 &a, const float3 &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline float dot(const float4 &a, const float4 &b) {
  return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}
static inline float3 cross(const float3 &a, const float3 &b) {
  return float3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static inline float length(const float3 &a) { return sqrt(dot(a, a)); }
static inline float3 normalize(const float3 &a) { return a / float3(sqrt(dot(a, a))); }
static inline float4 normalize(const float4 &a) { return a / float4(sqrt(dot(a, a))); }

// ---- images -------------------------------------------------------------------------
struct image2d_t {
  int w, h;
  const unsigned char *rgba;  // row-major, top row first, 4 bytes per texel
};
typedef int sampler_t;
enum { CLK_NORMALIZED_COORDS_FALSE = 0, CLK_ADDRESS_CLAMP_TO_EDGE = 2, CLK_FILTER_LINEAR = 16 };
static inline int get_image_width(const image2d_t &im) { return im.w; }
static inline int get_image_height(const image2d_t &im) { return im.h; }
static inline float4 read_imagef(const image2d_t &im, sampler_t, const int2 &c) {
  int x = c.x < 0 ? 0 : (c.x > im.w - 1 ? im.w - 1 : c.x);
  int y = c.y < 0 ? 0 : (c.y > im.h - 1 ? im.h - 1 : c.y);
  const unsigned char *p = im.rgba + 4 * ((size_t)y * (size_t)im.w + (size_t)x);
  return float4(p[0] / 255.0f, p[1] / 255.0f, p[2] / 255.0f, p[3] / 255.0f);
}

}  // namespace clref
