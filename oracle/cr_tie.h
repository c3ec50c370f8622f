/* TEST INFRASTRUCTURE — how close a binary64 value lies to a binary32 rounding boundary.
 *
 * The oracle (rt_oracle.c), the reference shim (ref_shim/cl_shim.h) and the hard-case generator
 * (tests/golden/make_cr_hard_cases.py) share this one definition; the kernels restate it in
 * csrc/rt_math.cuh (cr_tie_dist).  C and C++.
 *
 * cr_tie_dist(r): the distance, counted in binary64 ulps (bit patterns), from |r| to the nearer of the two
 * binary32 rounding boundaries (midpoints) that enclose it, i.e. to the boundary of the interval that rounds
 * to RN32(|r|).  The boundary below a power of two lies at a quarter of the upper ulp and is found as
 * such, because it is computed as the mean of two neighbouring floats, which binary64 holds exactly.
 * A binary64 evaluation with an error of e ulps, rounded once to binary32, is the correctly rounded
 * value whenever cr_tie_dist of the computed value exceeds e.  Non-finite values and values above
 * FLT_MAX give INT64_MAX.
 */
#ifndef CR_TIE_H
#define CR_TIE_H
#include <math.h>
#include <stdint.h>
#include <string.h>

/* binary64 ulps of distance below which the oracle re-evaluates a function in extended precision
 * (and the kernels look the input up in their table of hard cases) */
#define CR_TIE_GUARD 16

static inline int64_t cr_tie_dist(double r) {
  const double a = fabs(r);
  if (!(a <= 3.4028234663852886e38)) return INT64_MAX;
  const float f = (float)a;
  uint32_t fb, nb;
  float nf;
  int64_t ab, mb, best;
  memcpy(&fb, &f, 4);
  memcpy(&ab, &a, 8);
  nb = fb + 1u;
  memcpy(&nf, &nb, 4);
  const double up = 0.5 * ((double)f + (double)nf);
  memcpy(&mb, &up, 8);
  best = mb - ab;
  if (fb != 0u) {
    nb = fb - 1u;
    memcpy(&nf, &nb, 4);
    const double dn = 0.5 * ((double)f + (double)nf);
    memcpy(&mb, &dn, 8);
    if (ab - mb < best) best = ab - mb;
  }
  return best;
}

#endif
