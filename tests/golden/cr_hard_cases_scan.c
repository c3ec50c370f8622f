/* Binary64 pass of make_cr_hard_cases.py: every binary32 input in [lo, hi] (bit patterns) through glibc's binary64
 * function, and the inputs whose result lies within `window` binary64 ulps of a binary32 rounding boundary
 * (oracle/cr_tie.h).  glibc's binary64 functions are within 1 ulp, so every input whose once-rounded result could
 * differ from the correctly rounded one is among them as long as the window exceeds that error.  OpenMP over the
 * inputs; the flagged ones are returned unsorted. */
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../oracle/cr_tie.h"

static inline double eval(int fn, float x) {
  switch (fn) {
    case 0: return sin((double)x);
    case 1: return cos((double)x);
    case 2: return acos((double)x);
    case 3: return asin((double)x);
    default: return pow((double)x, (double)2.2f);
  }
}

/* fn: 0 sin, 1 cos, 2 acos, 3 asin, 4 pow(x, 2.2f).  Returns the number of flagged inputs (only the first `cap`
 * are stored). */
int64_t cr_scan(int fn, uint32_t lo, uint32_t hi, int64_t window, uint32_t *out, int64_t cap) {
  int64_t cnt = 0;
#pragma omp parallel for schedule(dynamic, 1 << 18)
  for (int64_t i = (int64_t)lo; i <= (int64_t)hi; ++i) {
    const uint32_t u = (uint32_t)i;
    float x;
    memcpy(&x, &u, 4);
    if (cr_tie_dist(eval(fn, x)) <= window) {
      int64_t k;
#pragma omp atomic capture
      k = cnt++;
      if (k < cap) out[k] = u;
    }
  }
  return cnt;
}

/* glibc's binary64 result rounded once, for the flagged inputs */
void cr_eval(int fn, const uint32_t *in, int64_t n, float *out) {
  for (int64_t i = 0; i < n; ++i) {
    float x;
    memcpy(&x, &in[i], 4);
    out[i] = (float)eval(fn, x);
  }
}
