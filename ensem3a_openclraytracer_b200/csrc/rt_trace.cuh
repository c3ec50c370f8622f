// BVH traversal and ray/triangle intersection for the b200rt kernels.
//
// Contract: every closest-hit routine here returns, for any ray, exactly the (triangle, distance) the
// reference's rayTrace() keeps (MathLib.cl:234-288):
//   * a triangle is a CANDIDATE iff the slab test of MathLib.cl:167-190 — six TRUE divisions, a line/box
//     test with no clipping to t >= 0 — passes for its leaf box and for every ancestor box, and
//     Möller–Trumbore (MathLib.cl:117-160) reports k > 1e-7 with the reference's u/v rejections;
//   * among candidates with 1e-4 < k < 1000 the smallest k wins; equal k is resolved in favour of the
//     triangle the reference visits first (it pushes left then right, so it walks right-first).
//
// Implementations:
//   closest_hit_reference  the reference's own visiting order on the as-is 9-float nodes, including its
//                          capped stack that silently drops pushes (stack.cl:21-26);
//   closest_hit_nodrop     the same walk with a stack that never drops (the fallback of the fast path, and the
//                          path of rays whose direction has a zero / denormal / huge component);
//   closest_hit_fast       the production path.  It rests on one observation about the reference's slab test:
//
//       For a ray whose direction components are all non-zero finite numbers, if a box B' is nested in a
//       box B (B.min <= B'.min <= B'.max <= B.max per axis) then slab(B') passing implies slab(B) passing.
//       Proof: RN(p - o) and RN(x / d) are monotone in p resp. x, so per axis the floating-point interval
//       [min(t1,t2), max(t1,t2)] of B contains that of B'; hence tmin(B) <= tmin(B') and tmax(B) >= tmax(B'),
//       and tmax(B') >= tmin(B') gives tmax(B) >= tmin(B).  (No NaN can arise: x / d with d != 0.)
//
//     BVH.py builds every node box as the exact float32 min/max over the node's triangles (BVH.py:43-70), so
//     boxes are nested along every root-to-leaf chain (b200rt_set_scene verifies this; a tree that violates it
//     is walked by closest_hit_reference).  A triangle is therefore a candidate iff its LEAF box passes the
//     exact slab test and Möller–Trumbore accepts it; ancestor boxes matter for culling only.  The fast path
//     walks the tree with a CONSERVATIVE slab test (FMAs only, on boxes stored as centre / half-extent and
//     widened by a proven error margin), runs
//     the exact Möller–Trumbore on the leaves it reaches, and keeps the best hit; the winner's leaf box is
//     then put through the exact slab test once (validate_hit).  If it passes — always, except for rays that
//     graze a box edge within rounding — the winner is the reference's hit: the set searched is a superset of
//     the candidates and its minimum is a candidate.  If it fails the ray is re-traced by closest_hit_nodrop.
#pragma once
#include "rt_math.cuh"

namespace b200rt {

// ---- repacked scene -------------------------------------------------------------------------------
// node (32 B = 8 words, ONE 256-bit load per visit; 32 B apart in global memory, 48 B apart when the scene is
// staged in shared memory so that lanes reading different nodes spread over all bank groups), interior nodes only,
// root = 0.  A record holds the boxes of BOTH children as planes on a 2^15 grid spanning the root box:
//   w0 = L.x   w1 = L.y   w2 = L.z   w3 = R.x   w4 = R.y   w5 = R.z     one axis of one child per word:
//                                                   grid index of the max plane << 16 | grid index of the min plane
//   w6 = refL  w7 = refR                            ref >= 0: float4 offset of an interior node (index x node_f4),
//                                                   ref < 0: leaf of triangle ~ref
// Decoding is ONE instruction per plane and no conversion: PRMT drops the 15-bit index q into mantissa bits 22..8 under
// the exponent of 0.5, giving the binary32 fq = 0.5 + q / 65536 exactly; in real arithmetic the plane lies at
// grid_base + fq * grid_pitch.  Which half of the word a ray enters through (its NEAR plane) depends only on the sign of
// its direction on that axis, so every ray carries the two PRMT selectors per axis and a box costs six FMAs:
//     near = fma(fq_near, A, Bn),   far = fma(fq_far, A, Bf)          (slab_cons below)
// b200rt_set_scene chooses the indices so that [min plane, max plane] ENCLOSES the child's exact float32 [min, max]
// (checked there in binary64).  These boxes only cull; exactness lives in the leaf boxes of `tboxes` and in the as-is
// array `bvh9`.  History: round 1 read two boxes as 12 floats (64 B, two 256-bit loads; ncu had the L1TEX data pipe
// of k_trace at 83 %); the first 32-byte record held centre / half-extent pairs and cost twelve FMAs per box.
// triangle (48 B, 3 x float4):
//   t0 = A.x A.y A.z e1.x     t1 = e1.y e1.z e2.x e2.y     t2 = e2.z mat rank -   (mat, rank int bits)
//   with e1 = B - A, e2 = C - A rounded exactly as MathLib.cl:129-130 rounds them.
// normal (16 B): first-vertex normal of the triangle (MathLib.cl:151), w unused.
// leaf box (32 B, 2 x float4): min.xyz -, max.xyz -   of the leaf that holds the triangle (validate_hit).
struct SceneView {
  const uint4 *nodes;
  int node_f4;              // 16-byte units per node: 2, or 3 for a scene small enough to be staged in shared memory
  const float4 *tris;       // by triangle id
  const float4 *ctris;      // the same records in the order of the culling tree's leaves: what leaf refs index and the
                            // traversal tests (staged in shared memory for small scenes); t2.w = triangle id
  const float4 *normals;
  const float4 *tboxes;
  const float4 *frames;     // kFrameVec float4 per triangle (rt_shade.cuh)
  const float *mats;        // 6 floats per material
  // as-is reference buffers for closest_hit_reference
  const float *bvh9;
  const int *leafcnt;       // leaves in the sub-tree of each node of bvh9 (validate_chain)
  int root_ref;             // ~tri when the whole tree is one leaf
  float grid_base[3];       // decoded centre = grid_base + fc * grid_pitch   (fc in [0.5, 1))
  float grid_pitch[3];
  uint32_t root_w[3];       // node 0's box, one word per axis in the format of the node records (enclosing, like them)
  float cull_abs;           // absolute part of the culling margin (1e-3 x scene diagonal)
  uint32_t st_bias;         // traversal-stack entries (LaneStack): binary32 bits of 2^(E - 32), where 2^E bounds every culling limit
  uint32_t st_rmask;        //   and the mask of the low bits that hold the node ref
  float cmax;               // largest |coordinate| of any box plane, vertex or grid point
  int stack_cap;            // reference traversal
  int fast_ok;              // scene coordinates in the range the conservative test is proven for
};

struct TraceCounters {
  unsigned long long box_tests, tri_tests;
};

struct Hit {
  int tri;    // -1 = miss
  float k;    // 1000 on a miss, like H.k (MathLib.cl:239)
};

// Path state is read once per kernel and streams through the SM: these loads do not allocate a line in L1, which is
// left to the nodes and triangles the lanes come back to.
RT_DEV float4 ld_stream(const float4 *p) {
  float4 v;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
RT_DEV int2 ld_stream(const int2 *p) {
  int2 v;
  asm volatile("ld.global.L1::no_allocate.v2.s32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
RT_DEV int ld_stream(const int *p) {
  int v;
  asm volatile("ld.global.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
RT_DEV float ld_stream(const float *p) {
  float v;
  asm volatile("ld.global.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

template <bool SMEM>
RT_DEV float4 ld4(const float4 *p) {
  if (SMEM) return *p;
  return __ldg(p);
}

// triangle record `t` of `tris` or `ctris` (format above), decoded; SMEM: the copy staged in shared memory
struct Tri {
  v3 A, e1, e2;
  int mat, rank, id;   // id: ctris records only
};
template <bool SMEM = false>
RT_DEV Tri load_tri(const float4 *tris, int t) {
  const float4 *p = tris + 3 * (size_t)t;
  const float4 t0 = ld4<SMEM>(p), t1 = ld4<SMEM>(p + 1), t2 = ld4<SMEM>(p + 2);
  return {mk3(t0.x, t0.y, t0.z), mk3(t0.w, t1.x, t1.y), mk3(t1.z, t1.w, t2.x), __float_as_int(t2.y), __float_as_int(t2.z),
          __float_as_int(t2.w)};
}

// material id / visiting rank of triangle `tri`: the record's third float4 alone
RT_DEV int tri_material(const SceneView &S, int tri) { return __float_as_int(__ldg(S.tris + 3 * (size_t)tri + 2).y); }
RT_DEV int tri_rank(const SceneView &S, int tri) { return __float_as_int(__ldg(S.tris + 3 * (size_t)tri + 2).z); }

// One node = 32 contiguous bytes: one 256-bit load from global memory (LDG.E.256, sm_100+), two 128-bit loads from
// shared memory.  Lanes of a warp sit at unrelated nodes, so the L1 cost of a node visit is one wavefront per lane
// per load instruction.
template <bool SMEM>
RT_DEV void ld_node(const uint4 *p, uint4 &a, uint4 &b) {
  if (SMEM) {
    a = p[0]; b = p[1];
  } else {
    asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
        : "l"(p));
  }
}

constexpr uint32_t kSelMax = 0x7324u;   // PRMT selector: 0.5 + (w >> 16) / 65536      (the max plane of a node word)
constexpr uint32_t kSelMin = 0x7104u;   //                0.5 + (w & 0xffff) / 65536   (the min plane)
// prmt.b32 directly: __byte_perm() is specified to look at three bits per selector nibble only, so the compiler masks a
// selector that lives in a register with 0x7777 before every use — six extra instructions per node visit
RT_DEV float plane_fq(uint32_t w, uint32_t sel) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0x3f000000u), "r"(sel));
  return __uint_as_float(r);
}

// ---- exact slab test, MathLib.cl:169-188 --------------------------------------------------------------
// x / d, IEEE round-to-nearest.  The hardware division routine sends a zero numerator to its out-of-line slow path
// (~40 instructions behind a call), and zero numerators are the common case here: a ray leaving a wall at z = -1 and
// tested against a box that starts at z = -1.  (+-0) / d is the zero with the sign of x XOR d for every d other than
// 0 and NaN, which this returns directly.
RT_DEV float div_exact(float x, float d) {
  if (x == 0.0f && d != 0.0f && d == d) return __uint_as_float((__float_as_uint(x) ^ __float_as_uint(d)) & 0x80000000u);
  return __fdiv_rn(x, d);
}

RT_DEV bool slab_exact(v3 o, v3 d, float mnx, float mny, float mnz, float mxx, float mxy, float mxz, float *tmin,
                       float *tmax) {
  float a = div_exact(mnx - o.x, d.x), b = div_exact(mxx - o.x, d.x);
  float lo = fminf(a, b), hi = fmaxf(a, b);
  a = div_exact(mny - o.y, d.y); b = div_exact(mxy - o.y, d.y);
  lo = fmaxf(lo, fminf(a, b));
  hi = fminf(hi, fmaxf(a, b));
  a = div_exact(mnz - o.z, d.z); b = div_exact(mxz - o.z, d.z);
  lo = fmaxf(lo, fminf(a, b));
  hi = fminf(hi, fmaxf(a, b));
  *tmin = lo;
  *tmax = hi;
  return hi >= lo;
}

// ---- conservative slab test ----------------------------------------------------------------------------
// A box is held per axis as two grid planes fq_min <= fq_max, a plane lying at x = base + fq * pitch in real arithmetic,
// with [x_min, x_max] enclosing the exact [min, max].  Per ray and axis: r = RN(1/d),
//     A = RN(pitch * r),   B = RN(RN(base - o) * r),   Bn = B - m,   Bf = B + m,
//     near = fma(fq_near, A, Bn),   far = fma(fq_far, A, Bf),      fq_near = A >= 0 ? fq_min : fq_max, fq_far the other
// — one FMA per plane, no per-axis min / max because the sign of A orders the two planes (the ray carries the PRMT
// selectors that pick them out of the node word).  The three `near` and the three `far` values are reduced with one
// 3-input max / min each to lo and hi.
// Error budget per axis, in units of u (cmax + |o|) |r| with u = 2^-24.  b200rt_set_scene makes cmax bound every
// |box plane|, |vertex coordinate|, |base| and |base + pitch|, hence pitch <= 2 cmax and |x| <= cmax for every decoded
// plane.  A = RN(pitch·r), scaled by fq < 1: 2.  B: one rounding of base - o (<= cmax + |o|) and one of the product: 2.
// Bn / Bf: 1.  r (the hardware's approximate reciprocal, within 1 ulp) against 1/d: 2.  The FMA: 2 (|result| <= (2 cmax + |o|)|r| + m).  Together 9.  The reference's own
// t = RN(RN(p - o) / d) is within 2 of the real (p - o)/d.  The margin, PER AXIS (a ray with one tiny direction
// component must not lose the culling of the other two axes),
//     m = 2^-18 (cmax + |o|) |r|        (= 64 units, six times the sum of 11),
// gives  lo <= tmin_exact  and  hi >= tmax_exact: the box certainly fails the reference's test when hi < lo.
// Valid while every |d| component lies in [2^-40, 2^40] and |o|, cmax <= 2^40 (no overflow, no denormal r).
struct RayFast {
  v3 A, Bn, Bf;
  uint32_t sn[3], sf[3];   // PRMT selectors of the near / far plane per axis (kSelMin / kSelMax)
};

RT_DEV bool comp_ok(float d) {
  float a = fabsf(d);
  return a >= 9.094947017729282e-13f /* 2^-40 */ && a <= 1.099511627776e12f /* 2^40 */;
}

// every direction component is a non-zero finite number of moderate size: "the leaf box passes => every ancestor
// box passes" holds and validate_hit decides; otherwise validate_chain does
RT_DEV bool ray_is_regular(v3 d) { return comp_ok(d.x) && comp_ok(d.y) && comp_ok(d.z); }

// the conservative traversal applies (any direction; the scene and the origin are in the range the margins are proven for)
RT_DEV bool ray_is_fast(const SceneView &S, v3 o) {
  return S.fast_ok != 0 && fabsf(o.x) <= 1.099511627776e12f && fabsf(o.y) <= 1.099511627776e12f &&
         fabsf(o.z) <= 1.099511627776e12f;
}

// Irregular axes (ray_is_regular fails; the reference's test then involves infinities and NaNs, MathLib.cl:169-188):
//   * |d| < 2^-40, zero and denormals included: the ray's coordinate on this axis is practically constant.  The axis is
//     tested as if r were +-2^40 with the margin enlarged by 1002 + 2 cull_abs: a box whose (decoded) slab holds the
//     origin's coordinate gets an interval that covers [-cull_abs, 1001 + cull_abs] — everything the traversal can
//     still be interested in, so no constraint — and a slab further than ~2^-18 (cmax + |o|) from the coordinate fails,
//     as it does in the reference (both quotients +inf or both -inf, or beyond every distance of interest).
//   * |d| > 2^40, infinite or NaN: no constraint (A = 0, Bn = -inf, Bf = +inf give near = -inf, far = +inf).
// Either way the reference can only be stricter, so the traversal still visits a superset of the candidates;
// validate_chain then decides whether the winner is one.
RT_DEV void rayfast_axis(float o, float d, float cmax, float cull_abs, float base, float pitch, float *A, float *Bn,
                         float *Bf, uint32_t *sn, uint32_t *sf) {
  const float a = fabsf(d);
  const bool neg = (__float_as_uint(d) >> 31) != 0u;   // the sign of A = pitch * r (pitch > 0)
  *sn = neg ? kSelMax : kSelMin;
  *sf = neg ? kSelMin : kSelMax;
  float rr, extra = 0.0f;
  if (a >= 9.094947017729282e-13f /* 2^-40 */ && a <= 1.099511627776e12f /* 2^40 */) {
    // the hardware approximation (within 1 ulp of 1/d: 2 units of the budget above instead of 1; no denormal in or out
    // for |d| in [2^-40, 2^40]) — these intervals only cull, and the correctly rounded reciprocal costs four times as much
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rr) : "f"(d));
  } else if (a < 9.094947017729282e-13f) {
    rr = copysignf(1.099511627776e12f, d);
    extra = 1002.0f + 2.0f * cull_abs;
  } else {
    *A = 0.0f;
    *Bn = -INFINITY;
    *Bf = INFINITY;
    return;
  }
  const float b = (base - o) * rr;
  const float m = (3.814697265625e-06f /* 2^-18 */ * (cmax + fabsf(o))) * fabsf(rr) + extra;
  *A = pitch * rr;
  *Bn = b - m;
  *Bf = b + m;
}

RT_DEV RayFast make_rayfast(const SceneView &S, v3 o, v3 d) {
  RayFast Q;
  rayfast_axis(o.x, d.x, S.cmax, S.cull_abs, S.grid_base[0], S.grid_pitch[0], &Q.A.x, &Q.Bn.x, &Q.Bf.x, &Q.sn[0], &Q.sf[0]);
  rayfast_axis(o.y, d.y, S.cmax, S.cull_abs, S.grid_base[1], S.grid_pitch[1], &Q.A.y, &Q.Bn.y, &Q.Bf.y, &Q.sn[1], &Q.sf[1]);
  rayfast_axis(o.z, d.z, S.cmax, S.cull_abs, S.grid_base[2], S.grid_pitch[2], &Q.A.z, &Q.Bn.z, &Q.Bf.z, &Q.sn[2], &Q.sf[2]);
  return Q;
}

// lo <= tmin_exact and hi >= tmax_exact of the box whose three axis words are (wx, wy, wz); the box certainly fails
// when hi < lo
RT_DEV void slab_cons(const RayFast &Q, uint32_t wx, uint32_t wy, uint32_t wz, float *lo, float *hi) {
  const float nx = __fmaf_rn(plane_fq(wx, Q.sn[0]), Q.A.x, Q.Bn.x);
  const float ny = __fmaf_rn(plane_fq(wy, Q.sn[1]), Q.A.y, Q.Bn.y);
  const float nz = __fmaf_rn(plane_fq(wz, Q.sn[2]), Q.A.z, Q.Bn.z);
  const float fx = __fmaf_rn(plane_fq(wx, Q.sf[0]), Q.A.x, Q.Bf.x);
  const float fy = __fmaf_rn(plane_fq(wy, Q.sf[1]), Q.A.y, Q.Bf.y);
  const float fz = __fmaf_rn(plane_fq(wz, Q.sf[2]), Q.A.z, Q.Bf.z);
  *lo = fmaxf(fmaxf(nx, ny), nz);
  *hi = fminf(fminf(fx, fy), fz);
}

// ---- Möller–Trumbore, MathLib.cl:117-160 ---------------------------------------------------------------
// Returns true and k when the reference's intersect() sets bHit.
RT_DEV bool tri_hit(v3 o, v3 d, v3 A, v3 e1, v3 e2, float *k_out) {
  const float eps = 0.0000001f;
  v3 h = cross(d, e2);
  float a = dot(e1, h);
  if (a > -eps && a < eps) return false;
  float f = __frcp_rn(a);  // (float)(1.0 / (double)a) == RN(1/a): the double rounding is innocuous for a reciprocal
  v3 s = o - A;
  float u = f * dot(s, h);
  if (u < 0.0f || u > 1.0f) return false;
  v3 q = cross(s, e1);
  float v = f * dot(d, q);
  if (v < 0.0f || u + v > 1.0f) return false;
  float k = f * dot(e2, q);
  if (k > eps) { *k_out = k; return true; }
  return false;
}

template <bool SMEM>
RT_DEV void test_triangle(const SceneView &S, int leaf, v3 o, v3 d, Hit &best, int &best_rank) {
  const Tri t = load_tri<SMEM>(S.ctris, leaf);
  float k;
  if (tri_hit(o, d, t.A, t.e1, t.e2, &k) && k > 0.0001f) {
    if (k < best.k || (k == best.k && best.tri >= 0 && t.rank < best_rank)) {
      best.k = k;
      best.tri = t.id;
      best_rank = t.rank;
    }
  }
}

// the exact slab test of the leaf box that holds triangle `tri` (global memory: once per ray)
RT_DEV bool validate_hit(const SceneView &S, v3 o, v3 d, int tri) {
  const float4 mn = __ldg(S.tboxes + 2 * (size_t)tri), mx = __ldg(S.tboxes + 2 * (size_t)tri + 1);
  float lo, hi;
  return slab_exact(o, d, mn.x, mn.y, mn.z, mx.x, mx.y, mx.z, &lo, &hi);
}

// The reference accepts a triangle only if the exact slab test passes for its leaf box AND every ancestor box.  For
// a regular ray the leaf implies the ancestors (see the top of this file).  With a zero direction component the test
// involves (b - o) / 0: a plane the origin lies exactly on gives 0/0 = NaN, which fmin / fmax drop, and then an
// ancestor whose plane coincides with the origin's coordinate can fail although a (zero-thickness) leaf passes.  So
// for such rays the winner's whole root-to-leaf chain is put through the exact test: one descent without a stack,
// steered by the leaf's rank in the reference's visiting order (right sub-tree first, MathLib.cl:275-280) and the
// number of leaves under each node.  Canonical trees only (two children per interior node).
__device__ __noinline__ bool validate_chain(const SceneView &S, v3 o, v3 d, int tri, int rank) {
  int node = 0, first = 0;   // ranks [first, first + leafcnt[node]) live under `node`
  for (;;) {
    const float *n = S.bvh9 + 9 * (size_t)node;
    float lo, hi;
    if (!slab_exact(o, d, __ldg(n + 2), __ldg(n + 3), __ldg(n + 4), __ldg(n + 5), __ldg(n + 6), __ldg(n + 7), &lo, &hi))
      return false;
    const int t = (int)__ldg(n + 8);
    if (t != -1) return t == tri;
    const int l = (int)__ldg(n), r = (int)__ldg(n + 1);
    const int under_r = __ldg(S.leafcnt + r);
    if (rank < first + under_r) {
      node = r;
    } else {
      first += under_r;
      node = l;
    }
  }
}

// the winner of the conservative walk (triangle `tri`, visiting rank `rank`) is the reference's hit iff this holds
RT_DEV bool validate_winner(const SceneView &S, v3 o, v3 d, int tri, int rank) {
  return ray_is_regular(d) ? validate_hit(S, o, d, tri) : validate_chain(S, o, d, tri, rank);
}

// ---- reference-order traversal ---------------------------------------------------------------------------
constexpr int kRefStack = 64;   // b200rt_set_scene routes trees that need more to REFERENCE mode with the caller's cap

template <bool STATS>
RT_DEV Hit closest_hit_reference_cap(const SceneView &S, v3 o, v3 d, TraceCounters *cnt, const int cap) {
  Hit best;
  best.tri = -1;
  best.k = 1000.0f;
  int stack[kRefStack];
  int top = -1;
  stack[++top] = 0;
  while (top != -1) {
    int cur = stack[top--];
    const float *n = S.bvh9 + 9 * (size_t)cur;
    float tmin, tmax;
    if (STATS) cnt->box_tests++;
    if (!slab_exact(o, d, __ldg(n + 2), __ldg(n + 3), __ldg(n + 4), __ldg(n + 5), __ldg(n + 6), __ldg(n + 7), &tmin, &tmax))
      continue;
    int t = (int)__ldg(n + 8);
    if (t != -1) {
      if (STATS) cnt->tri_tests++;
      const Tri tr = load_tri(S.tris, t);
      float k;
      if (tri_hit(o, d, tr.A, tr.e1, tr.e2, &k) && k < best.k && k > 0.0001f) {
        best.k = k;
        best.tri = t;
      }
    }
    int l = (int)__ldg(n), r = (int)__ldg(n + 1);
    if (l != -1 && top != cap - 1) stack[++top] = l;
    if (r != -1 && top != cap - 1) stack[++top] = r;
  }
  return best;
}

template <bool STATS>
RT_DEV Hit closest_hit_reference(const SceneView &S, v3 o, v3 d, TraceCounters *cnt) {
  return closest_hit_reference_cap<STATS>(S, o, d, cnt, S.stack_cap);
}

// The reference's walk with a stack that cannot drop: what the fast path computes, obtained the slow way.  Out of
// line: reached only by rays with a zero / denormal / huge direction component and by the (very rare) rays whose
// fast-path winner fails validate_hit.
__device__ __noinline__ Hit closest_hit_nodrop(const SceneView &S, v3 o, v3 d) {
  TraceCounters dummy;
  return closest_hit_reference_cap<false>(S, o, d, &dummy, kRefStack);
}

// ---- fast traversal ---------------------------------------------------------------------------------------------
// Per-lane stack in shared memory: entry e of lane l lives at stack[e * stride + l] (bank-conflict free).
// An entry is ONE word, (distance code | node ref): the ref (16-byte offset of an interior node) in the low bits that
// SceneView::st_rmask covers, and above it the leading bits of the sub-tree's conservative entry distance, coded so
// that the word order is the distance order:
//     code(x) = (max(bits(x), st_bias) - st_bias) << 4,   bits() = the binary32 pattern read as a signed integer.
// st_bias is the pattern of 2^(E-32) with 2^E above every culling limit (1001 + cull_abs), so a pushed distance
// (always <= the limit of the moment) has bits(x) - st_bias < 2^28 and the shift loses nothing; negative distances and
// everything below 2^(E-32) code as 0.  code() is monotone, hence  code(lo) > code(lim)  implies  lo > lim: a pop may
// skip such an entry, exactly as the comparison of the full distances would, only a little less often (the code keeps
// 5 exponent bits and 27 - log2(refs) mantissa bits; a bench-scene entry keeps 12).  Half the bytes of the round-1
// (ref, distance) pair: the stacks of the resident CTAs are carved out of the SM's L1, which the node fetches need.
struct LaneStack {
  uint32_t *base;   // already offset to this thread
  int stride;       // threads per block
};

RT_DEV uint32_t stack_code(const SceneView &S, float x) {
  return (uint32_t)(max(__float_as_int(x), (int)S.st_bias) - (int)S.st_bias) << 4;
}

// One traversal in flight.  Kept in registers; advanced one node at a time so that a warp can interleave
// node steps, leaf tests and ray refills of its 32 lanes (k_trace), or simply looped (closest_hit_fast).
struct Trav {
  v3 o, d;
  RayFast Q;
  Hit best;
  int best_rank;
  float lim;     // sub-trees whose conservative entry distance exceeds this cannot hold a closer hit
  int cur, sp;   // cur: 16-byte offset of the node to visit next; < 0: the walk has ended
};

RT_DEV bool trav_active(const Trav &T) { return T.cur >= 0; }

RT_DEV float cull_limit(const SceneView &S, const Trav &T) { return __fmaf_rn(T.best.k, 1.001f, S.cull_abs); }

// Leaves whose box passes the conservative test are not tested on the spot (only a few lanes of a warp reach a
// leaf in the same turn) but parked, at most kParkCap per lane (entry e of lane l at parks[e * stride]); the
// warp tests parked triangles together.  Last in, first out; of a pair of leaves the farther is parked first.
constexpr int kParkCap = 6;

// starts a traversal of a ray for which ray_is_fast() holds
template <bool SMEM, bool STATS>
RT_DEV void trav_begin(const SceneView &S, Trav &T, v3 o, v3 d, int &pn, uint32_t *parks, TraceCounters *cnt) {
  T.o = o; T.d = d;
  T.Q = make_rayfast(S, o, d);
  T.best.tri = -1;
  T.best.k = 1000.0f;
  T.best_rank = 0x7fffffff;
  T.lim = cull_limit(S, T);
  T.sp = 0;
  float lo, hi;
  if (STATS) cnt->box_tests++;
  slab_cons(T.Q, S.root_w[0], S.root_w[1], S.root_w[2], &lo, &hi);
  const bool go = hi >= lo;
  T.cur = go ? 0 : -1;
  if (go && S.root_ref < 0) {
    parks[0] = (uint32_t)S.root_ref;
    pn = 1;
    T.cur = -1;
  }
}

// one node: both child boxes through the conservative test; leaf children are parked as their (negative) refs
// (needs pn <= kParkCap - 2)
template <bool SMEM, bool STATS>
RT_DEV void trav_step(const SceneView &S, Trav &T, int &pn, uint32_t *parks, int pstride, LaneStack st,
                      TraceCounters *cnt) {
  uint4 wa, wb;
  ld_node<SMEM>(S.nodes + T.cur, wa, wb);
  const int refL = (int)wb.z, refR = (int)wb.w;
  float loL, hiL, loR, hiR;
  if (STATS) cnt->box_tests += 2;
  slab_cons(T.Q, wa.x, wa.y, wa.z, &loL, &hiL);
  slab_cons(T.Q, wa.w, wb.x, wb.y, &loR, &hiR);
  const float lim = T.lim;
  const float behind = -S.cull_abs;
  const bool goL = hiL >= loL && !(loL > lim) && !(hiL < behind);
  const bool goR = hiR >= loR && !(loR > lim) && !(hiR < behind);
  const bool leafL = goL && refL < 0, leafR = goR && refR < 0;
  const bool inL = goL && refL >= 0, inR = goR && refR >= 0;
  // one comparison orders both the leaves (nearer leaf parked last = tested first) and the interior children
  const bool rNear = loR < loL;
  const int refNear = rNear ? refR : refL, refFar = rNear ? refL : refR;
  const bool both = leafL && leafR;
  if (both) { parks[pn * pstride] = (uint32_t)refFar; ++pn; }
  if (leafL || leafR) { parks[pn * pstride] = (uint32_t)(both ? refNear : (leafR ? refR : refL)); ++pn; }
  if (inL && inR) {
    st.base[T.sp * st.stride] = (stack_code(S, rNear ? loL : loR) & ~S.st_rmask) | (uint32_t)refFar;
    ++T.sp;
    T.cur = refNear;
  } else if (inL || inR) {
    T.cur = inL ? refL : refR;
  } else {
    T.cur = -1;
    const uint32_t keep = stack_code(S, lim) | S.st_rmask;   // entries above this lie beyond the culling limit
    while (T.sp > 0) {
      --T.sp;
      const uint32_t e = st.base[T.sp * st.stride];
      if (e <= keep) {
        T.cur = (int)(e & S.st_rmask);
        break;
      }
    }
  }
}

// a parked leaf: exact Möller–Trumbore, then the culling limit follows the best hit
template <bool SMEM>
RT_DEV void test_parked(const SceneView &S, Trav &T, uint32_t ref, v3 o, v3 d) {
  test_triangle<SMEM>(S, ~(int)ref, o, d, T.best, T.best_rank);
  T.lim = cull_limit(S, T);
}

// the whole walk by one thread (k_primary, k_trace_rays, verify mode); `parks` = kParkCap words of this thread
template <bool SMEM, bool STATS>
RT_DEV Hit closest_hit_fast(const SceneView &S, v3 o, v3 d, LaneStack st, uint32_t *parks, int pstride,
                            TraceCounters *cnt) {
  if (!ray_is_fast(S, o)) return closest_hit_nodrop(S, o, d);
  Trav T;
  int pn = 0;
  trav_begin<SMEM, STATS>(S, T, o, d, pn, parks, cnt);
  while (trav_active(T) || pn > 0) {
    if (pn > 0 && (!trav_active(T) || pn > kParkCap - 2)) {
      --pn;
      if (STATS) cnt->tri_tests++;
      test_parked<SMEM>(S, T, parks[pn * pstride], o, d);
    } else {
      trav_step<SMEM, STATS>(S, T, pn, parks, pstride, st, cnt);
    }
  }
  if (T.best.tri >= 0 && !validate_winner(S, o, d, T.best.tri, T.best_rank)) return closest_hit_nodrop(S, o, d);
  return T.best;
}

// TRAV: 0 fast, 1 reference, 2 verify (both; keeps reference, counts disagreements)
template <int TRAV, bool SMEM, bool STATS>
RT_DEV Hit closest_hit(const SceneView &S, v3 o, v3 d, LaneStack st, uint32_t *parks, int pstride, TraceCounters *cnt,
                       unsigned int *mismatch) {
  if (TRAV == 0) return closest_hit_fast<SMEM, STATS>(S, o, d, st, parks, pstride, cnt);
  if (TRAV == 1) return closest_hit_reference<STATS>(S, o, d, cnt);
  Hit a = closest_hit_reference<STATS>(S, o, d, cnt);
  TraceCounters dummy;
  dummy.box_tests = 0; dummy.tri_tests = 0;
  Hit b = closest_hit_fast<SMEM, false>(S, o, d, st, parks, pstride, &dummy);
  if (a.tri != b.tri || __float_as_int(a.k) != __float_as_int(b.k)) (*mismatch)++;
  return a;
}

}  // namespace b200rt
