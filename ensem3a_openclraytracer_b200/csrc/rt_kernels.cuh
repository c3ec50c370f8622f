// b200rt kernels (sm_100a).  One frame = k_primary, then (s1 - s0) * (max_bounce + 2) wavefront iterations of
// k_shade + k_trace, then one closing k_shade:
//
//   k_primary   one thread per pixel: camera ray + closest hit; stores the hit (the parity artefact), finishes
//               every pixel whose samples need no further ray (primary miss or emitter) and appends every other
//               pixel to the first path list.
//   k_shade     one thread per live path (= pixel; its samples run strictly in order): resolves the ray traced in
//               the previous iteration (Raytracing.cl:91-137), ends / starts samples, samples the next direction
//               (:51-87), and appends the path to the next list with a warp-aggregated atomic (ballot + popc).
//               Every live path leaves k_shade with exactly one ray to trace.
//   k_trace     persistent warps pull rays from the list (a chunk per warp per atomic), keep 32 traversals in
//               registers and advance them one node per turn; leaves are parked in shared memory and tested by
//               the warp together; a lane whose ray is done writes the hit and is refilled from the list, so
//               the node loop stays full whatever the individual traversal lengths.
//   k_reduce_finalize / k_img_processing   the accumulate / clamp / tonemap passes.
// An adaptive frame (b200rt_render_adaptive) runs k_adaptive_init before k_primary and k_shade<NEE, true>, whose
// end_sample block also applies the stopping rule (adaptive_end_sample); the host ends its loop once the list is empty.
// A jittered frame (opt-in pixel jitter) runs k_jitter_init instead of k_primary and k_shade<NEE, false, true>, in
// which every sample traces its own camera ray: one more wavefront iteration per sample.
#pragma once
#include "rt_shade.cuh"
#include "rt_trace.cuh"

namespace b200rt {

constexpr int kBlock = 128;        // k_primary, k_trace, k_trace_rays
constexpr int kShadeBlock = 128;
constexpr unsigned kChunk = 32;    // rays a warp claims from the list per atomic (64 / 128 lose to the longer tails)
// k_trace's lane scheduling: the node phase ends when fewer than kQuorum lanes can step; idle lanes pull new rays once
// kRefillMin are idle; the leaf phase repeats while at least kTriQuorum lanes hold a parked leaf
constexpr int kQuorum = 12, kRefillMin = 8, kTriQuorum = 2;
constexpr int kCompactEvery = 4;   // k_shade(i) hands its output to k_compact when (i + 1) % kCompactEvery == 0
constexpr int kHitNeedsExactWalk = -2;  // pHit.x of a ray k_trace did not walk (see k_trace); k_shade walks it exactly

struct DeviceCounters {
  unsigned long long rays, box_tests, tri_tests, mismatches, samples, revalidated, exact_walks, primary_rays;
};

// adaptive sampling (k_shade<NEE, true>, b200rt_render_adaptive): the stopping rule of b200rt.h's b200rt_adaptive
struct AdaptArgs {
  float2 *welford;        // per pixel (mean, m2) of the luminance of the samples taken so far; meaningful from sample 2 on
  int *spp_out;           // per pixel: samples taken (k_adaptive_init writes spp for every rendered pixel)
  float *err_out;         // per pixel: standard error of the mean luminance
  int min_spp, check_every;
  float rel_error, floor;
};

struct KernelArgs {
  FrameParams F;
  SceneView S;            // global-memory view (the SMEM variant rebuilds node / triangle pointers)
  cudaTextureObject_t ibl;
  float4 *prim_dirk;      // per pixel: primary direction xyz, hit distance
  int *prim_tri;          // per pixel: primary triangle
  float *out;             // width*height*3: running sums, then the image
  float4 *pA, *pB, *pC;   // path state (below); pC.w: density with which the surface the ray left drew its direction (light sampling only)
  int2 *pHit;
  // opt-in light sampling (k_shade<true>): the emitter triangles, and three more float4 of path state
  const int *light;       // triangles whose material is emissive, ascending (what FileManager.py:235-240 lists)
  int n_light;
  float4 *pS;             // while a light ray is in flight: incoming direction at the surface, its triangle
  float4 *pL;             //   and the weighted contribution that counts if the ray reaches the emitter `w`
  float4 *pR;             // direct light gathered by the current sample
  int *list[2];           // live paths, ping-pong, ALWAYS in the order of the frame's 8x4-pixel tiles; -1 = a path that
                          // left the wavefront since the last compaction (k_shade and k_trace skip such entries)
  int *slots;             // k_primary's / k_shade's output on the iterations that are followed by a compaction
  unsigned int *part_count;  // survivors per contiguous part of `slots` (one part per producer CTA)
  unsigned int *cnt;      // cnt[i] = entries of the list consumed by shade iteration i
  unsigned int *wc;       // wc[i]  = rays of trace iteration i handed out so far
  DeviceCounters *counters;
  int n_nodes, n_tris;    // repacked counts (for staging)
  int stack_depth;        // entries per lane
  int n_work;             // work items (32-pixel tiles x 32)
  int tiles_x;
  int validate;           // 1: hits come from the conservative traversal and must pass validate_hit
  AdaptArgs ad;           // k_shade<NEE, true> and k_adaptive_init only
};

// path state, one entry per pixel:
//   pA = origin.xyz, dir.x     pB = dir.y, dir.z, meta, rng     pC = throughput.rgb, -     pHit = triangle, distance
// origin / dir describe the ray in flight (for a sun ray `dir` keeps the escaped direction for the environment
// lookup and the ray itself points along FrameParams::sun_dir: trace_dir).
// meta: bit 0 first iteration (no ray traced yet), bit 1 light ray (opt-in light sampling), bit 2 camera ray (opt-in
// pixel jitter: the ray leaves cam_pos and the sample has not hit anything yet), bit 3 sun ray, bits 4-7 material type
// of the surface the ray left, bits 8-15 bounce j, bits 16-31 sample index
struct PathMeta {
  int first, light, sun, type, j, s, cam;
};

RT_DEV uint32_t meta_pack(int first, int sun, int type, int j, int s, int light = 0, int cam = 0) {
  return (uint32_t)first | ((uint32_t)light << 1) | ((uint32_t)cam << 2) | ((uint32_t)sun << 3) | ((uint32_t)(type & 15) << 4) | ((uint32_t)(j & 255) << 8) | ((uint32_t)s << 16);
}

RT_DEV PathMeta meta_unpack(uint32_t m) {
  return {(int)(m & 1u), (int)((m >> 1) & 1u), (int)((m >> 3) & 1u), (int)((m >> 4) & 15u), (int)((m >> 8) & 255u), (int)(m >> 16),
          (int)((m >> 2) & 1u)};
}

// direction of the ray a path traces, from its stored direction d
RT_DEV v3 trace_dir(const FrameParams &F, v3 d, int sun) { return sun ? F.sun_dir : d; }

// ---- counters -------------------------------------------------------------------------------------------------------
// the sum of v over the warp, in lane 0 (every lane calls it)
template <class T>
RT_DEV T warp_sum(T v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// adds a warp's sum (warp_sum) to a device counter: one atomic from lane 0, none for 0
template <class T>
RT_DEV void flush(unsigned long long *dst, T warp_total) {
  if ((threadIdx.x & 31u) == 0u && warp_total) atomicAdd(dst, (unsigned long long)warp_total);
}

// part_count[blockIdx.x] = the sum of v over the CTA (every thread calls it)
RT_DEV void cta_count(unsigned int *part_count, unsigned int v) {
  __shared__ unsigned int total;
  if (threadIdx.x == 0) total = 0u;
  __syncthreads();
  v = warp_sum(v);
  if ((threadIdx.x & 31u) == 0u && v) atomicAdd(&total, v);
  __syncthreads();
  if (threadIdx.x == 0) part_count[blockIdx.x] = total;
}

// ---- shared-memory staging of a small scene with the bulk-copy engine (TMA 1-D) ------------------------
RT_DEV uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

RT_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// copies nodes / triangles into shared memory; returns a view that points there
template <bool SMEM>
RT_DEV SceneView stage_scene(const KernelArgs &A, unsigned char *smem, size_t *used) {
  SceneView S = A.S;
  if (!SMEM) {
    *used = 0;
    return S;
  }
  __shared__ __align__(8) uint64_t bar;
  const uint32_t nb = (uint32_t)A.n_nodes * 16u * (uint32_t)A.S.node_f4, tb = (uint32_t)A.n_tris * 48u;
  uint4 *s_nodes = reinterpret_cast<uint4 *>(smem);
  float4 *s_tris = reinterpret_cast<float4 *>(smem + nb);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar)), "r"(nb + tb)
                 : "memory");
    if (nb) bulk_g2s(s_nodes, A.S.nodes, nb, &bar);
    bulk_g2s(s_tris, A.S.ctris, tb, &bar);
    uint32_t done = 0;  // one thread waits for the bytes to land; the block barrier publishes them
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(smem_u32(&bar))
          : "memory");
    }
  }
  __syncthreads();
  S.nodes = s_nodes;
  S.ctris = s_tris;
  *used = (size_t)nb + tb;
  return S;
}

// dynamic shared memory after the staged scene: per-lane traversal stacks, then per-lane parked leaves
__host__ __device__ inline size_t lane_smem_bytes(int stack_depth) {
  return (size_t)kBlock * ((size_t)stack_depth * sizeof(uint32_t) + (size_t)kParkCap * sizeof(uint32_t));
}

RT_DEV int work_to_pixel(const KernelArgs &A, unsigned int w) {
  // 32 consecutive work items = one 8x4 pixel tile; tiles in row-major order
  unsigned int tile = w >> 5, in = w & 31u;
  int tx = (int)(tile % (unsigned)A.tiles_x), ty = (int)(tile / (unsigned)A.tiles_x);
  int x = tx * 8 + (int)(in & 7u), y = ty * 4 + (int)(in >> 3);
  if (x >= A.F.width || y >= A.F.height) return -1;
  if (A.F.tile_row_mod > 1 && ty % A.F.tile_row_mod != A.F.tile_row_rem) return -1;
  int i = y * A.F.width + x;
  if (i < A.F.pixel_begin || i >= A.F.pixel_end) return -1;
  return i;
}

// a pixel's image from the sum of its n samples (Raytracing.cl:211-219)
RT_DEV void write_mean(float *o, v3 sum, float n) {
  o[0] = clamp01(sum.x / n);
  o[1] = clamp01(sum.y / n);
  o[2] = clamp01(sum.z / n);
}

RT_DEV void write_pixel(const KernelArgs &A, int i, v3 sum) {
  float *o = A.out + 3 * (size_t)i;
  if (A.F.out_mode == 1) {
    o[0] = sum.x; o[1] = sum.y; o[2] = sum.z;
  } else {
    write_mean(o, sum, (float)A.F.spp);
  }
}

// ---- adaptive sampling --------------------------------------------------------------------------------------------
// Called after the n-th sample of pixel i (n counted from 1; adaptive frames always cover [0, spp)) with that sample's
// contribution c and the running sum: the Welford update of the mean luminance and the stopping rule, exactly as
// b200rt.h states them (binary32, no contraction).  Returns true when the pixel stops here, before spp; its image,
// sample count and standard error are then written.  A pixel that reaches spp gets its standard error here and its
// image from write_pixel.
RT_DEV bool adaptive_end_sample(const KernelArgs &A, int i, int n, v3 c, v3 sum) {
  const AdaptArgs &ad = A.ad;
  const float y = (0.2126f * c.x + 0.7152f * c.y) + 0.0722f * c.z;
  float2 w = n > 1 ? ad.welford[i] : make_float2(0.0f, 0.0f);
  const float delta = y - w.x;
  w.x = w.x + delta / (float)n;
  w.y = w.y + delta * (y - w.x);
  bool stop = false;
  if (n < A.F.spp) {
    if (n >= ad.min_spp && (n - ad.min_spp) % ad.check_every == 0) {
      const float v = (w.y / (float)(n - 1)) / (float)n;
      const float e = ad.rel_error * fmaxf(fminf(w.x, 1.0f), ad.floor);
      stop = v <= e * e;   // false for a NaN anywhere: such a pixel runs to spp
    }
    if (!stop) {
      ad.welford[i] = w;
      return false;
    }
  }
  ad.err_out[i] = sqrtf((w.y / (float)(n - 1)) / (float)n);
  if (stop) {
    ad.spp_out[i] = n;
    write_mean(A.out + 3 * (size_t)i, sum, (float)n);
  }
  return stop;
}

// spp / 0 into the sample-count / standard-error maps for every pixel of the rendered set, before k_primary (ray-free
// pixels keep these; k_shade overwrites them for the others)
__global__ void k_adaptive_init(const __grid_constant__ KernelArgs A) {
  for (unsigned int w = blockIdx.x * blockDim.x + threadIdx.x; w < (unsigned)A.n_work; w += gridDim.x * blockDim.x) {
    const int i = work_to_pixel(A, w);
    if (i >= 0) {
      A.ad.spp_out[i] = A.F.spp;
      A.ad.err_out[i] = 0.0f;
    }
  }
}

// ---- jittered frames: the first path list without a primary-hit kernel -------------------------------------------
// Every pixel of the rendered set starts its first sample (s0) with a camera ray of its own in k_shade<NEE, false,
// true>, so no pixel is ray-free: pB (first iteration, s0, generator word i as Raytracing.cl:171 seeds it), a zero
// running sum, and the pixel into slots for k_count_parts + k_compact (-1 outside the rendered set).
__global__ void k_jitter_init(const __grid_constant__ KernelArgs A) {
  for (unsigned int w = blockIdx.x * blockDim.x + threadIdx.x; w < (unsigned)A.n_work; w += gridDim.x * blockDim.x) {
    const int i = work_to_pixel(A, w);
    if (i >= 0) {
      A.pB[i] = make_float4(0.0f, 0.0f, __uint_as_float(meta_pack(1, 0, 0, 0, A.F.s0)), __uint_as_float((uint32_t)i));
      float *acc_px = A.out + 3 * (size_t)i;
      acc_px[0] = 0.0f; acc_px[1] = 0.0f; acc_px[2] = 0.0f;
    }
    A.slots[w] = i;
  }
}

// ---- primary hits ---------------------------------------------------------------------------------------
// PARITY: write tri / k for every pixel of [pixel_begin,pixel_end) and nothing else.
template <int TRAV, bool SMEM, bool PARITY, bool STATS>
__global__ void __launch_bounds__(kBlock) k_primary(const __grid_constant__ KernelArgs A, int *tri_out, float *k_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  size_t used;
  SceneView S = stage_scene<SMEM>(A, smem, &used);
  LaneStack st;
  st.base = reinterpret_cast<uint32_t *>(smem + used) + threadIdx.x;
  st.stride = kBlock;
  uint32_t *parks = reinterpret_cast<uint32_t *>(smem + used + (size_t)kBlock * A.stack_depth * sizeof(uint32_t)) + threadIdx.x;
  TraceCounters tc;
  tc.box_tests = 0; tc.tri_tests = 0;
  unsigned int mism = 0;
  unsigned long long rays = 0;
  const unsigned int n_work = (unsigned)A.n_work;  // a multiple of 32: whole warps leave the loop together
  for (unsigned int w = blockIdx.x * kBlock + threadIdx.x; w < n_work; w += gridDim.x * kBlock) {
    const int i = work_to_pixel(A, w);
    bool live = false;  // the pixel's samples need rays: it joins the first path list
    if (i >= 0) {
      v3 d = camera_dir(A.F, i);
      Hit h = closest_hit<TRAV, SMEM, STATS>(S, A.F.cam_pos, d, st, parks, kBlock, &tc, &mism);
      rays++;
      if (PARITY) {
        tri_out[i] = h.tri;
        k_out[i] = h.k;
      } else {
        int mat_type = -1;
        float emit = 0.0f;
        if (h.tri >= 0) {
          Material m = load_material(S.mats, tri_material(S, h.tri));
          mat_type = m.type;
          emit = m.roughness;
        }
        if (h.tri >= 0 && mat_type != 0) {
          live = true;
          A.prim_dirk[i] = make_float4(d.x, d.y, d.z, h.k);
          A.prim_tri[i] = h.tri;
          // Raytracing.cl:171 (imgSize receives imgDim, so seed0 = i); the running sum lives in the output buffer
          A.pB[i] = make_float4(0.0f, 0.0f, __uint_as_float(meta_pack(1, 0, 0, 0, A.F.s0)), __uint_as_float((uint32_t)i));
          float *acc_px = A.out + 3 * (size_t)i;
          acc_px[0] = 0.0f; acc_px[1] = 0.0f; acc_px[2] = 0.0f;
        } else {
          // every sample of this pixel is the same ray-free value: Raytracing.cl:146-150 (miss) / :140-144 (emitter)
          v3 c;
          if (h.tri < 0) {
            c = (mk3(1.0f, 1.0f, 1.0f) * ibl_lookup(A.F, A.ibl, d)) * A.F.ibl_power;
          } else {
            c = mk3(1.0f, 1.0f, 1.0f) * emit;
          }
          v3 sum = mk3(0.0f, 0.0f, 0.0f);
          for (int s = A.F.s0; s < A.F.s1; ++s) sum = sum + c;  // the reference accumulates sample by sample
          write_pixel(A, i, sum);
        }
      }
    }
    if (!PARITY) A.slots[w] = live ? i : -1;   // work items are in tile order; k_count_parts + k_compact make the first list
  }
  rays = warp_sum(rays);
  flush(&A.counters->rays, rays);
  flush(&A.counters->primary_rays, rays);
  flush(&A.counters->mismatches, warp_sum(mism));
  if (STATS) {
    flush(&A.counters->box_tests, warp_sum(tc.box_tests));
    flush(&A.counters->tri_tests, warp_sum(tc.tri_tests));
  }
}

// ---- order-preserving list compaction -------------------------------------------------------------------------------
// entries per producer CTA: the same function on both sides of the hand-over (a multiple of the block size, so that
// warps read whole 128-byte lines)
RT_HD unsigned int part_size(unsigned int n, unsigned int parts) {
  const unsigned int per = (n + parts - 1u) / parts;
  return (per + 127u) & ~127u;
}

constexpr int kCompactBlock = 128;

// survivors per part of `slots` when the producer did not count them itself (k_primary's strided loop)
__global__ void __launch_bounds__(kCompactBlock) k_count_parts(const int *__restrict__ slots, unsigned int n,
                                                                unsigned int *__restrict__ part_count) {
  const unsigned int part = part_size(n, gridDim.x);
  const unsigned int end = min(n, (blockIdx.x + 1u) * part);
  unsigned int c = 0;
  for (unsigned int t = blockIdx.x * part + threadIdx.x; t < end; t += kCompactBlock) c += slots[t] >= 0 ? 1u : 0u;
  cta_count(part_count, c);
}

// list_out = the non-negative entries of slots[0 .. n), order kept; *n_out = their number.  One CTA per part (same
// grid as the producer); its base is the sum of the earlier parts' counts.  n is read from n_src when given.
__global__ void __launch_bounds__(kCompactBlock) k_compact(const int *__restrict__ slots, const unsigned int *n_src, unsigned int n_value,
                                                            const unsigned int *__restrict__ part_count, int *__restrict__ list_out,
                                                            unsigned int *__restrict__ n_out) {
  const unsigned int n = n_src ? *n_src : n_value;
  const unsigned int part = part_size(n, gridDim.x);
  __shared__ unsigned int s_base, s_warp[kCompactBlock / 32];
  const unsigned int lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  // sum of the earlier parts (and, in the last CTA, of all parts: the length of the new list)
  unsigned int before = 0, all = 0;
  for (unsigned int p = threadIdx.x; p < gridDim.x; p += kCompactBlock) {
    const unsigned int c = part_count[p];
    all += c;
    if (p < blockIdx.x) before += c;
  }
  if (threadIdx.x == 0) s_base = 0u;
  if (threadIdx.x < kCompactBlock / 32) s_warp[threadIdx.x] = 0u;
  __syncthreads();
  before = warp_sum(before);
  all = warp_sum(all);
  if (lane == 0) {
    if (before) atomicAdd(&s_base, before);
    if (all) atomicAdd(&s_warp[0], all);
  }
  __syncthreads();
  unsigned int base = s_base;
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *n_out = s_warp[0];
  __syncthreads();
  const unsigned int end = min(n, (blockIdx.x + 1u) * part);
  for (unsigned int t0 = blockIdx.x * part; t0 < end; t0 += kCompactBlock) {
    const unsigned int t = t0 + threadIdx.x;
    const int v = t < end ? slots[t] : -1;
    const unsigned int m = __ballot_sync(0xffffffffu, v >= 0);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    unsigned int off = base;
    for (unsigned int w = 0; w < warp; ++w) off += s_warp[w];
    if (v >= 0) list_out[off + __popc(m & ((1u << lane) - 1u))] = v;
    unsigned int step = 0;
    for (unsigned int w = 0; w < kCompactBlock / 32; ++w) step += s_warp[w];
    base += step;
    __syncthreads();
  }
}

// ---- opt-in smooth shading (b200rt_opts.sampling bit B200RT_SAMPLING_SMOOTH_NORMALS) ---------------------------------
// The shading normal of a hit on triangle `tri` at point x, by the rule b200rt.h states: n0 (the normals record) for a
// flat triangle, else the normalised barycentric interpolation of n0, n1, n2, or n0 when that is not a usable direction.  The
// normals buffer holds n_tris first-vertex normals, then 2 float4 per triangle: (n1.xyz, flat / curved flag), (n2.xyz, -)
// (scene_repack.h).  *curved: the triangle is not flat, so its precomputed frame does not apply and tri_frame_at builds
// one.
// The barycentrics (b0, b1, b2) of point x on triangle `tri` by the rule b200rt.h states for smooth shading, which
// albedo textures share.
RT_DEV v3 barycentrics(const SceneView &S, int tri, v3 x) {
  const Tri t = load_tri(S.tris, tri);
  const v3 p = x - t.A;
  const float d00 = dot(t.e1, t.e1), d01 = dot(t.e1, t.e2), d11 = dot(t.e2, t.e2);
  const float d20 = dot(p, t.e1), d21 = dot(p, t.e2);
  const float den = d00 * d11 - d01 * d01;
  const float b1 = (d11 * d20 - d01 * d21) / den;
  const float b2 = (d00 * d21 - d01 * d20) / den;
  const float b0 = (1.0f - b1) - b2;
  return mk3(b0, b1, b2);
}

template <bool SMOOTH>
RT_DEV v3 shading_normal(const SceneView &S, int n_tris, int tri, v3 n0, v3 x, bool *curved) {
  *curved = false;
  if (!SMOOTH) return n0;
  const float4 *nsmooth = S.normals + n_tris;
  const float4 c1 = __ldg(nsmooth + 2 * (size_t)tri);
  if (!(c1.w > 0.0f)) return n0;   // flat (scene_repack.h kSmoothFlat; kSmoothBadIndex never reaches a render)
  *curved = true;
  const float4 c2 = __ldg(nsmooth + 2 * (size_t)tri + 1);
  const v3 b = barycentrics(S, tri, x);
  const v3 n = unit(((n0 * b.x) + (mk3(c1.x, c1.y, c1.z) * b.y)) + (mk3(c2.x, c2.y, c2.z) * b.z));
  if (!isfinite(n.x) || !isfinite(n.y) || !isfinite(n.z) || !(dot(n, n) > 0.0f)) return n0;
  return n;
}

// ---- opt-in albedo textures (b200rt_opts.sampling bit B200RT_SAMPLING_TEXTURES) -----------------------------------------
// The albedo of a type-1 or type-2 hit on triangle `tri` (material `mat`, colour `color`) at point x, by the rule b200rt.h
// states: color times the texture factor at the interpolated UV, or color itself when the material has no texture.  The
// normals buffer holds, after the smooth-shading records, 2 float4 of UVs per triangle, (u0, v0, u1, v1), (u2, v2, -, -),
// and then one texture header (b200rt_api.cu write_tex_header): the address of the texture buffer (low, high word), the
// materials it covers, the textures it holds.  That buffer holds an int4 per texture (first texel, w, h, -), an int32 per
// material (its texture or -1, padded to a multiple of 4), then the texels.  Kept out of KernelArgs, so that no existing
// kernel's parameters move.
RT_DEV v3 surface_albedo(const SceneView &S, int n_tris, int tri, int mat, v3 color, v3 x) {
  const float4 *uv = S.normals + 3 * (size_t)n_tris;
  const uint4 hd = __ldg(reinterpret_cast<const uint4 *>(uv + 2 * (size_t)n_tris));
  if ((unsigned)mat >= hd.z) return color;
  TexView T;
  T.info = reinterpret_cast<const int4 *>(((unsigned long long)hd.y << 32) | hd.x);
  const int *mat_tex = reinterpret_cast<const int *>(T.info + hd.w);
  const int tex = __ldg(mat_tex + mat);
  if (tex < 0) return color;
  T.texels = reinterpret_cast<const uchar4 *>(mat_tex + ((hd.z + 3u) & ~3u));
  const float4 q0 = __ldg(uv + 2 * (size_t)tri), q1 = __ldg(uv + 2 * (size_t)tri + 1);
  const v3 b = barycentrics(S, tri, x);
  const float u = (q0.x * b.x + q0.z * b.y) + q1.x * b.z;
  const float v = (q0.y * b.x + q0.w * b.y) + q1.y * b.z;
  return color * texture_factor(T, tex, u, v);
}

// ---- shading ----------------------------------------------------------------------------------------------------
// The per-path state machine is written as a sequence of phases with the warp re-converged between them, so that
// e.g. the direction sampling runs once per warp for every lane that needs it, whichever way the lane got there
// (bounce hit, or sample ended and the next one starts from the cached primary hit).
// 8 CTAs per SM: the kernel is bound by the latency of its gathers; 5-7 (no spills) and 9-12 resident CTAs were all slower.
// NEE = opt-in light sampling (b200rt_opts.sampling bit 1): a separate instantiation, so that the reference's
// estimator runs exactly the code it ran before.  ADAPT = adaptive sampling (adaptive_end_sample at the end of every
// sample), likewise a separate instantiation.  JITTER = opt-in pixel jitter (sampling bit B200RT_SAMPLING_PIXEL_JITTER):
// a sample starts with a camera ray through a jittered point of its pixel (phase 3), which phase 2 resolves the way
// k_primary resolves the cached primary ray, instead of from the cached primary hit.  SMOOTH = opt-in smooth shading
// (B200RT_SAMPLING_SMOOTH_NORMALS): a hit on a curved triangle is shaded with the interpolated normal and a frame built
// in registers (shading_normal, tri_frame_at); a flat one keeps its precomputed frame.  GLASS = opt-in refractive glass
// (B200RT_SAMPLING_DIELECTRIC_GLASS): a glass hit whose ior slot is not 1 reflects or refracts (scatter_dielectric)
// instead of passing through.  TEX = opt-in albedo textures (B200RT_SAMPLING_TEXTURES): a diffuse or glossy surface
// whose material has a texture takes surface_albedo for its colour in the light sample (phase 3b) and the scatter (4).
// ROUGH = opt-in rough glass (B200RT_SAMPLING_ROUGH_GLASS, only with GLASS): a glass hit whose ior slot is not 1 and
// whose roughness is > 0 scatters off a GGX microfacet (scatter_rough_dielectric) and weighs the throughput by G1.
template <bool NEE, bool ADAPT, bool JITTER = false, bool SMOOTH = false, bool GLASS = false, bool TEX = false,
          bool ROUGH = false>
__global__ void __launch_bounds__(kShadeBlock, 8) k_shade(const __grid_constant__ KernelArgs A, int iter) {
  const FrameParams &F = A.F;
  const SceneView &S = A.S;
  const unsigned int n_in = A.cnt[iter];
  const int *list_in = A.list[iter & 1];
  const unsigned int lane = threadIdx.x & 31u;
  unsigned long long samples = 0;
  unsigned int reval = 0, exact = 0, survivors = 0;
  // Every CTA shades one contiguous part of the list and leaves, entry for entry, the path or -1 in the next list;
  // every kCompactEvery iterations k_compact closes the gaps without changing the order (paths leave the wavefront
  // only when their pixel is finished, so gaps accumulate slowly).  The list therefore stays sorted by tile for the whole
  // frame: the 32 paths of a warp — here and in k_trace — belong to neighbouring pixels, so the rays that restart
  // from the cached primary hits leave from neighbouring points.  (An atomically appended list is a random
  // permutation of the pixels after a few hundred iterations; on the 5 M-triangle scene that cost a third of the
  // traversal speed.)
  const bool compacting = ((iter + 1) % kCompactEvery) == 0;
  int *out = compacting ? A.slots : A.list[(iter + 1) & 1];
  const unsigned int part = part_size(n_in, gridDim.x);
  const unsigned int part_end = min(n_in, (blockIdx.x + 1u) * part);
  for (unsigned int tb = blockIdx.x * part + (threadIdx.x & ~31u); tb < part_end; tb += kShadeBlock) {
    const unsigned int t = tb + lane;
    const bool in_part = t < part_end;
    // ---- phase 0: load -------------------------------------------------------------------------------------------
    int pix = in_part ? ld_stream(list_in + t) : -1;
    const bool valid = pix >= 0;   // -1: past the part's end, or a path that left the wavefront since the last compaction
    if (!valid) pix = 0;
    uint32_t meta = 1u;
    rng_state g;
    g.a = 0u;
    v3 o = mk3(0.0f, 0.0f, 0.0f), d = mk3(0.0f, 0.0f, 1.0f), acc = mk3(1.0f, 1.0f, 1.0f);
    float hk = 0.0f, pb_ray = 0.0f;
    int htri = -1;
    if (valid) {
      // all four at once: they depend on pix only (on a path's first iteration pA / pC / pHit hold nothing yet and
      // are not looked at), and this kernel is bound by the latency of its chains of dependent loads
      const float4 sb = ld_stream(A.pB + pix), sa = ld_stream(A.pA + pix), sc = ld_stream(A.pC + pix);
      const int2 hh = ld_stream(A.pHit + pix);
      meta = __float_as_uint(sb.z);
      g.a = __float_as_uint(sb.w);
      if (!(meta & 1u)) {
        o = mk3(sa.x, sa.y, sa.z);
        d = mk3(sa.w, sb.x, sb.y);
        acc = mk3(sc.x, sc.y, sc.z);
        if (NEE) pb_ray = sc.w;
        htri = hh.x;
        hk = __int_as_float(hh.y);
      }
    }
    const PathMeta pm = meta_unpack(meta);
    const bool first = pm.first != 0;
    int sun_ray = pm.sun, seg_type = pm.type, j = pm.j, s = pm.s;
    const bool light_ray = NEE && pm.light != 0;
    const bool cam_ray = JITTER && pm.cam != 0;
    bool pixel_done = false, start = valid && first, shade = false, end_sample = false, sun_done = false;
    bool want_light = false, light_done = false, from_light = false, cam_out = false;

    // ---- phase 1: the winner of the conservative walk must pass the exact leaf-box test ---------------------------------
    if (valid && !first && A.validate && htri != -1) {
      const v3 dray = trace_dir(F, d, sun_ray);   // a light ray's direction sits in d
      if (htri == kHitNeedsExactWalk ||
          !validate_winner(S, o, dray, htri, tri_rank(S, htri))) {  // out-of-range or grazing ray: re-trace exactly
        const Hit h = closest_hit_nodrop(S, o, dray);
        if (htri != kHitNeedsExactWalk) ++reval; else ++exact;
        htri = h.tri;
        hk = h.k;
      }
    }
    __syncwarp();

    // ---- phase 2: resolve the traced ray (Raytracing.cl:91-137) ------------------------------------------------------------
    if (valid && !first) {
      if (cam_ray) {  // the sample's camera ray, as k_primary resolves the primary ray
        if (htri < 0) {  // :146-150
          acc = (mk3(1.0f, 1.0f, 1.0f) * ibl_lookup(F, A.ibl, d)) * F.ibl_power;
          end_sample = true;
        } else {
          const Material mc = load_material(S.mats, tri_material(S, htri));
          if (mc.type == 0) {  // :140-144
            acc = mk3(1.0f, 1.0f, 1.0f) * mc.roughness;
            end_sample = true;
          } else {  // the hit starts the path, as the cached primary hit does in phase 3
            j = 0;
            if (NEE && mc.type != 3) want_light = true; else shade = true;
          }
        }
      } else if (light_ray) {
        light_done = true;
      } else if (!sun_ray) {
        if (htri >= 0) {  // the bounce ray becomes the current segment (:91-93)
          const Material mb = load_material(S.mats, tri_material(S, htri));
          if (mb.type != 0) {
            if (j == F.max_bounce) {  // :99-103
              acc = mk3(0.0f, 0.0f, 0.0f);
              end_sample = true;
            } else {
              ++j;
              if (NEE && mb.type != 3) want_light = true; else shade = true;
            }
          } else {  // :105-109
            acc = acc * mb.roughness;
            if (NEE && seg_type != 3) {
              // the light sample at the surface this ray left could have made the same connection: balance heuristic
              const Tri t = load_tri(S.tris, htri);
              const float pl = light_pdf(t.e1, t.e2, A.n_light, unit(d), (hk * hk) * dot(d, d));
              const float den = pb_ray + pl;
              acc = acc * (den > 0.0f ? pb_ray / den : 0.0f);
            }
            end_sample = true;
          }
        } else {  // escaped: shadow ray towards the sun from the same origin (:115-124); d keeps the escaped direction
          sun_ray = 1;
        }
      } else {
        sun_done = true;
      }
    }
    __syncwarp();
    if (sun_done) {  // sun ray finished, :125-137
      v3 sun = mk3(0.0f, 0.0f, 0.0f);
      if (htri < 0) {
        if (seg_type != 3) sun = mk3(F.sun_power, F.sun_power, F.sun_power);
      } else {
        const Material ms = load_material(S.mats, tri_material(S, htri));
        if (ms.type == 3) sun = ms.color * F.sun_power;
      }
      v3 envl;
      if (F.ibl_power == 0.0f) {
        // texel/255 is a finite value >= 0, so texel/255 * 0 is a zero of ibl_power's sign whatever the texel
        envl = mk3(0.5f * F.ibl_power, 0.5f * F.ibl_power, 0.5f * F.ibl_power);
      } else {
        envl = ibl_lookup(F, A.ibl, d) * F.ibl_power;
      }
      acc = acc * (sun + envl);
      end_sample = true;
    }
    __syncwarp();
    if (NEE && light_done) {  // the light ray is back: its contribution counts iff it reached the emitter it aimed at
      const float4 pl = A.pL[pix], ps = A.pS[pix];
      if (htri == __float_as_int(pl.w)) {
        float4 r = A.pR[pix];
        r.x += pl.x; r.y += pl.y; r.z += pl.z;
        A.pR[pix] = r;
      }
      d = mk3(ps.x, ps.y, ps.z);     // back at the surface: o is the light ray's origin, the surface point
      htri = __float_as_int(ps.w);
      hk = 0.0f;
      from_light = true;
      shade = true;
    }
    if (end_sample) {
      float *acc_px = A.out + 3 * (size_t)pix;
      v3 sum = mk3(ld_stream(acc_px), ld_stream(acc_px + 1), ld_stream(acc_px + 2));
      if (NEE) {
        const float4 r = A.pR[pix];
        acc = mk3(r.x, r.y, r.z) + acc;   // direct light gathered along the path + what the path ended on
      }
      sum = sum + acc;  // :207
      ++s;
      ++samples;
      bool finished = s >= F.s1;
      if (ADAPT) finished = adaptive_end_sample(A, pix, s, acc, sum) || finished;
      if (finished) {
        if (!ADAPT || s >= F.s1) write_pixel(A, pix, sum);
        pixel_done = true;
      } else {
        acc_px[0] = sum.x; acc_px[1] = sum.y; acc_px[2] = sum.z;
        start = true;
      }
    }
    // ---- phase 3: a new sample starts from the cached primary hit (Raytracing.cl:195-201), or with a jittered camera ray -------
    if (JITTER && start) {
      float ux, uy;
      if (F.rng_mode == 0) draw2_jitter<0>(g, (uint32_t)pix, (uint32_t)s, F.key0, F.key1, &ux, &uy);
      else draw2_jitter<1>(g, (uint32_t)pix, (uint32_t)s, F.key0, F.key1, &ux, &uy);
      o = F.cam_pos;
      d = camera_dir_jittered(F, pix, ux, uy);
      acc = mk3(1.0f, 1.0f, 1.0f);
      j = 0;
      sun_ray = 0;
      if (NEE) A.pR[pix] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      cam_out = true;
    } else if (start) {
      const float4 dk = ld_stream(A.prim_dirk + pix);
      o = F.cam_pos;
      d = mk3(dk.x, dk.y, dk.z);
      hk = dk.w;
      htri = ld_stream(A.prim_tri + pix);
      acc = mk3(1.0f, 1.0f, 1.0f);
      j = 0;
      if (NEE) {
        A.pR[pix] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if ((int)__ldg(S.mats + 6 * tri_material(S, htri)) != 3) want_light = true; else shade = true;
      } else {
        shade = true;
      }
    }
    __syncwarp();

    // ---- phase 3b (light sampling only): one emitter point seen from the surface, and the shadow ray towards it --------------
    if (NEE && want_light) {
      const float4 nn = __ldg(S.normals + htri);
      v3 n = mk3(nn.x, nn.y, nn.z);
      Material m = load_material(S.mats, tri_material(S, htri));
      v3 un = unit(n);
      float ul, ua, ub;
      if (F.rng_mode == 0) draw3<0>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, 1u, F.key0, F.key1, &ul, &ua, &ub);
      else draw3<1>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, 1u, F.key0, F.key1, &ul, &ua, &ub);
      int idx = (int)(ul * (float)A.n_light);
      if (idx > A.n_light - 1) idx = A.n_light - 1;
      const int lt = __ldg(A.light + idx);
      const Tri l = load_tri(S.tris, lt);
      const Material ml = load_material(S.mats, l.mat);
      const float Le = ml.type == 0 ? ml.roughness : 0.0f;
      const v3 x = o + unit(d) * hk;
      if (SMOOTH) {
        bool curved;
        n = shading_normal<true>(S, A.n_tris, htri, n, x, &curved);
        un = unit(n);
      }
      if (TEX) m.color = surface_albedo(S, A.n_tris, htri, tri_material(S, htri), m.color, x);
      v3 w;
      const v3 direct = sample_light(m, F.sampling, n, un, x, d, acc, l.A, l.e1, l.e2, Le, A.n_light, ua, ub, &w);
      A.pS[pix] = make_float4(d.x, d.y, d.z, __int_as_float(htri));
      A.pL[pix] = make_float4(direct.x, direct.y, direct.z, __int_as_float(lt));
      o = x;
      d = w;
      sun_ray = 0;
    }
    __syncwarp();

    // ---- phase 4: next direction, BRDF * cos / pdf (:51-87); segment = (o, d, hk, htri) ------------------------------------------
    if (shade) {
      const float4 nn = __ldg(S.normals + htri);
      bool curved;   // the surface point: o itself when the light ray is back at it (phase 3b moved o there)
      const v3 n = shading_normal<SMOOTH>(S, A.n_tris, htri, mk3(nn.x, nn.y, nn.z), (NEE && from_light) ? o : o + unit(d) * hk, &curved);
      Material m = load_material(S.mats, tri_material(S, htri));
      if (TEX && (m.type == 1 || m.type == 2))
        m.color = surface_albedo(S, A.n_tris, htri, tri_material(S, htri), m.color, (NEE && from_light) ? o : o + unit(d) * hk);
      const int which = m.type == 3 ? 0 : (m.type == 1 ? 1 : 2);
      const TriFrame tf = curved ? tri_frame_at(n, which) : load_tri_frame(S.frames, htri, which);
      v3 nd, brdf;
      float inv_pdf;
      bool dielectric = false, reflected = false;
      float wt = 1.0f;   // rough glass: G1 of the microfacet scatter, 0 for a direction on the wrong side
      if (m.type == 3) {
        const float v = GLASS ? load_material_ior(S.mats, tri_material(S, htri)) : 1.0f;
        if (v == 1.0f) {  // the reference's pass-through (always without GLASS)
          nd = d;
          brdf = m.color;
          inv_pdf = 1.0f / fabsf(dot(nd, tf.un));
        } else if (ROUGH && m.roughness > 0.0f) {
          float uf, u1, u2;
          if (F.rng_mode == 0) draw3<0>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, 0u, F.key0, F.key1, &uf, &u1, &u2);
          else draw3<1>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, 0u, F.key0, F.key1, &uf, &u1, &u2);
          nd = scatter_rough_dielectric(d, tf.un, v == 0.0f ? kGlassDefaultIor : v, m.roughness, uf, u1, u2, &reflected,
                                        &wt);
          dielectric = true;
        } else {
          float u;
          if (F.rng_mode == 0) u = draw1<0>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1);
          else u = draw1<1>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1);
          nd = scatter_dielectric(d, tf.un, v == 0.0f ? kGlassDefaultIor : v, u, &reflected);
          dielectric = true;
        }
      } else {
        float u0, u1;
        if (F.rng_mode == 0) draw2<0>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1, &u0, &u1);
        else draw2<1>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1, &u0, &u1);
        if (m.type == 1) {
          nd = sample_cosine(n, tf, u0, u1, &inv_pdf);
          brdf = m.color * (1.0f / 3.14f);
        } else {
          if (F.sampling & 1) nd = sample_glossy_importance(m.roughness, tf.un, d, u0, u1, &inv_pdf);
          else nd = sample_uniform(n, tf, u0, u1, &inv_pdf);
          brdf = bsdf_ggx(m, neg3(d), nd, n);
        }
      }
      if (NEE) pb_ray = m.type == 3 ? 0.0f : bsdf_pdf(m, F.sampling, tf.un, d, unit(nd));
      if (!NEE || !from_light) o = o + unit(d) * hk;  // :79 — no offset along the normal
      d = nd;
      if (GLASS && dielectric) {  // reflection keeps the throughput, refraction tints it; rough glass then weighs by G1
        if (!reflected) acc = acc * m.color;
        if (ROUGH) acc = wt == 0.0f ? mk3(0.0f, 0.0f, 0.0f) : acc * wt;
      } else {
        const float att = inv_pdf * fabsf(dot(nd, tf.un));
        acc = (acc * brdf) * att;
      }
      seg_type = m.type;
      sun_ray = 0;
    }
    __syncwarp();

    // ---- phase 5: store, join the next list -----------------------------------------------------------------------------------------
    const bool alive = valid && !pixel_done;
    if (alive) {
      A.pA[pix] = make_float4(o.x, o.y, o.z, d.x);
      A.pB[pix] = make_float4(d.y, d.z, __uint_as_float(meta_pack(0, sun_ray, seg_type, j, s, (NEE && want_light) ? 1 : 0,
                                                                  (JITTER && cam_out) ? 1 : 0)),
                              __uint_as_float(g.a));
      A.pC[pix] = make_float4(acc.x, acc.y, acc.z, NEE ? pb_ray : 0.0f);
    }
    if (in_part) out[t] = alive ? pix : -1;
    survivors += alive ? 1u : 0u;
  }
  if (!compacting) {  // the next list has this one's length
    if (blockIdx.x == 0 && threadIdx.x == 0) A.cnt[iter + 1] = n_in;
  } else {  // survivors of this CTA's part, for k_compact
    cta_count(A.part_count, survivors);
  }
  flush(&A.counters->samples, warp_sum(samples));
  flush(&A.counters->revalidated, warp_sum(reval));
  flush(&A.counters->exact_walks, warp_sum(exact));
}

// per-triangle sampling frames, once per scene upload
__global__ void k_tri_frames(const float4 *__restrict__ normals, int n_tris, float4 *__restrict__ frames) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris) return;
  const float4 nn = normals[t];
  float4 f[kFrameVec];
  make_tri_frame(mk3(nn.x, nn.y, nn.z), f);
  for (int k = 0; k < kFrameVec; ++k) frames[(size_t)kFrameVec * t + k] = f[k];
}

// ---- tracing ------------------------------------------------------------------------------------------------------
template <int TRAV, bool SMEM, bool STATS>
__global__ void __launch_bounds__(kBlock) k_trace(const __grid_constant__ KernelArgs A, int iter) {
  extern __shared__ __align__(16) unsigned char smem[];
  const unsigned int n = A.cnt[iter + 1];
  if (n == 0u) return;
  size_t used;
  const SceneView S = stage_scene<SMEM>(A, smem, &used);
  LaneStack st;
  st.base = reinterpret_cast<uint32_t *>(smem + used) + threadIdx.x;
  st.stride = kBlock;
  uint32_t *parks = reinterpret_cast<uint32_t *>(smem + used + (size_t)kBlock * A.stack_depth * sizeof(uint32_t)) + threadIdx.x;
  const int *list = A.list[(iter + 1) & 1];
  unsigned int *wc = A.wc + iter;
  const unsigned int lane = threadIdx.x & 31u;
  const unsigned int lt_mask = (1u << lane) - 1u;

  Trav T;
  T.best.tri = -1; T.best.k = 1000.0f; T.best_rank = 0x7fffffff; T.lim = 0.0f; T.cur = -1; T.sp = 0;
  T.o = mk3(0, 0, 0); T.d = mk3(1, 1, 1);
  T.Q.A = mk3(1, 1, 1); T.Q.Bn = mk3(0, 0, 0); T.Q.Bf = mk3(0, 0, 0);
  for (int a = 0; a < 3; ++a) { T.Q.sn[a] = kSelMin; T.Q.sf[a] = kSelMax; }
  int pn = 0;         // parked leaves of this lane
  int path = -1;      // path whose ray this lane is tracing
  unsigned int c_next = 0, c_end = 0;  // the warp's claimed chunk of the list (uniform)
  bool exhausted = false;

  unsigned int rays = 0;   // of this lane: far below 2^32
  unsigned int mism = 0;
  TraceCounters tc;
  tc.box_tests = 0; tc.tri_tests = 0;

  int thresh = kQuorum;  // the node phase runs while at least this many lanes can step
  for (;;) {
    // ---- node phase: one node per lane per turn -----------------------------------------------------------------------------
    for (;;) {
      const bool can = trav_active(T) && pn <= kParkCap - 2;
      if (__popc(__ballot_sync(0xffffffffu, can)) < thresh) break;
      if (can) trav_step<SMEM, STATS>(S, T, pn, parks, kBlock, st, &tc);
    }
    // ---- leaf phase: every lane that holds a parked leaf tests its most recent; again while many lanes hold one -------------
    for (unsigned int pm = __ballot_sync(0xffffffffu, pn > 0); pm != 0u;) {
      if (pn > 0) {
        --pn;
        if (STATS) tc.tri_tests++;
        test_parked<SMEM>(S, T, parks[pn * kBlock], T.o, T.d);
      }
      pm = __ballot_sync(0xffffffffu, pn > 0);
      if (__popc(pm) < kTriQuorum) break;
    }
    // ---- finished rays are handed back; idle lanes pull the next rays together ---------------------------------------------------
    const bool finished = (path >= 0) && !trav_active(T) && pn == 0;
    if (finished) {
      A.pHit[path] = make_int2(T.best.tri, __float_as_int(T.best.k));
      path = -1;
    }
    const unsigned int idle = __ballot_sync(0xffffffffu, path < 0);
    if (exhausted) {
      if (idle == 0xffffffffu) break;
      continue;
    }
    const int n_idle = __popc(idle);
    if (n_idle == 0) continue;
    if (n_idle < kRefillMin &&
        __popc(__ballot_sync(0xffffffffu, trav_active(T) && pn <= kParkCap - 2)) >= kQuorum)
      continue;  // enough lanes can still step: let more finish before paying for a refill
    {
      int need = n_idle;
      int rank = __popc(idle & lt_mask);
      bool want = path < 0;
      while (need > 0) {
        if (c_next == c_end) {
          unsigned int b = 0;
          if (lane == 0) b = atomicAdd(wc, kChunk);
          b = __shfl_sync(0xffffffffu, b, 0);
          if (b >= n) { exhausted = true; thresh = 1; break; }
          c_next = b;
          c_end = min(b + kChunk, n);
        }
        const int take = min(need, (int)(c_end - c_next));
        if (want && rank < take) {
          want = false;
          path = ld_stream(list + c_next + rank);
          if (path >= 0) {   // -1: the path left the wavefront since the last compaction; the lane waits for the next refill
            const float4 sa = ld_stream(A.pA + path), sb = ld_stream(A.pB + path);
            const v3 o = mk3(sa.x, sa.y, sa.z);
            const v3 d = trace_dir(A.F, mk3(sa.w, sb.x, sb.y), meta_unpack(__float_as_uint(sb.z)).sun);
            rays++;
            if (TRAV == 0) {
              if (ray_is_fast(S, o)) {
                trav_begin<SMEM, STATS>(S, T, o, d, pn, parks, &tc);
              } else {
                // the margins of the conservative test are not proven for this origin / scene (|coordinate| > 2^40):
                // k_shade's validation phase walks the ray exactly (closest_hit_nodrop), which keeps that walk's
                // registers and local stack out of this kernel
                T.best.tri = kHitNeedsExactWalk;
                T.best.k = 1000.0f;
                T.cur = -1;
              }
            } else {  // reference / verify traversal: whole walk at once
              T.best = closest_hit<TRAV, SMEM, STATS>(S, o, d, st, parks, kBlock, &tc, &mism);
              T.cur = -1;
            }
          }
        }
        rank -= take;
        c_next += take;
        need -= take;
      }
    }
  }

  flush(&A.counters->rays, warp_sum(rays));
  flush(&A.counters->mismatches, warp_sum(mism));
  if (STATS) {
    flush(&A.counters->box_tests, warp_sum(tc.box_tests));
    flush(&A.counters->tri_tests, warp_sum(tc.tri_tests));
  }
}

// ---- closest hit of caller-supplied rays (traversal on its own) ---------------------------------------------------------
template <int TRAV, bool SMEM, bool STATS>
__global__ void __launch_bounds__(kBlock) k_trace_rays(const __grid_constant__ KernelArgs A, const float *rays, long long n,
                                                       int *tri_out, float *k_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  size_t used;
  SceneView S = stage_scene<SMEM>(A, smem, &used);
  LaneStack st;
  st.base = reinterpret_cast<uint32_t *>(smem + used) + threadIdx.x;
  st.stride = kBlock;
  uint32_t *parks = reinterpret_cast<uint32_t *>(smem + used + (size_t)kBlock * A.stack_depth * sizeof(uint32_t)) + threadIdx.x;
  TraceCounters tc;
  tc.box_tests = 0; tc.tri_tests = 0;
  unsigned int mism = 0;
  for (long long i = blockIdx.x * (long long)kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
    const float *r = rays + 6 * i;
    Hit h = closest_hit<TRAV, SMEM, STATS>(S, mk3(r[0], r[1], r[2]), mk3(r[3], r[4], r[5]), st, parks, kBlock, &tc, &mism);
    tri_out[i] = h.tri;
    k_out[i] = h.k;
  }
  flush(&A.counters->mismatches, warp_sum(mism));
  if (STATS) {
    flush(&A.counters->box_tests, warp_sum(tc.box_tests));
    flush(&A.counters->tri_tests, warp_sum(tc.tri_tests));
  }
}

// ---- accumulate / clamp / tonemap ---------------------------------------------------------------------------------------------
// out = clamp(sum of the parts / spp)   (Raytracing.cl:211-219), float4-vectorised when aligned; parts[] may live on peer
// GPUs (NVLink P2P loads) and are summed in rank order
struct PartList {
  const float *p[16];
  int n;
};
// spp <= 0: plain sum (partial sums of a partial sample range stay partial sums)
__global__ void k_reduce_finalize(const __grid_constant__ PartList parts, float *__restrict__ out, long long n4, long long n,
                                  float spp) {
  const bool fin = spp > 0.0f;
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long v = i; v < n4; v += stride) {
    float4 a = reinterpret_cast<const float4 *>(parts.p[0])[v];
    for (int r = 1; r < parts.n; ++r) {
      float4 b = reinterpret_cast<const float4 *>(parts.p[r])[v];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (fin) {
      a.x = clamp01(a.x / spp);
      a.y = clamp01(a.y / spp);
      a.z = clamp01(a.z / spp);
      a.w = clamp01(a.w / spp);
    }
    reinterpret_cast<float4 *>(out)[v] = a;
  }
  for (long long e = 4 * n4 + i; e < n; e += stride) {
    float a = parts.p[0][e];
    for (int r = 1; r < parts.n; ++r) a += parts.p[r][e];
    out[e] = fin ? clamp01(a / spp) : a;
  }
}

// 8-bit image as FileManager.saveImg makes it (FileManager.py:334-338): (data * 255).astype('uint8') — a float32
// product truncated toward zero; the input is already clamped to [0,1]
__global__ void k_quantize8(const float *__restrict__ in, uint8_t *__restrict__ out, long long n) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[i] = (uint8_t)__float2int_rz(in[i] * 255.0f);
}

// ImgProcessing.cl:1-9
__global__ void k_img_processing(const float *__restrict__ in, float *__restrict__ out, long long n, long long global) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < global; i += stride) {
    if (i < n) {
      float p = in[i];
      p = (1.0f < p) ? 1.0f : p;  // OpenCL min(x, y) = y < x ? y : x  (a NaN input stays NaN)
      out[i] = cr_pow(p, 2.2f);
    }
  }
}

// ---- probes -----------------------------------------------------------------------------------------------------------------------
// extent: the environment map's width (fn 11/12) or height (fn 13/14)
__global__ void k_math_probe(int fn, const float *a, const float *b, long long n, int extent, float *out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x = a[i], y = b[i], r = 0.0f;
  switch (fn) {
    case 0: r = cr_sin(x); break;
    case 1: r = cr_cos(x); break;
    case 2: r = cr_acos(x); break;
    case 3: r = cr_asin(x); break;
    case 4: r = cr_atan2(x, y); break;
    case 5: r = cr_tan(x); break;
    case 6: r = cr_pow(x, y); break;
    case 7: r = __fdiv_rn(x, y); break;
    case 8: r = sqrtf(x); break;
    case 9: { float s, c; cr_sincos(x, &s, &c); r = s; break; }
    case 10: { float s, c; cr_sincos(x, &s, &c); r = c; break; }
    case 11: r = (float)ibl_texel_u(x, y, extent); break;                       // fast path with its fallback
    case 12: r = (float)texel_coord(cr_atan2(x, y), 0.1591f, extent); break;    // correctly rounded angle only
    case 13: r = (float)ibl_texel_v(x, extent); break;
    case 14: r = (float)texel_coord(cr_asin(x), 0.3183f, extent); break;
    case 15: { const float a = atan2f(x, y), del = fabsf(a) * 4.76837158203125e-07f;   // 1 = the column needs the exact angle (600 wide)
               r = texel_coord(a - del, 0.1591f, 600) != texel_coord(a + del, 0.1591f, 600) ? 1.0f : 0.0f; break; }
    case 16: r = atan2f(x, y); break;
    case 17: r = asinf(x); break;
  }
  out[i] = r;
}

// One record of b200rt_rule_probe per thread: 16 floats in, 8 out (rule codes and layout in b200rt.h).  Every rule calls
// the functions k_shade calls and restates none of their statements.  What k_shade computes inline arrives as an input:
// the hit point x (o + unit(d) * k), the emitter triangle it picks with the light sample's first uniform, and the
// surface's material.  frames: per record, the frame k_tri_frames made of the record's normal (rules 2, 4, 6).
// b200rt_rule_probe has checked every index field.
__global__ void k_rule_probe(int rule, const float *__restrict__ in, long long n, const float4 *__restrict__ frames,
                             const SceneView S, int n_tris, const TexView T, float *__restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *a = in + 16 * i;
  const v3 d = mk3(a[0], a[1], a[2]), nr = mk3(a[3], a[4], a[5]), x = mk3(a[6], a[7], a[8]);
  const int i9 = __float_as_int(a[9]), i10 = __float_as_int(a[10]), i11 = __float_as_int(a[11]);
  const float u0 = bits_to_unit(__float_as_uint(a[12])), u1 = bits_to_unit(__float_as_uint(a[13]));
  const float u2 = bits_to_unit(__float_as_uint(a[14]));
  float r[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  v3 v = mk3(0.0f, 0.0f, 0.0f);
  bool flag = false;
  switch (rule) {
    case 0: v = scatter_dielectric(d, nr, a[6], u0, &flag); r[3] = flag ? 1.0f : 0.0f; break;
    case 1: v = scatter_rough_dielectric(d, nr, a[6], a[7], u0, u1, u2, &flag, &r[4]); r[3] = flag ? 1.0f : 0.0f; break;
    case 2: v = sample_cosine(nr, load_tri_frame(frames, (int)i, 1), u0, u1, &r[3]); break;
    case 3: v = sample_cosine(nr, tri_frame_at(nr, 1), u0, u1, &r[3]); break;
    case 4: v = sample_uniform(nr, load_tri_frame(frames, (int)i, 2), u0, u1, &r[3]); break;
    case 5: v = sample_uniform(nr, tri_frame_at(nr, 2), u0, u1, &r[3]); break;
    case 6: {
      const TriFrame tf = load_tri_frame(frames, (int)i, 2);
      Material m;
      m.type = 2;
      m.color = mk3(1.0f, 1.0f, 1.0f);
      m.roughness = a[6];
      v = sample_glossy_importance(m.roughness, tf.un, d, u0, u1, &r[3]);
      r[4] = bsdf_pdf(m, 1, tf.un, d, unit(v));
      break;
    }
    case 7: {
      Material m;
      m.type = 2;
      m.color = mk3(a[9], a[10], a[11]);
      m.roughness = a[12];
      v = bsdf_ggx(m, d, x, nr);
      break;
    }
    case 8: {
      const Material m = load_material(S.mats, i10);
      const Tri l = load_tri(S.tris, i9);
      const Material ml = load_material(S.mats, l.mat);
      const float Le = ml.type == 0 ? ml.roughness : 0.0f;
      const v3 un = unit(nr);
      const int sampling = __float_as_int(a[15]);
      v3 w;
      v = sample_light(m, sampling, nr, un, x, d, mk3(1.0f, 1.0f, 1.0f), l.A, l.e1, l.e2, Le, i11, u1, u2, &w);
      const float dist2 = dot(w, w);
      const v3 wi = w / sqrtf(dist2);
      r[3] = w.x; r[4] = w.y; r[5] = w.z;
      r[6] = light_pdf(l.e1, l.e2, i11, wi, dist2);
      r[7] = bsdf_pdf(m, sampling, un, d, wi);
      break;
    }
    case 9: {
      const float4 nn = __ldg(S.normals + i9);
      v = shading_normal<true>(S, n_tris, i9, mk3(nn.x, nn.y, nn.z), x, &flag);
      r[3] = flag ? 1.0f : 0.0f;
      break;
    }
    case 10: v = surface_albedo(S, n_tris, i9, i10, d, x); break;
    case 11: v = texture_factor(T, i9, a[6], a[7]); break;
  }
  r[0] = v.x; r[1] = v.y; r[2] = v.z;
  float *o = out + 8 * i;
  for (int k = 0; k < 8; ++k) o[k] = r[k];
}

__global__ void k_philox_probe(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out) {
  uint32_t o[4];
  philox4x32_10(c0, c1, c2, c3, k0, k1, o);
  out[0] = o[0]; out[1] = o[1]; out[2] = o[2]; out[3] = o[3];
}

}  // namespace b200rt
