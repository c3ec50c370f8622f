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
// meta: bit 0 first iteration (no ray traced yet), bit 1 light ray (opt-in light sampling), bit 3 sun ray, bits 4-7
// material type of the surface the ray left, bits 8-15 bounce j, bits 16-31 sample index
struct PathMeta {
  int first, light, sun, type, j, s;
};

RT_DEV uint32_t meta_pack(int first, int sun, int type, int j, int s, int light = 0) {
  return (uint32_t)first | ((uint32_t)light << 1) | ((uint32_t)sun << 3) | ((uint32_t)(type & 15) << 4) | ((uint32_t)(j & 255) << 8) | ((uint32_t)s << 16);
}

RT_DEV PathMeta meta_unpack(uint32_t m) {
  return {(int)(m & 1u), (int)((m >> 1) & 1u), (int)((m >> 3) & 1u), (int)((m >> 4) & 15u), (int)((m >> 8) & 255u), (int)(m >> 16)};
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

// ---- shading ----------------------------------------------------------------------------------------------------
// The per-path state machine is written as a sequence of phases with the warp re-converged between them, so that
// e.g. the direction sampling runs once per warp for every lane that needs it, whichever way the lane got there
// (bounce hit, or sample ended and the next one starts from the cached primary hit).
// 8 CTAs per SM: the kernel is bound by the latency of its gathers; 5-7 (no spills) and 9-12 resident CTAs were all slower.
// NEE = opt-in light sampling (b200rt_opts.sampling bit 1): a separate instantiation, so that the reference's
// estimator runs exactly the code it ran before.  ADAPT = adaptive sampling (adaptive_end_sample at the end of every
// sample), likewise a separate instantiation.
template <bool NEE, bool ADAPT>
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
    bool pixel_done = false, start = valid && first, shade = false, end_sample = false, sun_done = false;
    bool want_light = false, light_done = false, from_light = false;

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
      if (light_ray) {
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
    // ---- phase 3: a new sample starts from the cached primary hit (Raytracing.cl:195-201) --------------------------------------
    if (start) {
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
      const v3 n = mk3(nn.x, nn.y, nn.z);
      const Material m = load_material(S.mats, tri_material(S, htri));
      const v3 un = unit(n);
      float ul, ua, ub;
      if (F.rng_mode == 0) draw3_light<0>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1, &ul, &ua, &ub);
      else draw3_light<1>(g, (uint32_t)pix, (uint32_t)s, (uint32_t)j, F.key0, F.key1, &ul, &ua, &ub);
      int idx = (int)(ul * (float)A.n_light);
      if (idx > A.n_light - 1) idx = A.n_light - 1;
      const int lt = __ldg(A.light + idx);
      const Tri l = load_tri(S.tris, lt);
      const Material ml = load_material(S.mats, l.mat);
      const float Le = ml.type == 0 ? ml.roughness : 0.0f;
      const v3 x = o + unit(d) * hk;
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
      const v3 n = mk3(nn.x, nn.y, nn.z);
      const Material m = load_material(S.mats, tri_material(S, htri));
      const TriFrame tf = load_tri_frame(S.frames, htri, m.type == 3 ? 0 : (m.type == 1 ? 1 : 2));
      v3 nd, brdf;
      float inv_pdf;
      if (m.type == 3) {
        nd = d;
        brdf = m.color;
        inv_pdf = 1.0f / fabsf(dot(nd, tf.un));
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
      const float att = inv_pdf * fabsf(dot(nd, tf.un));
      acc = (acc * brdf) * att;
      seg_type = m.type;
      sun_ray = 0;
    }
    __syncwarp();

    // ---- phase 5: store, join the next list -----------------------------------------------------------------------------------------
    const bool alive = valid && !pixel_done;
    if (alive) {
      A.pA[pix] = make_float4(o.x, o.y, o.z, d.x);
      A.pB[pix] = make_float4(d.y, d.z, __uint_as_float(meta_pack(0, sun_ray, seg_type, j, s, (NEE && want_light) ? 1 : 0)),
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
__global__ void k_math_probe(int fn, const float *a, const float *b, long long n, float *out) {
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
    case 11: r = (float)ibl_texel_u(x, y, 8192); break;                       // fast path with its fallback
    case 12: r = (float)texel_coord(cr_atan2(x, y), 0.1591f, 8192); break;    // correctly rounded angle only
    case 13: r = (float)ibl_texel_v(x, 4096); break;
    case 14: r = (float)texel_coord(cr_asin(x), 0.3183f, 4096); break;
    case 15: { const float a = atan2f(x, y), del = fabsf(a) * 4.76837158203125e-07f;   // 1 = the column needs the exact angle (600 wide)
               r = texel_coord(a - del, 0.1591f, 600) != texel_coord(a + del, 0.1591f, 600) ? 1.0f : 0.0f; break; }
    case 16: r = atan2f(x, y); break;
  }
  out[i] = r;
}

__global__ void k_philox_probe(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out) {
  uint32_t o[4];
  philox4x32_10(c0, c1, c2, c3, k0, k1, o);
  out[0] = o[0]; out[1] = o[1]; out[2] = o[2]; out[3] = o[3];
}

}  // namespace b200rt
