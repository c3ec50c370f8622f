// b200rt — host side of the C ABI declared in include/b200rt.h.
//
// Owns the CUDA context objects of one GPU, validates and repacks the reference-layout scene
// buffers (SURVEY.md §8a) into the float4 layouts rt_trace.cuh consumes, evaluates the per-frame
// constants, and launches the kernels of rt_kernels.cuh.  No CPU rendering path exists here: every
// entry point that produces pixels, hits or tonemapped values does so by launching a kernel.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/b200rt.h"
#include "rt_denoise.cuh"
#include "scene_repack.h"

using namespace b200rt;

namespace {

thread_local std::string g_create_error;

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  bool borrowed = false;  // a helper context's view of its parent's scene buffer: never freed or resized here
};

// the scene's device buffers, which sample-stream helpers borrow as a set
enum SceneBuf { kNodes, kTris, kCtris, kNormals, kTboxes, kFrames, kMats, kBvh9, kLeafcnt, kLight, kSceneBufs };

// Resident k_trace CTAs per SM while three or more sample streams share the GPU.  A k_trace that fills every SM's
// register file leaves the other streams' kernels nothing but its tail to run in; capped, one stream's shading and
// another's tracing are resident side by side (bench scene -4 %, Cornell 1080p -12 %, measured with 3 streams).
constexpr int kStreamTraceCtas = 4;

}  // namespace

struct b200rt_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;      // stream in use
  cudaStream_t own_stream = nullptr;  // created by b200rt_create
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> kev;  // per-launch events of the last time_kernels render
  int kev_used = 0;
  std::string err;
  int sm_count = 0;
  size_t smem_optin = 0;

  // scene
  bool have_scene = false;
  bool have_scene_cached = false;  // scene_hash / ibl_hash are valid
  uint64_t scene_hash = 0, mat_hash = 0;
  DevBuf d_scene[kSceneBufs];  // kLight: triangles whose material is emissive, ascending (opt-in light sampling)
  SceneDesc scene;
  int n_mats = 0;
  int n_light = 0;
  int frame_trace_cap = 0; // resident k_trace CTAs per SM in the frame being enqueued (0 = what fits; set by render_frame)
  std::vector<int32_t> tri_mat;  // for re-validating material edits
  DevBuf d_pS, d_pL, d_pR;       // light sampling: three more float4 of path state

  // environment map
  bool have_ibl = false;
  uint64_t ibl_hash = 0;
  cudaArray_t ibl_array = nullptr;
  cudaTextureObject_t ibl_tex = 0;
  int ibl_w = 0, ibl_h = 0;

  // per-frame
  DevBuf d_prim_dirk, d_prim_tri, d_out, d_misc, d_tmp_a, d_tmp_b;
  DevBuf d_pA, d_pB, d_pC, d_pHit, d_list0, d_list1, d_cnt;  // wavefront path state (rt_kernels.cuh)
  DevBuf d_slots, d_part_count;                               // order-preserving list compaction
  DevBuf d_welford, d_ad_spp, d_ad_err;                       // adaptive sampling (AdaptArgs)
  DevBuf d_dn_tri, d_dn_k, d_gb[3], d_dn_col[2];              // denoising: primary hits, G-buffer (GBufferView), colour
  unsigned int *h_live = nullptr;   // adaptive sampling: pinned, the path-list length after each of the two batches in flight
  cudaEvent_t ev_batch[2] = {nullptr, nullptr};
  DeviceCounters *d_counters = nullptr;

  b200rt_stats stats;
  bool stats_pending = false;  // async render enqueued; counters/events not read yet

  // sample streams (b200rt_opts.sample_streams): helper contexts on the same GPU, each with its own stream and path
  // state, that borrow this context's scene and environment
  std::vector<b200rt_ctx *> helpers;
  bool is_helper = false;
  uint64_t scene_epoch = 1, shared_epoch = 0;   // helpers re-borrow when the parent's scene / materials / map changed
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_done = nullptr;
  DevBuf d_part;               // this context's own partial sums when the frame is cut into streams
  int streams_used = 1;        // of the last render
};

namespace {

// B200RT_CULL_TREE=0 keeps the caller's tree topology in the node records (development A/B; default: own tree)
bool own_cull_tree() {
  const char *q = getenv("B200RT_CULL_TREE");
  return !(q && q[0] == '0');
}

int fail(b200rt_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(c, B200RT_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

}  // namespace

static_assert(kRefStack == kRefStackMax, "scene_repack.h and rt_trace.cuh disagree on the exact walk's stack");
size_t b200rt::lane_smem_bytes_host(int stack_depth) { return lane_smem_bytes(stack_depth); }

namespace {

int ensure(b200rt_ctx *c, DevBuf &b, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (b.borrowed) return fail(c, B200RT_ERR_INVALID, "internal: resize of a borrowed scene buffer");
  if (b.cap >= bytes) return 0;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  CU(cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return 0;
}

uint64_t hash_bytes(const void *p, size_t n, uint64_t h) {
  const unsigned char *b = static_cast<const unsigned char *>(p);
  size_t i = 0;
  for (; i + 8 <= n; i += 8) {
    uint64_t w;
    memcpy(&w, b + i, 8);
    h = (h ^ w) * 0x9E3779B97F4A7C15ull;
    h ^= h >> 29;
  }
  for (; i < n; ++i) h = (h ^ b[i]) * 0x100000001B3ull;
  return h ^ (uint64_t)n;
}

// correctly-rounded binary32 cos/sin/tan on the host: binary64 libm, one rounding (rt_math.cuh contract)
float h_cos(float a) { return (float)std::cos((double)a); }
float h_sin(float a) { return (float)std::sin((double)a); }
float h_tan(float a) { return (float)std::tan((double)a); }

rotor h_rotor(float angle, v3 axis) {
  float half = angle * 0.5f;
  return make_rotor(h_cos(half), h_sin(half), axis);
}

const float kDeg2Rad = 3.14f / 180.0f;

// Per-frame constants.  Raytracing.cl:24,27,33-35,115-118 and MathLib.cl:73-74.
void frame_setup(const b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp,
                 int max_bounce, const b200rt_opts &o, FrameParams *F) {
  F->width = width;
  F->height = height;
  F->cam_pos = mk3(cam[0], cam[1], cam[2]);
  F->focal_off = 1.0f / (2.0f * h_tan(cam[9] / 2.0f));
  F->step = (float)(1.0 / (double)cam[6]);
  F->cam_rx = h_rotor(cam[3] * kDeg2Rad, mk3(1, 0, 0));
  F->cam_ry = h_rotor(cam[4] * kDeg2Rad, mk3(0, 1, 0));
  F->cam_rz = h_rotor(cam[5] * kDeg2Rad, mk3(0, 0, 1));
  v3 s = mk3(1, 1, 1);
  if (env) {
    s = apply_rotor(h_rotor(env[0] * kDeg2Rad, mk3(1, 0, 0)), s);
    s = apply_rotor(h_rotor(env[1] * kDeg2Rad, mk3(0, 1, 0)), s);
    s = apply_rotor(h_rotor(env[2] * kDeg2Rad, mk3(0, 0, 1)), s);
  }
  F->sun_dir = s;
  F->sun_power = env ? env[3] : 0.0f;
  F->ibl_power = env ? env[4] : 0.0f;
  F->ibl_r1 = h_rotor(90 * kDeg2Rad, mk3(1, 0, 0));
  F->ibl_r2 = h_rotor(90 * kDeg2Rad, mk3(0, 1, 0));
  F->ibl_w = c->ibl_w;
  F->ibl_h = c->ibl_h;
  F->spp = spp;
  F->max_bounce = max_bounce;
  F->s0 = o.sample_begin;
  F->s1 = o.sample_end;
  if (F->s1 <= 0) { F->s0 = 0; F->s1 = spp; }
  F->pixel_begin = o.pixel_begin;
  F->pixel_end = o.pixel_end;
  if (F->pixel_end <= 0) { F->pixel_begin = 0; F->pixel_end = width * height; }
  F->tile_row_mod = o.tile_row_mod;
  F->tile_row_rem = o.tile_row_rem;
  F->out_mode = o.output;
  F->rng_mode = o.rng_mode;
  F->key0 = (uint32_t)(o.seed & 0xffffffffull);
  F->key1 = (uint32_t)(o.seed >> 32);
  F->sampling = o.sampling;
}

size_t scene_smem_bytes(const b200rt_ctx *c) { return (size_t)c->scene.n_inner * 48 + (size_t)c->scene.n_tris * 48; }

bool use_smem_scene(const b200rt_ctx *c) { return c->scene.node_f4 == 3; }

// entries of the per-lane shared-memory traversal stack: the near-first walk holds at most one entry per level;
// trees walked in reference order keep their stack in thread-local memory instead
int stack_entries(const b200rt_ctx *c) { return c->scene.canonical ? c->scene.cull_depth + 2 : 2; }

size_t smem_bytes(const b200rt_ctx *c, bool smem_scene) {
  return lane_smem_bytes(stack_entries(c)) + (smem_scene ? scene_smem_bytes(c) : 0);
}

int effective_stack_cap(const b200rt_ctx *c, const b200rt_opts &o);

void fill_args(b200rt_ctx *c, const FrameParams &F, const b200rt_opts &o, float *d_out, KernelArgs *A) {
  A->F = F;
  const SceneDesc &D = c->scene;
  const DevBuf *B = c->d_scene;
  SceneView &S = A->S;
  S.nodes = static_cast<const uint4 *>(B[kNodes].p);
  S.node_f4 = D.node_f4;
  S.tris = static_cast<const float4 *>(B[kTris].p);
  S.ctris = static_cast<const float4 *>(B[kCtris].p);
  S.normals = static_cast<const float4 *>(B[kNormals].p);
  S.tboxes = static_cast<const float4 *>(B[kTboxes].p);
  S.frames = static_cast<const float4 *>(B[kFrames].p);
  S.mats = static_cast<const float *>(B[kMats].p);
  S.bvh9 = static_cast<const float *>(B[kBvh9].p);
  S.leafcnt = static_cast<const int *>(B[kLeafcnt].p);
  S.root_ref = D.root_ref;
  for (int i = 0; i < 3; ++i) {
    S.grid_base[i] = D.grid_base[i];
    S.grid_pitch[i] = D.grid_pitch[i];
    S.root_w[i] = D.root_w[i];
  }
  S.cull_abs = D.cull_abs;
  S.cmax = D.cmax;
  {
    // traversal-stack entry layout (rt_trace.cuh, LaneStack): 2^E above every culling limit, refs in the low bits
    const int E = std::ilogb((1001.0f + D.cull_abs) * 1.01f) + 1;
    S.st_bias = (uint32_t)(E - 32 + 127) << 23;
    unsigned long long m = 1;
    while (m < (unsigned long long)std::max(1, D.n_inner) * (unsigned long long)std::max(1, D.node_f4)) m <<= 1;
    S.st_rmask = (uint32_t)(m - 1ull);
  }
  S.stack_cap = effective_stack_cap(c, o);
  S.fast_ok = D.fast_ok;
  A->ibl = c->ibl_tex;
  A->prim_dirk = static_cast<float4 *>(c->d_prim_dirk.p);
  A->prim_tri = static_cast<int *>(c->d_prim_tri.p);
  A->out = d_out;
  A->pA = static_cast<float4 *>(c->d_pA.p);
  A->pB = static_cast<float4 *>(c->d_pB.p);
  A->pC = static_cast<float4 *>(c->d_pC.p);
  A->pHit = static_cast<int2 *>(c->d_pHit.p);
  A->light = static_cast<const int *>(B[kLight].p);
  A->n_light = c->n_light;
  A->pS = static_cast<float4 *>(c->d_pS.p);
  A->pL = static_cast<float4 *>(c->d_pL.p);
  A->pR = static_cast<float4 *>(c->d_pR.p);
  A->list[0] = static_cast<int *>(c->d_list0.p);
  A->list[1] = static_cast<int *>(c->d_list1.p);
  A->cnt = static_cast<unsigned int *>(c->d_cnt.p);
  A->slots = static_cast<int *>(c->d_slots.p);
  A->part_count = static_cast<unsigned int *>(c->d_part_count.p);
  A->wc = nullptr;
  A->counters = c->d_counters;
  A->n_nodes = D.n_inner;
  A->n_tris = D.n_tris;
  A->stack_depth = stack_entries(c);
  A->tiles_x = (F.width + 7) / 8;
  int tiles_y = (F.height + 3) / 4;
  A->n_work = A->tiles_x * tiles_y * 32;
  A->validate = 0;
  A->ad = AdaptArgs();
}

// The fast path needs a strict two-child tree with nested boxes; any other tree is walked in reference order.  When
// the caller asked for FAST (a walk that never drops a push) the substitute keeps that promise as far as its
// thread-local stack reaches: it runs with the largest cap instead of the reference's 20.
int effective_traversal(const b200rt_ctx *c, const b200rt_opts &o) {
  if (!c->scene.canonical) return B200RT_TRAVERSAL_REFERENCE;
  return o.traversal;
}

int effective_stack_cap(const b200rt_ctx *c, const b200rt_opts &o) {
  if (!c->scene.canonical && o.traversal == B200RT_TRAVERSAL_FAST) return kRefStack;
  return o.stack_cap <= 0 ? 20 : (o.stack_cap > kRefStack ? kRefStack : o.stack_cap);
}

template <typename K>
int set_smem_attr(b200rt_ctx *c, K kernel, size_t bytes) {
  if (bytes > 48 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

template <typename K>
int persistent_grid(b200rt_ctx *c, K kernel, size_t smem, int *grid) {
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem));
  if (per_sm < 1) return fail(c, B200RT_ERR_CUDA, "kernel does not fit on an SM (smem %zu)", smem);
  *grid = per_sm * c->sm_count;
  return 0;
}

// Calls f(trav, smem, stats) with the three as std::integral_constant, so that f can name the kernel instance.  VERIFY
// has no STATS instance: asked for stats, it runs the one without.
template <int TRAV, bool SMEM, class F>
int with_stats(bool stats, F &f) {
  using T = std::integral_constant<int, TRAV>;
  using S = std::bool_constant<SMEM>;
  if constexpr (TRAV != B200RT_TRAVERSAL_VERIFY) {
    if (stats) return f(T{}, S{}, std::true_type{});
  }
  return f(T{}, S{}, std::false_type{});
}

template <class F>
int with_variant(b200rt_ctx *c, int trav, bool smem, bool stats, F &&f) {
  switch (trav) {
    case 0: return smem ? with_stats<0, true>(stats, f) : with_stats<0, false>(stats, f);
    case 1: return smem ? with_stats<1, true>(stats, f) : with_stats<1, false>(stats, f);
    case 2: return smem ? with_stats<2, true>(stats, f) : with_stats<2, false>(stats, f);
  }
  return fail(c, B200RT_ERR_INVALID, "bad traversal mode %d", trav);
}

template <int TRAV, bool SMEM, bool PARITY, bool STATS>
int launch_primary_t(b200rt_ctx *c, const KernelArgs &A, int *tri_out, float *k_out) {
  auto k = k_primary<TRAV, SMEM, PARITY, STATS>;
  size_t smem = smem_bytes(c, SMEM);
  int grid = 0;
  if (set_smem_attr(c, k, smem)) return B200RT_ERR_CUDA;
  if (persistent_grid(c, k, smem, &grid)) return B200RT_ERR_CUDA;
  int need = (A.n_work + kBlock - 1) / kBlock;
  if (grid > need) grid = need;
  k<<<grid, kBlock, smem, c->stream>>>(A, tri_out, k_out);
  CU(cudaGetLastError());
  c->stats.kernel_launches++;
  return 0;
}

int launch_primary(b200rt_ctx *c, const KernelArgs &A, int trav, bool smem, bool parity, bool stats, int *tri_out,
                   float *k_out) {
  return with_variant(c, trav, smem, stats, [&](auto t, auto s, auto st) {
    constexpr int T = decltype(t)::value;
    constexpr bool S = decltype(s)::value, ST = decltype(st)::value;
    return parity ? launch_primary_t<T, S, true, ST>(c, A, tri_out, k_out)
                  : launch_primary_t<T, S, false, ST>(c, A, tri_out, k_out);
  });
}

// Launch geometry of the wavefront kernels, resolved once per frame (the occupancy queries are host calls)
struct WaveLaunch {
  void (*shade)(const KernelArgs, int) = nullptr;
  void (*trace)(const KernelArgs, int) = nullptr;
  int trace_grid = 0;
  size_t trace_smem = 0;
  int shade_grid = 0;
};

template <int TRAV, bool SMEM, bool STATS>
int prepare_trace_t(b200rt_ctx *c, WaveLaunch *w) {
  auto k = k_trace<TRAV, SMEM, STATS>;
  w->trace_smem = smem_bytes(c, SMEM);
  if (set_smem_attr(c, k, w->trace_smem)) return B200RT_ERR_CUDA;
  if (persistent_grid(c, k, w->trace_smem, &w->trace_grid)) return B200RT_ERR_CUDA;
  const int cap = c->frame_trace_cap;
  if (cap > 0 && w->trace_grid > cap * c->sm_count) w->trace_grid = cap * c->sm_count;
  w->trace = k;
  return 0;
}

int prepare_wave(b200rt_ctx *c, int trav, bool smem, bool stats, bool nee, bool adaptive, WaveLaunch *w) {
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_shade<false, false>, kShadeBlock, 0));
  if (per_sm < 1) return fail(c, B200RT_ERR_CUDA, "k_shade does not fit on an SM");
  w->shade_grid = per_sm * c->sm_count;
  if (nee) w->shade = adaptive ? k_shade<true, true> : k_shade<true, false>;
  else w->shade = adaptive ? k_shade<false, true> : k_shade<false, false>;
  return with_variant(c, trav, smem, stats, [&](auto t, auto s, auto st) {
    return prepare_trace_t<decltype(t)::value, decltype(s)::value, decltype(st)::value>(c, w);
  });
}

template <int TRAV, bool SMEM, bool STATS>
int launch_trace_t(b200rt_ctx *c, const KernelArgs &A, const float *rays, long long n, int *tri, float *k) {
  auto kern = k_trace_rays<TRAV, SMEM, STATS>;
  size_t smem = smem_bytes(c, SMEM);
  if (set_smem_attr(c, kern, smem)) return B200RT_ERR_CUDA;
  int grid = 0;
  if (persistent_grid(c, kern, smem, &grid)) return B200RT_ERR_CUDA;
  long long need = (n + kBlock - 1) / kBlock;
  if (grid > need) grid = (int)(need < 1 ? 1 : need);
  kern<<<grid, kBlock, smem, c->stream>>>(A, rays, n, tri, k);
  CU(cudaGetLastError());
  c->stats.kernel_launches++;
  return 0;
}

int read_counters_one(b200rt_ctx *c) {
  DeviceCounters h;
  CU(cudaSetDevice(c->device));
  CU(cudaMemcpyAsync(&h, c->d_counters, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->stats.rays = h.rays;
  c->stats.primary_rays = h.primary_rays;
  c->stats.box_tests = h.box_tests;
  c->stats.tri_tests = h.tri_tests;
  c->stats.mismatches = h.mismatches;
  c->stats.samples = h.samples;
  c->stats.revalidated = (int32_t)(h.revalidated > 0x7fffffffull ? 0x7fffffffull : h.revalidated);
  c->stats.exact_walks = (int32_t)(h.exact_walks > 0x7fffffffull ? 0x7fffffffull : h.exact_walks);
  float ms = 0;
  if (cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]) == cudaSuccess) c->stats.primary_ms = ms;
  if (cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]) == cudaSuccess) c->stats.trace_ms = ms;
  if (cudaEventElapsedTime(&ms, c->ev[0], c->ev[2]) == cudaSuccess) c->stats.total_ms = ms;
  c->stats.shade_kernel_ms = 0.0f;
  c->stats.trace_kernel_ms = 0.0f;
  for (int i = 0; i + 1 < c->kev_used; ++i)  // event i sits before launch i; launches alternate shade, trace, shade, ...
    if (cudaEventElapsedTime(&ms, c->kev[i], c->kev[i + 1]) == cudaSuccess)
      ((i & 1) ? c->stats.trace_kernel_ms : c->stats.shade_kernel_ms) += ms;
  c->kev_used = 0;
  c->stats_pending = false;
  return 0;
}

// the additive work counters of one render; times, scene facts and primary_rays are each caller's own rule
void add_work(b200rt_stats &dst, const b200rt_stats &src) {
  dst.rays += src.rays;
  dst.box_tests += src.box_tests;
  dst.tri_tests += src.tri_tests;
  dst.mismatches += src.mismatches;
  dst.samples += src.samples;
  dst.revalidated += src.revalidated;
  dst.exact_walks += src.exact_walks;
  dst.kernel_launches += src.kernel_launches;
}

// Counters and timings of the last render.  A frame cut into sample streams sums the work of its helper contexts
// (the primary rays, which every stream traces for itself, count once) and is timed from the fork to the reduce.
int read_counters(b200rt_ctx *c) {
  int rc = read_counters_one(c);
  if (rc || c->streams_used <= 1) return rc;
  for (int k = 1; k < c->streams_used; ++k) {
    b200rt_ctx *h = c->helpers[(size_t)k - 1];
    rc = read_counters_one(h);
    if (rc) return fail(c, rc, "sample stream %d: %s", k, h->err.c_str());
    add_work(c->stats, h->stats);
    c->stats.rays -= h->stats.primary_rays;
    c->stats.shade_kernel_ms += h->stats.shade_kernel_ms;   // kernels of different streams overlap: these are sums of
    c->stats.trace_kernel_ms += h->stats.trace_kernel_ms;   // durations, not a partition of total_ms
    c->stats.primary_ms = std::max(c->stats.primary_ms, h->stats.primary_ms);
  }
  float ms = 0;
  if (cudaEventElapsedTime(&ms, c->ev_fork, c->ev_done) == cudaSuccess) {
    c->stats.total_ms = ms;
    c->stats.trace_ms = ms - c->stats.primary_ms;
  }
  c->stats.kernel_launches += 1;  // the reduce
  return 0;
}

int check_frame_args(b200rt_ctx *c, const float *cam, int width, int height, int spp, int max_bounce,
                     const b200rt_opts &o, bool need_env, const float *env) {
  if (!cam) return fail(c, B200RT_ERR_INVALID, "cam is NULL");
  if (need_env && !env) return fail(c, B200RT_ERR_INVALID, "envData is NULL");
  if (!c->have_scene) return fail(c, B200RT_ERR_NO_SCENE, "no scene: call b200rt_set_scene first");
  if (width <= 0 || height <= 0 || (long long)width * height > 0x7fffffffLL / 4)
    return fail(c, B200RT_ERR_INVALID, "bad frame size %d x %d", width, height);
  if ((int)cam[6] != width)
    return fail(c, B200RT_ERR_INVALID, "cam[6] = %g but width = %d (the kernel derives rows/columns from cam[6])",
                (double)cam[6], width);
  if (spp <= 0) return fail(c, B200RT_ERR_INVALID, "spp must be positive (got %d)", spp);
  if (max_bounce < 0) return fail(c, B200RT_ERR_INVALID, "maxBounce must be >= 0 (got %d)", max_bounce);
  // the per-path state packs the sample index into 16 bits and the bounce into 8 (rt_kernels.cuh meta_pack)
  if (spp > 65535) return fail(c, B200RT_ERR_UNSUPPORTED, "spp %d exceeds 65535 per launch; accumulate several launches with sample ranges", spp);
  if (max_bounce > 254) return fail(c, B200RT_ERR_UNSUPPORTED, "maxBounce %d exceeds 254", max_bounce);
  if (o.rng_mode != B200RT_RNG_REFERENCE && o.rng_mode != B200RT_RNG_PHILOX)
    return fail(c, B200RT_ERR_INVALID, "bad rng_mode %d", o.rng_mode);
  if (o.traversal < 0 || o.traversal > 2) return fail(c, B200RT_ERR_INVALID, "bad traversal %d", o.traversal);
  if (o.sampling < 0 || o.sampling > (B200RT_SAMPLING_IMPORTANCE | B200RT_SAMPLING_LIGHTS))
    return fail(c, B200RT_ERR_INVALID, "bad sampling mode %d", o.sampling);
  if (o.output != B200RT_OUT_FINAL && o.output != B200RT_OUT_SUMS)
    return fail(c, B200RT_ERR_INVALID, "bad output mode %d", o.output);
  if (o.sample_end > 0) {
    if (o.sample_begin < 0 || o.sample_begin >= o.sample_end || o.sample_end > spp)
      return fail(c, B200RT_ERR_INVALID, "bad sample range [%d,%d) for spp %d", o.sample_begin, o.sample_end, spp);
    if (o.sample_begin != 0 && o.rng_mode == B200RT_RNG_REFERENCE)
      return fail(c, B200RT_ERR_INVALID,
                  "a sample range that does not start at 0 needs B200RT_RNG_PHILOX: the reference generator is one "
                  "serial stream per pixel");
    if ((o.sample_begin != 0 || o.sample_end != spp) && o.output != B200RT_OUT_SUMS)
      return fail(c, B200RT_ERR_INVALID, "a partial sample range only makes sense with B200RT_OUT_SUMS");
  }
  if (o.tile_row_mod > 1 && (o.tile_row_rem < 0 || o.tile_row_rem >= o.tile_row_mod))
    return fail(c, B200RT_ERR_INVALID, "bad tile row split %d mod %d", o.tile_row_rem, o.tile_row_mod);
  if (o.pixel_end > 0 && (o.pixel_begin < 0 || o.pixel_begin >= o.pixel_end || o.pixel_end > width * height))
    return fail(c, B200RT_ERR_INVALID, "bad pixel range [%d,%d)", o.pixel_begin, o.pixel_end);
  return 0;
}

constexpr int kAdaptBatch = 32;  // adaptive renders: wavefront iterations enqueued between two looks at the list length

// ad != NULL: adaptive sampling (b200rt_render_adaptive has validated ad and opts; the frame covers [0, spp) on one
// stream).  The launch loop then runs in batches and stops once the path list is empty; it is synchronous.
int render_impl(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                const b200rt_opts *opts, float *d_out, const b200rt_adaptive *ad) {
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  c->streams_used = 1;
  int rc = check_frame_args(c, cam, width, height, spp, max_bounce, o, true, env);
  if (rc) return rc;
  if (!c->have_ibl) return fail(c, B200RT_ERR_NO_SCENE, "no environment map: call b200rt_set_ibl first");
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)width * height;
  FrameParams F;
  frame_setup(c, cam, env, width, height, spp, max_bounce, o, &F);
  // every live path traces exactly one ray per iteration and a sample needs at most max_bounce + 1 bounce rays
  // plus one sun ray (Raytracing.cl:46-137)
  // with light sampling every surface that scatters adds one shadow ray towards an emitter: up to 2 (max_bounce + 1) + 1
  const bool nee = (o.sampling & B200RT_SAMPLING_LIGHTS) != 0 && c->n_light > 0;
  const long long per_sample = nee ? 2 * ((long long)max_bounce + 1) + 1 : (long long)max_bounce + 2;
  const long long n_iter_ll = (long long)(F.s1 - F.s0) * per_sample;
  if (n_iter_ll > (1 << 22)) return fail(c, B200RT_ERR_UNSUPPORTED, "%lld wavefront iterations exceed 2^22", n_iter_ll);
  const int n_iter = (int)n_iter_ll;
  if (ensure(c, c->d_prim_dirk, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_prim_tri, npix * sizeof(int))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_pA, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_pB, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_pC, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_pHit, npix * sizeof(int2))) return B200RT_ERR_CUDA;
  if (nee) {
    if (ensure(c, c->d_pS, npix * sizeof(float4))) return B200RT_ERR_CUDA;
    if (ensure(c, c->d_pL, npix * sizeof(float4))) return B200RT_ERR_CUDA;
    if (ensure(c, c->d_pR, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  }
  if (ensure(c, c->d_list0, npix * sizeof(int))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_list1, npix * sizeof(int))) return B200RT_ERR_CUDA;
  const size_t n_work = (size_t)((width + 7) / 8) * ((height + 3) / 4) * 32;   // tile-ordered work items of k_primary
  if (ensure(c, c->d_slots, n_work * sizeof(int))) return B200RT_ERR_CUDA;
  const size_t n_cnt = (size_t)n_iter + 2;             // cnt[0 .. n_iter + 1]
  const size_t cnt_bytes = (n_cnt + (size_t)n_iter + 1) * sizeof(unsigned int);  // then wc[0 .. n_iter]
  if (ensure(c, c->d_cnt, cnt_bytes)) return B200RT_ERR_CUDA;
  KernelArgs A;
  fill_args(c, F, o, d_out, &A);
  A.wc = A.cnt + n_cnt;
  const int trav = effective_traversal(c, o);
  A.validate = (trav == B200RT_TRAVERSAL_FAST) ? 1 : 0;
  const bool smem = use_smem_scene(c);
  WaveLaunch wl;
  rc = prepare_wave(c, trav, smem, o.collect_stats != 0, nee, ad != nullptr, &wl);
  if (rc) return rc;
  if (ensure(c, c->d_part_count, (size_t)wl.shade_grid * sizeof(unsigned int))) return B200RT_ERR_CUDA;
  A.part_count = static_cast<unsigned int *>(c->d_part_count.p);
  A.slots = static_cast<int *>(c->d_slots.p);
  c->stats.kernel_launches = 0;
  c->stats.sample_streams = 1;
  c->stats.scene_in_smem = smem ? 1 : 0;
  CU(cudaMemsetAsync(c->d_counters, 0, sizeof(DeviceCounters), c->stream));
  CU(cudaMemsetAsync(c->d_cnt.p, 0, cnt_bytes, c->stream));
  CU(cudaEventRecord(c->ev[0], c->stream));
  if (ad) {
    if (ensure(c, c->d_welford, npix * sizeof(float2))) return B200RT_ERR_CUDA;
    if (ensure(c, c->d_ad_spp, npix * sizeof(int))) return B200RT_ERR_CUDA;
    if (ensure(c, c->d_ad_err, npix * sizeof(float))) return B200RT_ERR_CUDA;
    A.ad.welford = static_cast<float2 *>(c->d_welford.p);
    A.ad.spp_out = static_cast<int *>(c->d_ad_spp.p);
    A.ad.err_out = static_cast<float *>(c->d_ad_err.p);
    A.ad.min_spp = ad->min_spp;
    A.ad.check_every = ad->check_every;
    A.ad.rel_error = ad->rel_error;
    A.ad.floor = ad->floor;
    if (!c->h_live) CU(cudaMallocHost(&c->h_live, 2 * sizeof(unsigned int)));
    for (int k = 0; k < 2; ++k)
      if (!c->ev_batch[k]) CU(cudaEventCreateWithFlags(&c->ev_batch[k], cudaEventDisableTiming));
    // pixels outside the rendered set read 0 in both maps
    CU(cudaMemsetAsync(c->d_ad_spp.p, 0, npix * sizeof(int), c->stream));
    CU(cudaMemsetAsync(c->d_ad_err.p, 0, npix * sizeof(float), c->stream));
    const int grid = (int)std::min<long long>(((long long)A.n_work + 255) / 256, (long long)c->sm_count * 8);
    k_adaptive_init<<<grid, 256, 0, c->stream>>>(A);
    CU(cudaGetLastError());
    c->stats.kernel_launches++;
  }
  rc = launch_primary(c, A, trav, smem, false, o.collect_stats != 0, nullptr, nullptr);
  if (rc) return rc;
  // the first path list: k_primary's live pixels in tile order
  k_count_parts<<<wl.shade_grid, kCompactBlock, 0, c->stream>>>(A.slots, (unsigned)A.n_work, A.part_count);
  k_compact<<<wl.shade_grid, kCompactBlock, 0, c->stream>>>(A.slots, nullptr, (unsigned)A.n_work, A.part_count, A.list[0], A.cnt);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ev[1], c->stream));
  c->kev_used = 0;
  if (o.time_kernels) {
    const size_t need = 2 * (size_t)n_iter + 2;
    while (c->kev.size() < need) {
      cudaEvent_t e;
      CU(cudaEventCreate(&e));
      c->kev.push_back(e);
    }
  }
  // A fixed-spp frame is one batch of every iteration, enqueued without a look back.  An adaptive frame runs batches of
  // kAdaptBatch iterations rounded up to a multiple of kCompactEvery, so that every batch ends with a compaction and its
  // last cnt word is the number of live paths.  That word is copied to pinned memory behind an event; before batch k + 2
  // is enqueued the host waits for batch k's and stops once it is 0.  One batch is always in flight, so the GPU does not
  // wait for the host.  A k_shade on an empty list does nothing, so stopping there leaves the image the full loop would
  // make.
  const int batch = ad ? (kAdaptBatch + kCompactEvery - 1) / kCompactEvery * kCompactEvery : n_iter + 1;
  int it = 0, n_shade = 0, n_trace = 0, n_compactions = 0;
  for (int b = 0; it <= n_iter; ++b) {
    if (ad && b >= 2) {
      CU(cudaEventSynchronize(c->ev_batch[b & 1]));
      if (c->h_live[b & 1] == 0u) break;
    }
    const int end = std::min(it + batch, n_iter + 1);
    for (; it < end; ++it) {
      if (o.time_kernels) CU(cudaEventRecord(c->kev[c->kev_used++], c->stream));
      wl.shade<<<wl.shade_grid, kShadeBlock, 0, c->stream>>>(A, it);
      ++n_shade;
      if (it < n_iter && (it + 1) % kCompactEvery == 0) {  // close the gaps the finished pixels left, order kept (timed with k_shade)
        k_compact<<<wl.shade_grid, kCompactBlock, 0, c->stream>>>(A.slots, A.cnt + it, 0u, A.part_count, A.list[(it + 1) & 1], A.cnt + it + 1);
        ++n_compactions;
      }
      if (o.time_kernels) CU(cudaEventRecord(c->kev[c->kev_used++], c->stream));
      if (it < n_iter) {
        wl.trace<<<wl.trace_grid, kBlock, wl.trace_smem, c->stream>>>(A, it);
        ++n_trace;
      }
    }
    CU(cudaGetLastError());
    if (ad) {
      CU(cudaMemcpyAsync(&c->h_live[b & 1], A.cnt + end, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
      CU(cudaEventRecord(c->ev_batch[b & 1], c->stream));
    }
  }
  // k_count_parts + k_compact for the first list, then what the loop launched
  c->stats.kernel_launches += 2 + n_shade + n_compactions + n_trace;
  c->stats.wave_iterations = n_trace;
  CU(cudaEventRecord(c->ev[2], c->stream));
  c->stats_pending = true;
  return 0;
}

// ---- sample streams ------------------------------------------------------------------------------------------------
// One path per pixel is in flight inside a render (a pixel's samples run in order).  With the counter-based
// generator a frame's sample range can be cut into N contiguous parts that do not depend on each other; each part is
// an ordinary render into its own partial-sum buffer, issued on its own CUDA stream by a helper context that borrows
// this context's scene, and one k_reduce_finalize on this context's stream adds the parts in order.  The GPU then
// holds N samples of a pixel at once: small frames fill it, and on large frames one part's shading overlaps another
// part's tracing (the two kernels are bound by different units).
void borrow_scene(b200rt_ctx *p, b200rt_ctx *h) {
  for (int i = 0; i < kSceneBufs; ++i) {
    h->d_scene[i] = p->d_scene[i];
    h->d_scene[i].borrowed = true;
  }
  h->scene = p->scene;
  h->n_light = p->n_light;
  h->have_scene = p->have_scene;
  h->ibl_tex = p->ibl_tex; h->ibl_w = p->ibl_w; h->ibl_h = p->ibl_h; h->have_ibl = p->have_ibl;
  h->shared_epoch = p->scene_epoch;
}

// Runs fn(k) for every part k in [0, n) on a host thread of its own: a frame is thousands of small launches, and one
// thread feeding several streams or GPUs would be the bottleneck.  Returns 0, or the code of the first part that
// failed with its index in *failed.
template <class F>
int run_parts(int n, int *failed, F &&fn) {
  std::vector<int> rcs((size_t)n, 0);
#pragma omp parallel for num_threads(n) schedule(static, 1)
  for (int k = 0; k < n; ++k) rcs[(size_t)k] = fn(k);
  for (int k = 0; k < n; ++k)
    if (rcs[(size_t)k]) {
      *failed = k;
      return rcs[(size_t)k];
    }
  return 0;
}

// One k_reduce_finalize on c's stream: out[0, n) = the parts' sums in part order, divided by spp and clamped, or left as
// sums when spp is 0.  It reads float4s when every pointer is 16-byte aligned.
int launch_reduce(b200rt_ctx *c, const PartList &parts, float *out, long long n, float spp) {
  bool aligned = reinterpret_cast<uintptr_t>(out) % 16 == 0;
  for (int i = 0; i < parts.n; ++i) aligned = aligned && reinterpret_cast<uintptr_t>(parts.p[i]) % 16 == 0;
  const int grid = (int)std::min<long long>((n / 4 + 255) / 256 + 1, (long long)c->sm_count * 8);
  k_reduce_finalize<<<grid, 256, 0, c->stream>>>(parts, out, aligned ? n / 4 : 0, n, spp);
  CU(cudaGetLastError());
  return 0;
}

int resolve_streams(const b200rt_opts &o, int width, int height, int s0, int s1) {
  if (o.rng_mode != B200RT_RNG_PHILOX) return 1;   // the reference generator is one serial stream per pixel
  int n = o.sample_streams;
  if (n < 0) {
    const long long npix = (long long)width * height;
    n = npix >= 1000000 ? 3 : (npix >= 200000 ? 4 : 8);
  }
  if (n > 16) n = 16;
  if (n > s1 - s0) n = s1 - s0;
  return n < 1 ? 1 : n;
}

// ad != NULL: an adaptive frame, which runs on one stream (b200rt_render_adaptive has validated ad and opts)
int render_frame(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                 const b200rt_opts *opts, float *d_out, const b200rt_adaptive *ad = nullptr) {
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  if (o.sample_streams < -1 || o.sample_streams > 16)
    return fail(c, B200RT_ERR_INVALID, "bad sample_streams %d (-1 automatic, 0 / 1 off, up to 16)", o.sample_streams);
  int s0 = o.sample_begin, s1 = o.sample_end;
  if (s1 <= 0) { s0 = 0; s1 = spp; }
  const int n = (!ad && width > 0 && height > 0 && spp > 0) ? resolve_streams(o, width, height, s0, s1) : 1;
  if (!c->is_helper) c->frame_trace_cap = 0;
  if (n <= 1 || c->is_helper) return render_impl(c, cam, env, width, height, spp, max_bounce, &o, d_out, ad);
  int rc = check_frame_args(c, cam, width, height, spp, max_bounce, o, true, env);
  if (rc) return rc;
  if (!c->have_ibl) return fail(c, B200RT_ERR_NO_SCENE, "no environment map: call b200rt_set_ibl first");
  CU(cudaSetDevice(c->device));
  while ((int)c->helpers.size() < n - 1) {
    b200rt_ctx *h = nullptr;
    rc = b200rt_create(c->device, &h);
    if (rc) return fail(c, rc, "sample stream context: %s", b200rt_last_error(nullptr));
    h->is_helper = true;
    c->helpers.push_back(h);
  }
  if (!c->ev_fork) {
    CU(cudaEventCreate(&c->ev_fork));
    CU(cudaEventCreate(&c->ev_done));
  }
  const size_t bytes = (size_t)width * height * 3 * sizeof(float);
  if (ensure(c, c->d_part, bytes)) return B200RT_ERR_CUDA;
  CU(cudaEventRecord(c->ev_fork, c->stream));   // the parts start after whatever the caller enqueued before this frame
  const int total = s1 - s0, base = total / n, extra = total % n;
  int bad = 0;
  rc = run_parts(n, &bad, [&](int k) {
    b200rt_ctx *h = k == 0 ? c : c->helpers[(size_t)k - 1];
    b200rt_opts ok = o;
    ok.sample_streams = 1;
    ok.output = B200RT_OUT_SUMS;
    ok.sample_begin = s0 + k * base + (k < extra ? k : extra);
    ok.sample_end = ok.sample_begin + base + (k < extra ? 1 : 0);
    int r = 0;
    if (cudaSetDevice(c->device) != cudaSuccess) r = B200RT_ERR_CUDA;
    float *part = nullptr;
    if (!r && k > 0) {
      if (h->shared_epoch != c->scene_epoch) borrow_scene(c, h);
      if (!h->ev_join && cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) r = B200RT_ERR_CUDA;
      if (!r && cudaStreamWaitEvent(h->stream, c->ev_fork, 0) != cudaSuccess) r = B200RT_ERR_CUDA;
      if (!r) r = ensure(h, h->d_part, bytes);
      part = static_cast<float *>(h->d_part.p);
    } else if (!r) {
      part = static_cast<float *>(c->d_part.p);
    }
    if (!r && cudaMemsetAsync(part, 0, bytes, h->stream) != cudaSuccess) r = B200RT_ERR_CUDA;
    h->frame_trace_cap = n >= 3 ? kStreamTraceCtas : 0;
    if (!r) r = render_impl(h, cam, env, width, height, spp, max_bounce, &ok, part, nullptr);
    if (!r && k > 0 && cudaEventRecord(h->ev_join, h->stream) != cudaSuccess) r = B200RT_ERR_CUDA;
    if (r == B200RT_ERR_CUDA && h->err.empty()) h->err = "CUDA call failed while enqueueing a sample stream";
    return r;
  });
  if (rc) {
    const std::string msg = (bad == 0 ? c : c->helpers[(size_t)bad - 1])->err;
    return fail(c, rc, "sample stream %d: %s", bad, msg.c_str());
  }
  // join on this context's stream, add the parts in order; a whole frame is finalised, a partial range stays sums
  PartList pl;
  pl.n = n;
  pl.p[0] = static_cast<const float *>(c->d_part.p);
  for (int k = 1; k < n; ++k) {
    CU(cudaStreamWaitEvent(c->stream, c->helpers[(size_t)k - 1]->ev_join, 0));
    pl.p[k] = static_cast<const float *>(c->helpers[(size_t)k - 1]->d_part.p);
  }
  rc = launch_reduce(c, pl, d_out, (long long)width * height * 3, o.output == B200RT_OUT_FINAL ? (float)spp : 0.0f);
  if (rc) return rc;
  CU(cudaEventRecord(c->ev_done, c->stream));
  c->streams_used = n;
  c->stats.sample_streams = n;
  c->stats_pending = true;
  return 0;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char *b200rt_version(void) { return "b200rt 0.2 (sm_100a)"; }

int b200rt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void b200rt_default_opts(b200rt_opts *o) {
  memset(o, 0, sizeof *o);
  o->rng_mode = B200RT_RNG_REFERENCE;
  o->traversal = B200RT_TRAVERSAL_FAST;
  o->stack_cap = 20;
  o->output = B200RT_OUT_FINAL;
}

const char *b200rt_last_error(const b200rt_ctx *c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int b200rt_create(int device, b200rt_ctx **out) {
  b200rt_ctx *c = nullptr;
  if (!out) return fail(nullptr, B200RT_ERR_INVALID, "out_ctx is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, B200RT_ERR_CUDA, "no CUDA device available (%s); b200rt has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  if (device < 0 || device >= n) return fail(nullptr, B200RT_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, B200RT_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, B200RT_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library contains sm_100a code only", device,
                prop.major, prop.minor);
  c = new b200rt_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  memset(&c->stats, 0, sizeof c->stats);
  auto bail = [&](const char *what, cudaError_t err) {
    fail(nullptr, B200RT_ERR_CUDA, "%s: %s", what, cudaGetErrorString(err));
    delete c;
    return B200RT_ERR_CUDA;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  c->stream = c->own_stream;
  for (int i = 0; i < 3; ++i)
    if ((e = cudaEventCreate(&c->ev[i])) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaMalloc(&c->d_counters, sizeof(DeviceCounters))) != cudaSuccess) return bail("cudaMalloc", e);
  *out = c;
  return 0;
}

void b200rt_destroy(b200rt_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (b200rt_ctx *h : c->helpers) b200rt_destroy(h);
  c->helpers.clear();
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_done) cudaEventDestroy(c->ev_done);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->d_part.p) cudaFree(c->d_part.p);
  if (c->is_helper) {  // the environment map belongs to the parent
    c->ibl_tex = 0;
    c->ibl_array = nullptr;
  }
  for (DevBuf &b : c->d_scene)
    if (b.p && !b.borrowed) cudaFree(b.p);
  DevBuf *bufs[] = {&c->d_prim_dirk, &c->d_prim_tri, &c->d_out, &c->d_misc, &c->d_tmp_a, &c->d_tmp_b, &c->d_pA, &c->d_pB,
                    &c->d_pC, &c->d_pHit, &c->d_list0, &c->d_list1, &c->d_cnt, &c->d_slots, &c->d_part_count, &c->d_pS,
                    &c->d_pL, &c->d_pR, &c->d_welford, &c->d_ad_spp, &c->d_ad_err, &c->d_dn_tri, &c->d_dn_k,
                    &c->d_gb[0], &c->d_gb[1], &c->d_gb[2], &c->d_dn_col[0], &c->d_dn_col[1]};
  for (DevBuf *b : bufs)
    if (b->p) cudaFree(b->p);
  if (c->h_live) cudaFreeHost(c->h_live);
  for (cudaEvent_t e : c->ev_batch)
    if (e) cudaEventDestroy(e);
  if (c->ibl_tex) cudaDestroyTextureObject(c->ibl_tex);
  if (c->ibl_array) cudaFreeArray(c->ibl_array);
  if (c->d_counters) cudaFree(c->d_counters);
  for (int i = 0; i < 3; ++i)
    if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (cudaEvent_t e : c->kev) cudaEventDestroy(e);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int b200rt_set_materials(b200rt_ctx *c, const float *mat, int64_t n_mat) {
  if (!c) return B200RT_ERR_INVALID;
  if (!mat || n_mat <= 0 || n_mat % 6) return fail(c, B200RT_ERR_INVALID, "material_data must hold 6 floats per material (got %lld)", (long long)n_mat);
  const int nm = (int)(n_mat / 6);
  for (int m = 0; m < nm; ++m) {
    float t = mat[6 * m];
    if (!(t >= 0.0f && t < 4.0f))
      return fail(c, B200RT_ERR_INVALID, "material %d has type %g; the kernel defines types 0..3 only (Raytracing.cl:58-78)", m, (double)t);
  }
  for (int32_t m : c->tri_mat)
    if (m < 0 || m >= nm) return fail(c, B200RT_ERR_INVALID, "a triangle uses material %d but only %d materials were given", m, nm);
  CU(cudaSetDevice(c->device));
  uint64_t h = hash_bytes(mat, (size_t)n_mat * 4, 0x6d617473ull);
  DevBuf &d_mats = c->d_scene[kMats], &d_light = c->d_scene[kLight];
  if (c->n_mats == nm && c->mat_hash != 0 && h == c->mat_hash && d_mats.p) return 0;
  if (ensure(c, d_mats, (size_t)n_mat * 4)) return B200RT_ERR_CUDA;
  CU(cudaMemcpyAsync(d_mats.p, mat, (size_t)n_mat * 4, cudaMemcpyHostToDevice, c->stream));
  // The emitter list of the opt-in light sampling: what FileManager.py:235-240 builds as lightData — the triangles
  // whose material is emissive, in triangle order — derived here from the materials just given, so that it can never
  // be stale after a material edit (the reference's kernel receives lightData and never reads it, Raytracing.cl:163).
  {
    std::vector<int32_t> lights;
    for (size_t t = 0; t < c->tri_mat.size(); ++t)
      if ((int)mat[6 * (size_t)c->tri_mat[t]] == 0) lights.push_back((int32_t)t);
    c->n_light = (int)lights.size();
    if (!lights.empty()) {
      if (ensure(c, d_light, lights.size() * sizeof(int32_t))) return B200RT_ERR_CUDA;
      CU(cudaMemcpy(d_light.p, lights.data(), lights.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
  }
  CU(cudaStreamSynchronize(c->stream));
  c->n_mats = nm;
  c->mat_hash = h;
  ++c->scene_epoch;
  return 0;
}

}  // extern "C"

namespace {

struct SceneArgs {
  const float *vp; int64_t n_vp;
  const float *vn; int64_t n_vn;
  const int32_t *face; int64_t n_face;
  const float *mat; int64_t n_mat;
  const float *bvh; int64_t n_bvh;
};

// shape checks of the reference-layout buffers; the message goes to the context (or to the create-error slot)
int check_scene_args(b200rt_ctx *c, const SceneArgs &a) {
  if (!a.vp || !a.vn || !a.face || !a.mat || !a.bvh) return fail(c, B200RT_ERR_INVALID, "NULL scene buffer");
  if (a.n_vp <= 0 || a.n_vp % 3) return fail(c, B200RT_ERR_INVALID, "vertex_p length %lld is not a positive multiple of 3", (long long)a.n_vp);
  if (a.n_vn <= 0 || a.n_vn % 3) return fail(c, B200RT_ERR_INVALID, "vertex_n length %lld is not a positive multiple of 3", (long long)a.n_vn);
  if (a.n_face <= 0 || a.n_face % 10) return fail(c, B200RT_ERR_INVALID, "face_data length %lld is not a positive multiple of 10", (long long)a.n_face);
  if (a.n_bvh <= 0 || a.n_bvh % 9) return fail(c, B200RT_ERR_INVALID, "BVH length %lld is not a positive multiple of 9", (long long)a.n_bvh);
  if (a.n_bvh / 9 >= (1 << 24)) return fail(c, B200RT_ERR_UNSUPPORTED, "%lld nodes: float32-encoded child indices are exact only below 2^24 (BVH.py:165)", (long long)(a.n_bvh / 9));
  if (a.n_mat <= 0 || a.n_mat % 6) return fail(c, B200RT_ERR_INVALID, "material_data must hold 6 floats per material (got %lld)", (long long)a.n_mat);
  return 0;
}

uint64_t scene_hash_of(const SceneArgs &a) {
  uint64_t h = 0x7363656e65ull;
  h = hash_bytes(a.vp, (size_t)a.n_vp * 4, h);
  h = hash_bytes(a.vn, (size_t)a.n_vn * 4, h);
  h = hash_bytes(a.face, (size_t)a.n_face * 4, h);
  h = hash_bytes(a.bvh, (size_t)a.n_bvh * 4, h);
  return h;
}

bool scene_is_cached(const b200rt_ctx *c, uint64_t h) { return c->have_scene && c->have_scene_cached && h == c->scene_hash; }

// Copies a repacked scene to the context's GPU and, only after every copy has succeeded, commits the fields the
// kernels' launch geometry and margins derive from.  `R` is shared by every GPU of a multi-GPU handle.
int upload_scene(b200rt_ctx *c, const Repacked &R, const SceneArgs &a, uint64_t h) {
  // From here on the context describes no scene until the new one is complete: a caller that catches an error and
  // resubmits the previous scene must not hit the content-hash shortcut with half-replaced buffers.
  c->have_scene = false;
  c->have_scene_cached = false;
  c->scene_hash = 0;
  const int n_tris = R.n_tris;
  DevBuf *B = c->d_scene;
  CU(cudaSetDevice(c->device));
  if (ensure(c, B[kTris], R.tris.size() * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kCtris], R.ctris.size() * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kNormals], R.normals.size() * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kTboxes], R.tboxes.size() * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kFrames], (size_t)n_tris * kFrameVec * sizeof(float4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kNodes], R.nodes.size() * sizeof(uint4))) return B200RT_ERR_CUDA;
  if (ensure(c, B[kBvh9], (size_t)a.n_bvh * 4)) return B200RT_ERR_CUDA;
  if (ensure(c, B[kLeafcnt], R.leaf_count.size() * sizeof(int32_t))) return B200RT_ERR_CUDA;
  CU(cudaMemcpyAsync(B[kLeafcnt].p, R.leaf_count.data(), R.leaf_count.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(B[kTris].p, R.tris.data(), R.tris.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(B[kCtris].p, R.ctris.data(), R.ctris.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(B[kNormals].p, R.normals.data(), R.normals.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(B[kTboxes].p, R.tboxes.data(), R.tboxes.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  if (!R.nodes.empty())
    CU(cudaMemcpyAsync(B[kNodes].p, R.nodes.data(), R.nodes.size() * sizeof(uint4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(B[kBvh9].p, a.bvh, (size_t)a.n_bvh * 4, cudaMemcpyHostToDevice, c->stream));
  k_tri_frames<<<(n_tris + 127) / 128, 128, 0, c->stream>>>(static_cast<const float4 *>(B[kNormals].p), n_tris,
                                                           static_cast<float4 *>(B[kFrames].p));
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(c->stream));
  c->scene = R;
  c->tri_mat = R.tri_mat;
  c->mat_hash = 0;
  c->n_mats = 0;
  int rc = b200rt_set_materials(c, a.mat, a.n_mat);
  if (rc) return rc;
  c->have_scene = true;
  c->have_scene_cached = true;
  c->scene_hash = h;
  ++c->scene_epoch;
  c->stats.repack_ms = (float)(R.ms_tris + R.ms_walk + R.ms_nodes);
  c->stats.ref_stack_need = R.ref_stack_need;
  c->stats.nodes = R.n_nodes9;
  c->stats.triangles = n_tris;
  c->stats.bvh_depth = R.depth;
  return 0;
}

// What every host-output render does: render into the zeroed d_out on the context's stream, enqueue `read_back` (the
// copies to the caller's memory), wait for them and read the counters.
template <class ReadBack>
int render_to_host(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                   const b200rt_opts *opts, const b200rt_adaptive *ad, ReadBack &&read_back) {
  const size_t bytes = (size_t)width * height * 3 * sizeof(float);
  CU(cudaSetDevice(c->device));
  if (ensure(c, c->d_out, bytes)) return B200RT_ERR_CUDA;
  CU(cudaMemsetAsync(c->d_out.p, 0, bytes, c->stream));
  int rc = render_frame(c, cam, env, width, height, spp, max_bounce, opts, static_cast<float *>(c->d_out.p), ad);
  if (!rc) rc = read_back();
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return read_counters(c);
}

// ---- denoising (rt_denoise.cuh) --------------------------------------------------------------------------------------
// Validates the filter's parameters and resolves sigma_position to the scale s_x = sigma_position^2 (b200rt.h).
int check_denoise(b200rt_ctx *c, const b200rt_denoise_params *dn, float *s_x) {
  if (!dn) return fail(c, B200RT_ERR_INVALID, "denoise parameters are NULL");
  if (dn->passes < 1 || dn->passes > kDnMaxPasses)
    return fail(c, B200RT_ERR_INVALID, "denoise passes %d outside [1, %d]", dn->passes, kDnMaxPasses);
  if (!std::isfinite(dn->sigma_color) || !(dn->sigma_color > 0.0f))
    return fail(c, B200RT_ERR_INVALID, "denoise sigma_color %g must be finite and > 0", (double)dn->sigma_color);
  if (!std::isfinite(dn->sigma_normal) || !(dn->sigma_normal > 0.0f))
    return fail(c, B200RT_ERR_INVALID, "denoise sigma_normal %g must be finite and > 0", (double)dn->sigma_normal);
  if (!std::isfinite(dn->sigma_position))
    return fail(c, B200RT_ERR_INVALID, "denoise sigma_position %g must be finite (<= 0: automatic)", (double)dn->sigma_position);
  float sp = dn->sigma_position;
  if (!(sp > 0.0f)) {
    if (!c->have_scene) return fail(c, B200RT_ERR_NO_SCENE, "an automatic sigma_position needs a scene: call b200rt_set_scene first");
    const float *b = c->scene.root_box;
    const float dx = b[3] - b[0], dy = b[4] - b[1], dz = b[5] - b[2];
    sp = 0.01f * std::sqrt((dx * dx + dy * dy) + dz * dz);
    if (!(sp > 0.0f) || !std::isfinite(sp))
      return fail(c, B200RT_ERR_INVALID, "automatic sigma_position is %g (degenerate BVH root box): give one", (double)sp);
  }
  *s_x = sp * sp;
  return 0;
}

// the filter needs the whole finalised frame
int check_denoise_frame(b200rt_ctx *c, const b200rt_opts &o, int spp) {
  if (o.output != B200RT_OUT_FINAL) return fail(c, B200RT_ERR_INVALID, "denoising needs B200RT_OUT_FINAL");
  if (o.sample_end > 0 && (o.sample_begin != 0 || o.sample_end != spp))
    return fail(c, B200RT_ERR_INVALID, "denoising needs the whole sample range [0, spp)");
  if (o.pixel_end > 0) return fail(c, B200RT_ERR_INVALID, "denoising needs the whole frame: no pixel range");
  if (o.tile_row_mod > 1) return fail(c, B200RT_ERR_INVALID, "denoising needs the whole frame: no tile rows");
  return 0;
}

int ensure_denoise_bufs(b200rt_ctx *c, size_t npix) {
  for (DevBuf &b : c->d_gb)
    if (ensure(c, b, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  for (DevBuf &b : c->d_dn_col)
    if (ensure(c, b, npix * sizeof(float4))) return B200RT_ERR_CUDA;
  return 0;
}

GBufferView gbuffer_view(b200rt_ctx *c) {
  return GBufferView{static_cast<float4 *>(c->d_gb[0].p), static_cast<float4 *>(c->d_gb[1].p), static_cast<float4 *>(c->d_gb[2].p)};
}

// k_primary (PARITY: the hit the render's k_primary finds, same traversal and stack cap) + k_gbuffer over the whole frame,
// on c's stream.  d_rgb (may be NULL): the frame's image on the device, packed into d_dn_col[0] for the passes.
int launch_gbuffer(b200rt_ctx *c, const float *cam, int width, int height, const b200rt_opts &o, const float *d_rgb) {
  const size_t npix = (size_t)width * height;
  if (ensure(c, c->d_dn_tri, npix * sizeof(int))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_dn_k, npix * sizeof(float))) return B200RT_ERR_CUDA;
  if (ensure_denoise_bufs(c, npix)) return B200RT_ERR_CUDA;
  b200rt_opts og = o;
  og.sample_begin = og.sample_end = 0;
  og.pixel_begin = og.pixel_end = 0;
  og.tile_row_mod = og.tile_row_rem = 0;
  FrameParams F;
  frame_setup(c, cam, nullptr, width, height, 1, 0, og, &F);
  KernelArgs A;
  fill_args(c, F, og, nullptr, &A);
  int *tri = static_cast<int *>(c->d_dn_tri.p);
  float *k = static_cast<float *>(c->d_dn_k.p);
  int rc = launch_primary(c, A, effective_traversal(c, og), use_smem_scene(c), true, og.collect_stats != 0, tri, k);
  if (rc) return rc;
  k_gbuffer<<<(unsigned)((npix + kBlock - 1) / kBlock), kBlock, 0, c->stream>>>(A, tri, k, gbuffer_view(c), d_rgb,
                                                                                 static_cast<float4 *>(c->d_dn_col[0].p));
  CU(cudaGetLastError());
  c->stats.kernel_launches++;
  return 0;
}

// The passes over the G-buffer and input colour (d_dn_col[0]) already on the device; the image goes to d_out.
int launch_atrous(b200rt_ctx *c, int width, int height, const b200rt_denoise_params &dn, float s_x, float *d_out) {
  const dim3 block(kDnBlockX, kDnBlockY);
  const dim3 grid((unsigned)((width + kDnBlockX - 1) / kDnBlockX), (unsigned)((height + kDnBlockY - 1) / kDnBlockY));
  if (grid.y > 65535u) return fail(c, B200RT_ERR_UNSUPPORTED, "denoising a frame of %d rows: at most %d", height, 65535 * kDnBlockY);
  const GBufferView G = gbuffer_view(c);
  float4 *col[2] = {static_cast<float4 *>(c->d_dn_col[0].p), static_cast<float4 *>(c->d_dn_col[1].p)};
  AtrousArgs P;
  P.gn = G.gn; P.gx = G.gx; P.ga = G.ga;
  P.out = d_out;
  P.width = width;
  P.height = height;
  P.s_n = dn.sigma_normal * dn.sigma_normal;
  P.s_x = s_x;
  for (int l = 0; l < dn.passes; ++l) {
    P.cin = col[l & 1];
    P.cout = col[(l + 1) & 1];
    P.step = 1 << l;
    P.s_c = (dn.sigma_color * dn.sigma_color) * std::ldexp(1.0f, -2 * l);   // sigma_color halves every pass
    const bool first = l == 0, last = l == dn.passes - 1;
    auto k = first ? (last ? k_atrous<true, true> : k_atrous<true, false>) : (last ? k_atrous<false, true> : k_atrous<false, false>);
    k<<<grid, block, 0, c->stream>>>(P);
    CU(cudaGetLastError());
    c->stats.kernel_launches++;
  }
  return 0;
}

// G-buffer + passes over the image d_img (3 floats per pixel, on c's GPU), in place, on c's stream
int denoise_frame(b200rt_ctx *c, const float *cam, int width, int height, const b200rt_opts &o, const b200rt_denoise_params &dn,
                  float s_x, float *d_img) {
  int rc = launch_gbuffer(c, cam, width, height, o, d_img);
  if (rc) return rc;
  return launch_atrous(c, width, height, dn, s_x, d_img);
}

}  // namespace

extern "C" {

int b200rt_set_scene(b200rt_ctx *c, const float *vp, int64_t n_vp, const float *vn, int64_t n_vn, const float *vuv,
                     int64_t n_vuv, const int32_t *face, int64_t n_face, const float *mat, int64_t n_mat,
                     const int32_t *light, int64_t n_light, const float *bvh, int64_t n_bvh) {
  (void)vuv; (void)n_vuv; (void)light; (void)n_light;  // fetched / passed but never used by the kernel (MathLib.cl:217, Raytracing.cl:163)
  if (!c) return B200RT_ERR_INVALID;
  auto t0 = std::chrono::steady_clock::now();
  const SceneArgs a{vp, n_vp, vn, n_vn, face, n_face, mat, n_mat, bvh, n_bvh};
  int rc = check_scene_args(c, a);
  if (rc) return rc;
  const uint64_t h = scene_hash_of(a);
  if (scene_is_cached(c, h)) {  // geometry unchanged (the UI rebuilds identical arrays per render, UI.py:98)
    rc = b200rt_set_materials(c, mat, n_mat);
  } else {
    Repacked R;
    std::string msg;
    rc = repack_scene(vp, n_vp, vn, n_vn, face, n_face, n_mat / 6, bvh, n_bvh, &R, &msg, own_cull_tree());
    if (rc) {
      c->have_scene = false;   // as before an upload: the context describes no scene after a rejected one
      c->have_scene_cached = false;
      c->scene_hash = 0;
      return fail(c, rc, "%s", msg.c_str());
    }
    rc = upload_scene(c, R, a, h);
  }
  c->stats.upload_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int b200rt_set_ibl(b200rt_ctx *c, const uint8_t *rgba, int width, int height) {
  if (!c) return B200RT_ERR_INVALID;
  if (!rgba || width <= 0 || height <= 0) return fail(c, B200RT_ERR_INVALID, "bad environment map (%p, %d x %d)", (const void *)rgba, width, height);
  if (width > 131072 || height > 65536) return fail(c, B200RT_ERR_UNSUPPORTED, "environment map %d x %d exceeds the 2-D texture limits", width, height);
  auto t0 = std::chrono::steady_clock::now();
  uint64_t h = hash_bytes(rgba, (size_t)width * height * 4, 0x69626cull);
  if (c->have_ibl && c->ibl_hash != 0 && h == c->ibl_hash && width == c->ibl_w && height == c->ibl_h) return 0;
  CU(cudaSetDevice(c->device));
  if (c->ibl_array && c->ibl_tex && width == c->ibl_w && height == c->ibl_h) {
    // same shape: refill the existing array (allocating / freeing device memory synchronises the whole device,
    // peers and collectives included)
    c->have_ibl = false;
    CU(cudaMemcpy2DToArrayAsync(c->ibl_array, 0, 0, rgba, (size_t)width * 4, (size_t)width * 4, (size_t)height,
                                cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  } else {
    CU(cudaStreamSynchronize(c->stream));
    if (c->ibl_tex) { cudaDestroyTextureObject(c->ibl_tex); c->ibl_tex = 0; }
    if (c->ibl_array) { cudaFreeArray(c->ibl_array); c->ibl_array = nullptr; }
    c->have_ibl = false;
    cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
    CU(cudaMallocArray(&c->ibl_array, &fmt, (size_t)width, (size_t)height));
    CU(cudaMemcpy2DToArrayAsync(c->ibl_array, 0, 0, rgba, (size_t)width * 4, (size_t)width * 4, (size_t)height,
                                cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    cudaResourceDesc res;
    memset(&res, 0, sizeof res);
    res.resType = cudaResourceTypeArray;
    res.res.array.array = c->ibl_array;
    cudaTextureDesc td;
    memset(&td, 0, sizeof td);
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;  // CLK_ADDRESS_CLAMP_TO_EDGE (Raytracing.cl:179)
    td.filterMode = cudaFilterModePoint;                          // integer coordinates address single texels
    td.readMode = cudaReadModeElementType;                        // raw bytes; the kernel divides by 255 itself
    td.normalizedCoords = 0;                                      // CLK_NORMALIZED_COORDS_FALSE
    CU(cudaCreateTextureObject(&c->ibl_tex, &res, &td, nullptr));
  }
  c->ibl_w = width;
  c->ibl_h = height;
  c->ibl_hash = h;
  ++c->scene_epoch;
  c->have_ibl = true;
  c->stats.upload_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return 0;
}

int b200rt_render_device(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp,
                         int max_bounce, const b200rt_opts *opts, float *d_out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!d_out) return fail(c, B200RT_ERR_INVALID, "d_out_rgb is NULL");
  return render_frame(c, cam, env, width, height, spp, max_bounce, opts, d_out);
}

int b200rt_render(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                  const b200rt_opts *opts, float *out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!out) return fail(c, B200RT_ERR_INVALID, "out_rgb is NULL");
  if (width <= 0 || height <= 0) return fail(c, B200RT_ERR_INVALID, "bad frame size %d x %d", width, height);
  return render_to_host(c, cam, env, width, height, spp, max_bounce, opts, nullptr, [&] {
    CU(cudaMemcpyAsync(out, c->d_out.p, (size_t)width * height * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));  // blocking read-back, KernelLauncher.py:78
    return 0;
  });
}

int b200rt_render_adaptive(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp,
                           int max_bounce, const b200rt_opts *opts, const b200rt_adaptive *ad, float *out,
                           int32_t *out_spp, float *out_stderr) {
  if (!c) return B200RT_ERR_INVALID;
  if (!out) return fail(c, B200RT_ERR_INVALID, "out_rgb is NULL");
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  int rc = check_frame_args(c, cam, width, height, spp, max_bounce, o, true, env);
  if (rc) return rc;
  if (!ad) return fail(c, B200RT_ERR_INVALID, "adaptive parameters are NULL");
  if (ad->min_spp < 2 || ad->min_spp > spp)
    return fail(c, B200RT_ERR_INVALID, "adaptive min_spp %d outside [2, spp = %d]", ad->min_spp, spp);
  if (ad->check_every < 1) return fail(c, B200RT_ERR_INVALID, "adaptive check_every %d must be >= 1", ad->check_every);
  if (!std::isfinite(ad->rel_error) || !(ad->rel_error >= 0.0f))
    return fail(c, B200RT_ERR_INVALID, "adaptive rel_error %g must be finite and >= 0", (double)ad->rel_error);
  if (!std::isfinite(ad->floor) || !(ad->floor > 0.0f))
    return fail(c, B200RT_ERR_INVALID, "adaptive floor %g must be finite and > 0", (double)ad->floor);
  if (o.output != B200RT_OUT_FINAL) return fail(c, B200RT_ERR_INVALID, "adaptive sampling needs B200RT_OUT_FINAL");
  if (o.sample_end > 0 && (o.sample_begin != 0 || o.sample_end != spp))
    return fail(c, B200RT_ERR_INVALID, "adaptive sampling needs the whole sample range [0, spp)");
  // the stopping rule needs the pixel's samples as one serial sequence; -1 (automatic) resolves to that one stream
  if (o.sample_streams < -1 || o.sample_streams > 1)
    return fail(c, B200RT_ERR_INVALID, "adaptive sampling runs one sample stream (sample_streams -1, 0 or 1, got %d)",
                o.sample_streams);
  const size_t npix = (size_t)width * height;
  return render_to_host(c, cam, env, width, height, spp, max_bounce, &o, ad, [&] {
    CU(cudaMemcpyAsync(out, c->d_out.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (out_spp) CU(cudaMemcpyAsync(out_spp, c->d_ad_spp.p, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (out_stderr) CU(cudaMemcpyAsync(out_stderr, c->d_ad_err.p, npix * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    return 0;
  });
}

int b200rt_render_denoised(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp,
                           int max_bounce, const b200rt_opts *opts, const b200rt_denoise_params *dn, float *out,
                           float *out_noisy) {
  if (!c) return B200RT_ERR_INVALID;
  if (!out) return fail(c, B200RT_ERR_INVALID, "out_rgb is NULL");
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  int rc = check_frame_args(c, cam, width, height, spp, max_bounce, o, true, env);
  if (!rc) rc = check_denoise_frame(c, o, spp);
  float s_x = 0.0f;
  if (!rc) rc = check_denoise(c, dn, &s_x);
  if (rc) return rc;
  const size_t bytes = (size_t)width * height * 3 * sizeof(float);
  return render_to_host(c, cam, env, width, height, spp, max_bounce, &o, nullptr, [&] {
    float *img = static_cast<float *>(c->d_out.p);
    if (out_noisy) CU(cudaMemcpyAsync(out_noisy, img, bytes, cudaMemcpyDeviceToHost, c->stream));
    const int r = denoise_frame(c, cam, width, height, o, *dn, s_x, img);
    if (r) return r;
    CU(cudaMemcpyAsync(out, img, bytes, cudaMemcpyDeviceToHost, c->stream));
    return 0;
  });
}

int b200rt_gbuffer(b200rt_ctx *c, const float *cam, int width, int height, const b200rt_opts *opts, float *albedo,
                   float *normal, float *position, int32_t *kind) {
  if (!c) return B200RT_ERR_INVALID;
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  int rc = check_frame_args(c, cam, width, height, 1, 0, o, false, nullptr);
  if (!rc && (o.pixel_end > 0 || o.tile_row_mod > 1))
    rc = fail(c, B200RT_ERR_INVALID, "the G-buffer covers the whole frame: no pixel range or tile rows");
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)width * height;
  c->stats.kernel_launches = 0;
  c->streams_used = 1;
  CU(cudaMemsetAsync(c->d_counters, 0, sizeof(DeviceCounters), c->stream));
  CU(cudaEventRecord(c->ev[0], c->stream));
  rc = launch_gbuffer(c, cam, width, height, o, nullptr);
  if (rc) return rc;
  CU(cudaEventRecord(c->ev[1], c->stream));
  CU(cudaEventRecord(c->ev[2], c->stream));
  // float4 records -> 3 floats per pixel (a strided copy); kind travels as the float .w of the normal record
  float *dst[3] = {normal, position, albedo};
  for (int r = 0; r < 3; ++r)
    if (dst[r]) CU(cudaMemcpy2DAsync(dst[r], 3 * sizeof(float), c->d_gb[r].p, sizeof(float4), 3 * sizeof(float), npix,
                                     cudaMemcpyDeviceToHost, c->stream));
  std::vector<float> kind_f(kind ? npix : 0);
  if (kind) CU(cudaMemcpy2DAsync(kind_f.data(), sizeof(float), static_cast<const float *>(c->d_gb[0].p) + 3, sizeof(float4),
                                 sizeof(float), npix, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i < kind_f.size(); ++i) kind[i] = (int32_t)kind_f[i];
  return read_counters(c);
}

int b200rt_denoise(b200rt_ctx *c, const float *rgb, const float *albedo, const float *normal, const float *position,
                   const int32_t *kind, int width, int height, const b200rt_denoise_params *dn, float *out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!rgb || !albedo || !normal || !position || !kind || !out) return fail(c, B200RT_ERR_INVALID, "NULL denoise buffer");
  if (width <= 0 || height <= 0 || (long long)width * height > 0x7fffffffLL / 4)
    return fail(c, B200RT_ERR_INVALID, "bad frame size %d x %d", width, height);
  float s_x = 0.0f;
  int rc = check_denoise(c, dn, &s_x);
  if (rc) return rc;
  const size_t npix = (size_t)width * height;
  for (size_t i = 0; i < npix; ++i)
    if (kind[i] < -1 || kind[i] > 1) return fail(c, B200RT_ERR_INVALID, "kind[%zu] = %d is not -1, 0 or 1", i, (int)kind[i]);
  // host records in the layout of GBufferView and the passes' colour buffer
  std::vector<float4> rec[4];
  for (auto &r : rec) r.resize(npix);
  for (size_t i = 0; i < npix; ++i) {
    const size_t e = 3 * i;
    rec[0][i] = make_float4(normal[e], normal[e + 1], normal[e + 2], (float)kind[i]);
    rec[1][i] = make_float4(position[e], position[e + 1], position[e + 2], 0.0f);
    rec[2][i] = make_float4(albedo[e], albedo[e + 1], albedo[e + 2], 0.0f);
    rec[3][i] = make_float4(rgb[e], rgb[e + 1], rgb[e + 2], 0.0f);
  }
  CU(cudaSetDevice(c->device));
  if (ensure_denoise_bufs(c, npix)) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_misc, npix * 3 * sizeof(float))) return B200RT_ERR_CUDA;
  for (int r = 0; r < 3; ++r)
    CU(cudaMemcpyAsync(c->d_gb[r].p, rec[r].data(), npix * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_dn_col[0].p, rec[3].data(), npix * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  c->stats.kernel_launches = 0;
  rc = launch_atrous(c, width, height, *dn, s_x, static_cast<float *>(c->d_misc.p));
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, c->d_misc.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int b200rt_render_rgb8(b200rt_ctx *c, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                       const b200rt_opts *opts, uint8_t *out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!out) return fail(c, B200RT_ERR_INVALID, "out_rgb8 is NULL");
  if (width <= 0 || height <= 0) return fail(c, B200RT_ERR_INVALID, "bad frame size %d x %d", width, height);
  if (opts && opts->output != B200RT_OUT_FINAL) return fail(c, B200RT_ERR_INVALID, "8-bit output needs B200RT_OUT_FINAL");
  const size_t n = (size_t)width * height * 3;
  CU(cudaSetDevice(c->device));
  if (ensure(c, c->d_tmp_a, n)) return B200RT_ERR_CUDA;
  return render_to_host(c, cam, env, width, height, spp, max_bounce, opts, nullptr, [&] {
    int grid = (int)std::min<long long>(((long long)n + 255) / 256, (long long)c->sm_count * 16);
    k_quantize8<<<grid, 256, 0, c->stream>>>(static_cast<const float *>(c->d_out.p), static_cast<uint8_t *>(c->d_tmp_a.p), (long long)n);
    CU(cudaGetLastError());
    c->stats.kernel_launches++;
    CU(cudaMemcpyAsync(out, c->d_tmp_a.p, n, cudaMemcpyDeviceToHost, c->stream));
    return 0;
  });
}

int b200rt_sync(b200rt_ctx *c) {
  if (!c) return B200RT_ERR_INVALID;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->stats_pending) return read_counters(c);
  return 0;
}

int b200rt_set_stream(b200rt_ctx *c, void *cuda_stream) {
  if (!c) return B200RT_ERR_INVALID;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->stats_pending) read_counters(c);
  c->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->own_stream;
  return 0;
}

int b200rt_invalidate(b200rt_ctx *c) {
  if (!c) return B200RT_ERR_INVALID;
  c->scene_hash = 0;
  c->mat_hash = 0;
  c->ibl_hash = 0;
  c->have_scene_cached = false;
  return 0;
}

int b200rt_finalize_device(b200rt_ctx *c, const float *d_sums, float *d_out, int64_t n_pixels, int spp) {
  if (!c) return B200RT_ERR_INVALID;
  if (!d_sums || !d_out || n_pixels <= 0 || spp <= 0) return fail(c, B200RT_ERR_INVALID, "bad finalize arguments");
  CU(cudaSetDevice(c->device));
  PartList pl;
  pl.n = 1;
  pl.p[0] = d_sums;
  return launch_reduce(c, pl, d_out, (long long)n_pixels * 3, (float)spp);
}

int b200rt_reduce_finalize_device(b200rt_ctx *c, const float *const *d_parts, int n_parts, float *d_out,
                                  int64_t n_pixels, int spp) {
  if (!c) return B200RT_ERR_INVALID;
  if (!d_parts || n_parts < 1 || n_parts > 16 || !d_out || n_pixels <= 0 || spp <= 0)
    return fail(c, B200RT_ERR_INVALID, "bad reduce_finalize arguments (1..16 parts)");
  CU(cudaSetDevice(c->device));
  PartList pl;
  pl.n = n_parts;
  for (int i = 0; i < n_parts; ++i) {
    if (!d_parts[i]) return fail(c, B200RT_ERR_INVALID, "part %d is NULL", i);
    pl.p[i] = d_parts[i];
  }
  return launch_reduce(c, pl, d_out, (long long)n_pixels * 3, (float)spp);
}

int b200rt_primary_hits(b200rt_ctx *c, const float *cam, int width, int height, const b200rt_opts *opts,
                        int32_t *tri_out, float *k_out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!tri_out || !k_out) return fail(c, B200RT_ERR_INVALID, "NULL output");
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  int rc = check_frame_args(c, cam, width, height, 1, 0, o, false, nullptr);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)width * height;
  if (ensure(c, c->d_tmp_a, npix * sizeof(int))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_tmp_b, npix * sizeof(float))) return B200RT_ERR_CUDA;
  FrameParams F;
  frame_setup(c, cam, nullptr, width, height, 1, 0, o, &F);
  KernelArgs A;
  fill_args(c, F, o, nullptr, &A);
  c->stats.kernel_launches = 0;
  CU(cudaMemsetAsync(c->d_tmp_a.p, 0xff, npix * sizeof(int), c->stream));
  CU(cudaMemsetAsync(c->d_tmp_b.p, 0, npix * sizeof(float), c->stream));
  CU(cudaMemsetAsync(c->d_counters, 0, sizeof(DeviceCounters), c->stream));
  CU(cudaEventRecord(c->ev[0], c->stream));
  rc = launch_primary(c, A, effective_traversal(c, o), use_smem_scene(c), true, o.collect_stats != 0, static_cast<int *>(c->d_tmp_a.p),
                      static_cast<float *>(c->d_tmp_b.p));
  if (rc) return rc;
  CU(cudaEventRecord(c->ev[1], c->stream));
  CU(cudaEventRecord(c->ev[2], c->stream));
  CU(cudaMemcpyAsync(tri_out, c->d_tmp_a.p, npix * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(k_out, c->d_tmp_b.p, npix * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return read_counters(c);
}

int b200rt_trace_rays(b200rt_ctx *c, const float *rays, int64_t n, const b200rt_opts *opts, int32_t *tri_out, float *k_out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!rays || !tri_out || !k_out || n <= 0) return fail(c, B200RT_ERR_INVALID, "bad trace_rays arguments");
  if (!c->have_scene) return fail(c, B200RT_ERR_NO_SCENE, "no scene: call b200rt_set_scene first");
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  if (o.traversal < 0 || o.traversal > 2) return fail(c, B200RT_ERR_INVALID, "bad traversal %d", o.traversal);
  CU(cudaSetDevice(c->device));
  if (ensure(c, c->d_misc, (size_t)n * 6 * sizeof(float))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_tmp_a, (size_t)n * sizeof(int))) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_tmp_b, (size_t)n * sizeof(float))) return B200RT_ERR_CUDA;
  CU(cudaMemcpyAsync(c->d_misc.p, rays, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(c->d_counters, 0, sizeof(DeviceCounters), c->stream));
  FrameParams F;
  memset(&F, 0, sizeof F);
  KernelArgs A;
  fill_args(c, F, o, nullptr, &A);
  c->stats.kernel_launches = 0;
  const float *dr = static_cast<const float *>(c->d_misc.p);
  int *dt = static_cast<int *>(c->d_tmp_a.p);
  float *dk = static_cast<float *>(c->d_tmp_b.p);
  CU(cudaEventRecord(c->ev[0], c->stream));
  CU(cudaEventRecord(c->ev[1], c->stream));
  int rc = with_variant(c, effective_traversal(c, o), use_smem_scene(c), o.collect_stats != 0, [&](auto t, auto s, auto st) {
    return launch_trace_t<decltype(t)::value, decltype(s)::value, decltype(st)::value>(c, A, dr, n, dt, dk);
  });
  if (rc) return rc;
  CU(cudaEventRecord(c->ev[2], c->stream));
  CU(cudaMemcpyAsync(tri_out, dt, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(k_out, dk, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  rc = read_counters(c);
  c->stats.rays = (uint64_t)n;
  return rc;
}

int b200rt_img_processing(b200rt_ctx *c, const float *src, float *dst, int64_t n, int64_t global) {
  if (!c) return B200RT_ERR_INVALID;
  if (!src || !dst || global <= 0 || n < 0) return fail(c, B200RT_ERR_INVALID, "bad img_processing arguments");
  CU(cudaSetDevice(c->device));
  size_t bytes = (size_t)global * sizeof(float);
  if (ensure(c, c->d_tmp_a, bytes)) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_tmp_b, bytes)) return B200RT_ERR_CUDA;
  CU(cudaMemcpyAsync(c->d_tmp_a.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
  // work-items with i >= n leave dst untouched: start from the caller's dst contents
  CU(cudaMemcpyAsync(c->d_tmp_b.p, dst, bytes, cudaMemcpyHostToDevice, c->stream));
  int grid = (int)std::min<long long>(((long long)global + 255) / 256, (long long)c->sm_count * 16);
  k_img_processing<<<grid, 256, 0, c->stream>>>(static_cast<const float *>(c->d_tmp_a.p), static_cast<float *>(c->d_tmp_b.p),
                                                 (long long)n, (long long)global);
  CU(cudaGetLastError());
  c->stats.kernel_launches = 1;
  CU(cudaMemcpyAsync(dst, c->d_tmp_b.p, bytes, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int b200rt_get_stats(const b200rt_ctx *c, b200rt_stats *s) {
  if (!c || !s) return B200RT_ERR_INVALID;
  if (c->stats_pending) {
    int rc = b200rt_sync(const_cast<b200rt_ctx *>(c));
    if (rc) return rc;
  }
  *s = c->stats;
  return 0;
}

int b200rt_math_probe(b200rt_ctx *c, int fn, const float *a, const float *b, int64_t n, float *out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!a || !out || n <= 0 || fn < 0 || fn > 16) return fail(c, B200RT_ERR_INVALID, "bad math_probe arguments");
  CU(cudaSetDevice(c->device));
  size_t bytes = (size_t)n * sizeof(float);
  if (ensure(c, c->d_tmp_a, bytes)) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_tmp_b, bytes)) return B200RT_ERR_CUDA;
  if (ensure(c, c->d_misc, bytes)) return B200RT_ERR_CUDA;
  CU(cudaMemcpyAsync(c->d_tmp_a.p, a, bytes, cudaMemcpyHostToDevice, c->stream));
  if (b) CU(cudaMemcpyAsync(c->d_tmp_b.p, b, bytes, cudaMemcpyHostToDevice, c->stream));
  else CU(cudaMemsetAsync(c->d_tmp_b.p, 0, bytes, c->stream));
  k_math_probe<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(fn, static_cast<const float *>(c->d_tmp_a.p),
                                                                    static_cast<const float *>(c->d_tmp_b.p), (long long)n,
                                                                    static_cast<float *>(c->d_misc.p));
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, c->d_misc.p, bytes, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int b200rt_philox_probe(b200rt_ctx *c, const uint32_t ctr[4], uint32_t key0, uint32_t key1, uint32_t out[4]) {
  if (!c) return B200RT_ERR_INVALID;
  if (!ctr || !out) return fail(c, B200RT_ERR_INVALID, "NULL argument");
  CU(cudaSetDevice(c->device));
  if (ensure(c, c->d_misc, 16)) return B200RT_ERR_CUDA;
  k_philox_probe<<<1, 1, 0, c->stream>>>(ctr[0], ctr[1], ctr[2], ctr[3], key0, key1, static_cast<uint32_t *>(c->d_misc.p));
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, c->d_misc.p, 16, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int b200rt_alloc(b200rt_ctx *c, int64_t bytes, void **d_ptr_out) {
  if (!c) return B200RT_ERR_INVALID;
  if (bytes <= 0 || !d_ptr_out) return fail(c, B200RT_ERR_INVALID, "bad alloc arguments");
  CU(cudaSetDevice(c->device));
  CU(cudaMalloc(d_ptr_out, (size_t)bytes));
  CU(cudaMemsetAsync(*d_ptr_out, 0, (size_t)bytes, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int b200rt_free(b200rt_ctx *c, void *d_ptr) {
  if (!c) return B200RT_ERR_INVALID;
  CU(cudaSetDevice(c->device));
  CU(cudaFree(d_ptr));
  return 0;
}

int b200rt_ipc_export(b200rt_ctx *c, const void *d_ptr, uint8_t handle_out[64]) {
  if (!c) return B200RT_ERR_INVALID;
  if (!d_ptr || !handle_out) return fail(c, B200RT_ERR_INVALID, "NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CU(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, const_cast<void *>(d_ptr)));
  memcpy(handle_out, &h, 64);
  return 0;
}

int b200rt_ipc_open(b200rt_ctx *c, const uint8_t handle[64], void **d_ptr_out) {
  if (!c) return B200RT_ERR_INVALID;
  if (!handle || !d_ptr_out) return fail(c, B200RT_ERR_INVALID, "NULL argument");
  CU(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CU(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

int b200rt_ipc_close(b200rt_ctx *c, void *d_ptr) {
  if (!c) return B200RT_ERR_INVALID;
  CU(cudaSetDevice(c->device));
  CU(cudaIpcCloseMemHandle(d_ptr));
  return 0;
}

}  // extern "C"

// ================================================================================================
// Multi-GPU handle: one host process, one context + stream per GPU, NVLink peer reads for the reduce
// ================================================================================================
// SURVEY.md §8b/§8e: the frame is divided among the GPUs of one NVSwitch box — by contiguous sample ranges with the
// counter-based generator, by interleaved rows of 8x4-pixel tiles with the reference's serial per-pixel generator —
// every GPU renders raw per-pixel sums into its own buffer, and ONE kernel on the first GPU reads all of them through
// peer mappings (NVLink loads), sums in GPU order, divides by spp and clamps (k_reduce_finalize).  Kernel launches
// are issued by one host thread per GPU: a frame is thousands of small launches, and a single thread feeding eight
// GPUs would be the bottleneck.
struct b200rt_multi {
  std::vector<b200rt_ctx *> ctx;
  std::vector<cudaEvent_t> done;   // per GPU: its partial sums are complete
  std::vector<int> peer_ok;        // GPU 0 can read GPU i's memory directly
  std::vector<DevBuf> staging;     // on GPU 0, for GPUs it cannot read directly
  DevBuf d_final;                  // on GPU 0
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;  // on GPU 0's stream, around wait + reduce
  std::string err;
  b200rt_stats stats;
};

namespace {

int mfail(b200rt_multi *m, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (m) m->err = buf; else g_create_error = buf;
  return code;
}

#define MCU(call)                                                                                    \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) return mfail(m, B200RT_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

// what GPU `r` of `n` renders (ensem3a_openclraytracer_b200/multigpu.py::rank_work is the same rule)
void multi_share(int r, int n, int spp, int rng_mode, b200rt_opts *o) {
  o->output = B200RT_OUT_SUMS;
  if (rng_mode == B200RT_RNG_PHILOX) {
    const int base = spp / n, extra = spp % n;
    const int s0 = r * base + (r < extra ? r : extra);
    o->sample_begin = s0;
    o->sample_end = s0 + base + (r < extra ? 1 : 0);
    o->tile_row_mod = 0;
    o->tile_row_rem = 0;
  } else {
    o->sample_begin = 0;
    o->sample_end = spp;
    o->tile_row_mod = n > 1 ? n : 0;
    o->tile_row_rem = n > 1 ? r : 0;
  }
}

}  // namespace

extern "C" {

const char *b200rt_multi_last_error(const b200rt_multi *m) { return m ? m->err.c_str() : g_create_error.c_str(); }

void b200rt_multi_destroy(b200rt_multi *m) {
  if (!m) return;
  if (!m->ctx.empty() && m->ctx[0]) {
    cudaSetDevice(m->ctx[0]->device);
    cudaStreamSynchronize(m->ctx[0]->stream);
    for (DevBuf &b : m->staging)
      if (b.p) cudaFree(b.p);
    if (m->d_final.p) cudaFree(m->d_final.p);
    if (m->ev_begin) cudaEventDestroy(m->ev_begin);
    if (m->ev_end) cudaEventDestroy(m->ev_end);
  }
  for (size_t i = 0; i < m->ctx.size(); ++i) {
    if (!m->ctx[i]) continue;
    if (i < m->done.size() && m->done[i]) {
      cudaSetDevice(m->ctx[i]->device);
      cudaEventDestroy(m->done[i]);
    }
    b200rt_destroy(m->ctx[i]);
  }
  delete m;
}

int b200rt_multi_create(const int *devices, int n_devices, b200rt_multi **out) {
  b200rt_multi *m = nullptr;
  if (!out) return mfail(nullptr, B200RT_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!devices || n_devices < 1 || n_devices > 16) return mfail(nullptr, B200RT_ERR_INVALID, "1..16 devices expected (got %d)", n_devices);
  // A device may be listed several times: every entry gets its own context, buffers and stream, so a frame too small
  // to fill one GPU (one path per pixel in flight) runs as several concurrent sample-range renders on it.
  m = new b200rt_multi();
  memset(&m->stats, 0, sizeof m->stats);
  m->ctx.assign((size_t)n_devices, nullptr);
  m->done.assign((size_t)n_devices, nullptr);
  m->peer_ok.assign((size_t)n_devices, 1);
  m->staging.resize((size_t)n_devices);
  for (int i = 0; i < n_devices; ++i) {
    int rc = b200rt_create(devices[i], &m->ctx[i]);   // leaves its message in the create-error slot
    if (rc) { b200rt_multi_destroy(m); return rc; }
    cudaError_t e = cudaEventCreateWithFlags(&m->done[i], cudaEventDisableTiming);
    if (e != cudaSuccess) { mfail(nullptr, B200RT_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e)); b200rt_multi_destroy(m); return B200RT_ERR_CUDA; }
  }
  cudaSetDevice(devices[0]);
  for (int i = 1; i < n_devices; ++i) {
    if (devices[i] == devices[0]) continue;  // the same GPU: plain loads
    int can = 0;
    cudaDeviceCanAccessPeer(&can, devices[0], devices[i]);
    if (can) {
      cudaError_t e = cudaDeviceEnablePeerAccess(devices[i], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
      can = (e == cudaSuccess);
      if (!can) cudaGetLastError();
    }
    m->peer_ok[i] = can;
  }
  if (cudaEventCreate(&m->ev_begin) != cudaSuccess || cudaEventCreate(&m->ev_end) != cudaSuccess) {
    mfail(nullptr, B200RT_ERR_CUDA, "cudaEventCreate failed");
    b200rt_multi_destroy(m);
    return B200RT_ERR_CUDA;
  }
  *out = m;
  return 0;
}

int b200rt_multi_device_count(const b200rt_multi *m) { return m ? (int)m->ctx.size() : 0; }

b200rt_ctx *b200rt_multi_context(b200rt_multi *m, int index) {
  if (!m || index < 0 || index >= (int)m->ctx.size()) return nullptr;
  return m->ctx[index];
}

int b200rt_multi_set_scene(b200rt_multi *m, const float *vp, int64_t n_vp, const float *vn, int64_t n_vn, const float *vuv,
                           int64_t n_vuv, const int32_t *face, int64_t n_face, const float *mat, int64_t n_mat,
                           const int32_t *light, int64_t n_light, const float *bvh, int64_t n_bvh) {
  (void)vuv; (void)n_vuv; (void)light; (void)n_light;
  if (!m) return B200RT_ERR_INVALID;
  auto t0 = std::chrono::steady_clock::now();
  const SceneArgs a{vp, n_vp, vn, n_vn, face, n_face, mat, n_mat, bvh, n_bvh};
  int rc = check_scene_args(m->ctx[0], a);
  if (rc) { m->err = m->ctx[0]->err; return rc; }
  const uint64_t h = scene_hash_of(a);
  bool all_cached = true;
  for (b200rt_ctx *c : m->ctx) all_cached = all_cached && scene_is_cached(c, h);
  Repacked R;
  if (!all_cached) {  // validated and repacked once, uploaded to every GPU
    std::string msg;
    rc = repack_scene(vp, n_vp, vn, n_vn, face, n_face, n_mat / 6, bvh, n_bvh, &R, &msg, own_cull_tree());
    if (rc) {
      for (b200rt_ctx *c : m->ctx) { c->have_scene = false; c->have_scene_cached = false; c->scene_hash = 0; }
      return mfail(m, rc, "%s", msg.c_str());
    }
  }
  int bad = 0;
  rc = run_parts((int)m->ctx.size(), &bad, [&](int i) {
    b200rt_ctx *c = m->ctx[i];
    return scene_is_cached(c, h) ? b200rt_set_materials(c, mat, n_mat) : upload_scene(c, R, a, h);
  });
  if (rc) return mfail(m, rc, "GPU %d: %s", m->ctx[bad]->device, m->ctx[bad]->err.c_str());
  m->stats.upload_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  m->stats.nodes = m->ctx[0]->stats.nodes;
  m->stats.triangles = m->ctx[0]->stats.triangles;
  m->stats.bvh_depth = m->ctx[0]->stats.bvh_depth;
  m->stats.repack_ms = m->ctx[0]->stats.repack_ms;
  m->stats.ref_stack_need = m->ctx[0]->stats.ref_stack_need;
  return 0;
}

int b200rt_multi_set_ibl(b200rt_multi *m, const uint8_t *rgba, int width, int height) {
  if (!m) return B200RT_ERR_INVALID;
  int bad = 0;
  const int rc = run_parts((int)m->ctx.size(), &bad, [&](int i) { return b200rt_set_ibl(m->ctx[i], rgba, width, height); });
  if (rc) return mfail(m, rc, "GPU %d: %s", m->ctx[bad]->device, m->ctx[bad]->err.c_str());
  return 0;
}

int b200rt_multi_invalidate(b200rt_multi *m) {
  if (!m) return B200RT_ERR_INVALID;
  for (b200rt_ctx *c : m->ctx) b200rt_invalidate(c);
  return 0;
}

}  // extern "C"

namespace {

// b200rt_multi_render; dn != NULL: then b200rt_render_denoised's G-buffer and passes on GPU 0 after the reduce
int multi_render(b200rt_multi *m, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                 const b200rt_opts *opts, const b200rt_denoise_params *dn, float *out, float *out_noisy) {
  if (!m) return B200RT_ERR_INVALID;
  if (!out) return mfail(m, B200RT_ERR_INVALID, "out_rgb is NULL");
  if (width <= 0 || height <= 0) return mfail(m, B200RT_ERR_INVALID, "bad frame size %d x %d", width, height);
  b200rt_opts o;
  if (opts) o = *opts; else b200rt_default_opts(&o);
  if (o.output != B200RT_OUT_FINAL || o.sample_end > 0 || o.tile_row_mod > 1)
    return mfail(m, B200RT_ERR_INVALID, "the multi-GPU handle divides the frame itself: leave output / sample range / tile rows at their defaults");
  const int n = (int)m->ctx.size();
  const size_t npix = (size_t)width * height, bytes = npix * 3 * sizeof(float);
  b200rt_ctx *c0 = m->ctx[0];
  float s_x = 0.0f;
  if (dn) {
    int rc = check_denoise_frame(c0, o, spp);
    if (!rc) rc = check_denoise(c0, dn, &s_x);
    if (rc) return mfail(m, rc, "%s", c0->err.c_str());
  }
  MCU(cudaSetDevice(c0->device));
  if (m->d_final.cap < bytes) {
    if (m->d_final.p) cudaFree(m->d_final.p);
    m->d_final.p = nullptr; m->d_final.cap = 0;
    MCU(cudaMalloc(&m->d_final.p, bytes));
    m->d_final.cap = bytes;
  }
  // ---- every GPU renders its share into its own buffer; one host thread per GPU issues the launches ------------
  const int tile_rows = (height + 3) / 4;
  int bad = 0;
  int rc = run_parts(n, &bad, [&](int i) {
    b200rt_ctx *c = m->ctx[i];
    b200rt_opts oi = o;
    multi_share(i, n, spp, o.rng_mode, &oi);
    int r = 0;
    if (cudaSetDevice(c->device) != cudaSuccess) r = B200RT_ERR_CUDA;
    if (!r) r = ensure(c, c->d_out, bytes);
    if (!r && cudaMemsetAsync(c->d_out.p, 0, bytes, c->stream) != cudaSuccess) r = B200RT_ERR_CUDA;
    const bool empty = (oi.sample_begin == oi.sample_end) || (oi.tile_row_mod > 1 && oi.tile_row_rem >= tile_rows);
    c->stats.rays = 0; c->stats.samples = 0; c->stats.total_ms = 0; c->stats.kernel_launches = 0;
    if (!r && !empty) r = render_frame(c, cam, env, width, height, spp, max_bounce, &oi, static_cast<float *>(c->d_out.p));
    if (!r && cudaEventRecord(m->done[i], c->stream) != cudaSuccess) r = B200RT_ERR_CUDA;
    if (r == B200RT_ERR_CUDA && c->err.empty()) c->err = "CUDA call failed while enqueueing the frame";
    return r;
  });
  if (rc) return mfail(m, rc, "GPU %d: %s", m->ctx[bad]->device, m->ctx[bad]->err.c_str());
  // ---- GPU 0: wait for the peers (device-side), then one kernel reads every partial buffer and finalises ----------
  MCU(cudaSetDevice(c0->device));
  MCU(cudaEventRecord(m->ev_begin, c0->stream));
  PartList pl;
  pl.n = n;
  for (int i = 0; i < n; ++i) {
    if (i > 0) MCU(cudaStreamWaitEvent(c0->stream, m->done[i], 0));
    const float *src = static_cast<const float *>(m->ctx[i]->d_out.p);
    if (i > 0 && !m->peer_ok[i]) {  // no direct mapping: stage the partial sums on GPU 0
      DevBuf &sb = m->staging[i];
      if (sb.cap < bytes) {
        if (sb.p) cudaFree(sb.p);
        sb.p = nullptr; sb.cap = 0;
        MCU(cudaMalloc(&sb.p, bytes));
        sb.cap = bytes;
      }
      MCU(cudaMemcpyPeerAsync(sb.p, c0->device, src, m->ctx[i]->device, bytes, c0->stream));
      src = static_cast<const float *>(sb.p);
    }
    pl.p[i] = src;
  }
  rc = launch_reduce(c0, pl, static_cast<float *>(m->d_final.p), (long long)npix * 3, (float)spp);
  if (rc) return mfail(m, rc, "%s", c0->err.c_str());
  MCU(cudaEventRecord(m->ev_end, c0->stream));
  if (dn) {
    float *img = static_cast<float *>(m->d_final.p);
    if (out_noisy) MCU(cudaMemcpyAsync(out_noisy, img, bytes, cudaMemcpyDeviceToHost, c0->stream));
    rc = denoise_frame(c0, cam, width, height, o, *dn, s_x, img);   // its launches and rays count in GPU 0's stats
    if (rc) return mfail(m, rc, "GPU %d: %s", c0->device, c0->err.c_str());
  }
  MCU(cudaMemcpyAsync(out, m->d_final.p, bytes, cudaMemcpyDeviceToHost, c0->stream));
  MCU(cudaStreamSynchronize(c0->stream));
  // ---- statistics: work summed over the GPUs, device time = the slowest GPU + the reduce ---------------------------
  b200rt_stats agg = m->stats;
  const float upload_ms = agg.upload_ms;
  memset(&agg, 0, sizeof agg);
  agg.upload_ms = upload_ms;
  float slowest = 0.0f;
  for (int i = 0; i < n; ++i) {
    b200rt_ctx *c = m->ctx[i];
    if (c->stats_pending) {
      MCU(cudaSetDevice(c->device));
      rc = read_counters(c);
      if (rc) return mfail(m, rc, "GPU %d: %s", c->device, c->err.c_str());
    }
    add_work(agg, c->stats);
    slowest = std::max(slowest, c->stats.total_ms);
    agg.primary_ms = std::max(agg.primary_ms, c->stats.primary_ms);
    agg.trace_ms = std::max(agg.trace_ms, c->stats.trace_ms);
  }
  float red = 0.0f;
  MCU(cudaSetDevice(c0->device));
  cudaEventElapsedTime(&red, m->ev_begin, m->ev_end);  // includes waiting for the slowest peer after GPU 0 finished
  agg.total_ms = std::max(slowest, c0->stats.total_ms + red);
  agg.kernel_launches += 1;
  agg.nodes = c0->stats.nodes;
  agg.triangles = c0->stats.triangles;
  agg.bvh_depth = c0->stats.bvh_depth;
  agg.scene_in_smem = c0->stats.scene_in_smem;
  agg.repack_ms = c0->stats.repack_ms;
  agg.ref_stack_need = c0->stats.ref_stack_need;
  m->stats = agg;
  return 0;
}

}  // namespace

extern "C" {

int b200rt_multi_render(b200rt_multi *m, const float *cam, const float *env, int width, int height, int spp, int max_bounce,
                        const b200rt_opts *opts, float *out) {
  return multi_render(m, cam, env, width, height, spp, max_bounce, opts, nullptr, out, nullptr);
}

int b200rt_multi_render_denoised(b200rt_multi *m, const float *cam, const float *env, int width, int height, int spp,
                                 int max_bounce, const b200rt_opts *opts, const b200rt_denoise_params *dn, float *out,
                                 float *out_noisy) {
  if (m && !dn) return mfail(m, B200RT_ERR_INVALID, "denoise parameters are NULL");
  return multi_render(m, cam, env, width, height, spp, max_bounce, opts, dn, out, out_noisy);
}

int b200rt_multi_get_stats(const b200rt_multi *m, b200rt_stats *s) {
  if (!m || !s) return B200RT_ERR_INVALID;
  *s = m->stats;
  return 0;
}

}  // extern "C"

