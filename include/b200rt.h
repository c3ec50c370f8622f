/* b200rt — C ABI of the B200-native (sm_100a) path-tracing hot path.
 *
 * Drop-in boundary for the reference's KernelLauncher.py (QuentinHuan/ENSEM3A_OpenCLRaytracer):
 * every entry point below replaces a piece of that file's PyOpenCL plumbing, cited as
 * KernelLauncher.py:<line>.  Plain pointers and sizes only; all host buffers are owned by the
 * caller and are only read (inputs) or written (outputs) during the call; all calls are
 * synchronous unless the name ends in _device.  Every function returns 0 on success or a
 * negative b200rt_status; b200rt_last_error() gives the message.  There is no CPU, OpenCL,
 * OptiX or library fallback: without a usable CUDA device b200rt_create() fails.
 *
 * One context = one GPU = one host thread at a time.
 */
#ifndef B200RT_H
#define B200RT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200rt_ctx b200rt_ctx;

typedef enum {
  B200RT_OK = 0,
  B200RT_ERR_INVALID = -1,   /* bad argument / inconsistent buffers */
  B200RT_ERR_CUDA = -2,      /* CUDA runtime error (message holds cudaGetErrorString) */
  B200RT_ERR_NO_SCENE = -3,  /* render before b200rt_set_scene / b200rt_set_ibl */
  B200RT_ERR_UNSUPPORTED = -4
} b200rt_status;

/* random-number modes */
#define B200RT_RNG_REFERENCE 0 /* the reference's sequential per-pixel generator (MathLib.cl:294-310),
                                  seeded with the pixel index as Raytracing.cl:171-172 does */
#define B200RT_RNG_PHILOX 1    /* counter-based Philox4x32-10, counter = (pixel, sample, bounce, n), key = seed */

/* traversal modes — both return the hit the reference's rayTrace (MathLib.cl:234-288) returns */
#define B200RT_TRAVERSAL_FAST 0      /* front-to-back, conservatively culled, winner validated by the exact leaf-box test;
                                        ties resolved by the reference's visiting rank */
#define B200RT_TRAVERSAL_REFERENCE 1 /* the reference's visiting order incl. its capped stack (stack.cl:21-26) */
#define B200RT_TRAVERSAL_VERIFY 2    /* runs both per ray, counts disagreements in stats.mismatches, keeps REFERENCE */

/* better estimators of the same integral — SURVEY.md 8f-4, opt-in bit mask, changes the image (same expectation) */
#define B200RT_SAMPLING_REFERENCE 0  /* the reference's: uniform hemisphere with the GGX BRDF as a weight on glossy
                                        surfaces (MathLib.cl:342-366, Raytracing.cl:63-66), emitters found by chance */
#define B200RT_SAMPLING_IMPORTANCE 1 /* one-sample mixture of GGX visible-normal sampling (the lobe the author's dead
                                        rand_sample_GGX aims at, MathLib.cl:369-387) and cosine sampling of the BRDF's
                                        diffuse term; the same BRDF_GGX * cos / pdf estimator, far less variance at low
                                        roughness */
#define B200RT_SAMPLING_LIGHTS 2     /* direct sampling of the emissive triangles (the list FileManager.py:235-240 calls
                                        lightData; the reference kernel receives it and never reads it, Raytracing.cl:163;
                                        intent: the dead sampleLight, MathLib.cl:404-454) at every surface that scatters,
                                        combined with the surface's own sample by the balance heuristic; one more ray per
                                        such surface, three more float4 of path state */

/* output modes */
#define B200RT_OUT_FINAL 0 /* mean over spp, clamped to [0,1]  (Raytracing.cl:211-219) */
#define B200RT_OUT_SUMS 1  /* raw per-pixel sums over [sample_begin, sample_end) — multi-GPU partials */

typedef struct {
  int32_t rng_mode;      /* B200RT_RNG_*           default REFERENCE */
  int32_t traversal;     /* B200RT_TRAVERSAL_*     default FAST */
  int32_t stack_cap;     /* REFERENCE traversal only; <=0 -> 20 (MathLib.cl:248); max 64 */
  int32_t output;        /* B200RT_OUT_* */
  int32_t sample_begin;  /* sample range [sample_begin, sample_end); end <= 0 -> [0, spp).            */
  int32_t sample_end;    /*   a range not starting at 0 needs PHILOX (the reference stream is serial) */
  int32_t pixel_begin;   /* work-item range [pixel_begin, pixel_end); end <= 0 -> [0, width*height)   */
  int32_t pixel_end;
  uint64_t seed;         /* Philox key */
  int32_t collect_stats; /* 1: also count box / triangle tests (slower) */
  int32_t time_kernels;  /* 1: bracket every k_shade / k_trace launch with CUDA events and report the sums
                            (stats.shade_kernel_ms / trace_kernel_ms); adds two event records per iteration */
  int32_t tile_row_mod;  /* > 1: of the frame's rows of 8x4-pixel tiles (4 pixel rows each) only those with        */
  int32_t tile_row_rem;  /*   tile_row % tile_row_mod == tile_row_rem are rendered (interleaved multi-GPU split)  */
  int32_t sample_streams; /* B200RT_RNG_PHILOX only.  0 or 1: one path per pixel in flight, samples accumulated one by one (bit-
                             identical to the oracle's accumulation order).  N > 1: the sample range is cut into N contiguous
                             parts that run concurrently on N CUDA streams of the same GPU (each with its own path state) and
                             whose per-pixel sums are added in part order by the reduce kernel — several samples of a pixel in
                             flight, which fills the GPU on small frames and overlaps shading with tracing on large ones.
                             -1: chosen from the frame size (3 from 1 Mpixel, 4 from 0.2 Mpixel, else 8).  The image equals
                             the one-stream image up to the order of N float additions per pixel. */
  int32_t sampling;       /* bit mask of B200RT_SAMPLING_*; 0 = the reference's estimator (default) */
} b200rt_opts;

typedef struct {
  uint64_t rays;        /* rayTrace invocations: primary + bounce + sun shadow rays */
  uint64_t box_tests;   /* only with collect_stats */
  uint64_t tri_tests;   /* only with collect_stats */
  uint64_t mismatches;  /* TRAVERSAL_VERIFY only */
  uint64_t samples;     /* pixel-samples evaluated */
  float primary_ms;     /* device time of the primary-hit kernel (CUDA events) */
  float trace_ms;       /* device time of the wavefront iterations (all k_shade + k_trace launches) */
  float total_ms;       /* first launch to last launch of the call, device time */
  float upload_ms;      /* host->device copies of the call (wall clock) */
  int32_t kernel_launches; /* kernels launched by the last call */
  int32_t nodes;
  int32_t triangles;
  int32_t bvh_depth;
  int32_t scene_in_smem;  /* 1 when the repacked scene is staged in shared memory */
  int32_t revalidated;    /* rays whose fast-traversal winner failed the exact leaf-box test and were re-traced exactly */
  float shade_kernel_ms;  /* only with time_kernels: summed device time of the k_shade launches */
  float trace_kernel_ms;  /* only with time_kernels: summed device time of the k_trace launches */
  float repack_ms;        /* host time b200rt_set_scene spent validating and repacking the last scene (inside upload_ms) */
  int32_t ref_stack_need; /* stack entries the reference's own walk needs on this tree; above 20 its capped stack drops
                             pushes (stack.cl:21-26) and only B200RT_TRAVERSAL_REFERENCE reproduces that */
  int32_t exact_walks;    /* wavefront rays with a zero / denormal / huge direction component, which skip the conservative
                             traversal and are walked exactly by the shading kernel */
  int32_t wave_iterations; /* wavefront iterations of the last render = k_trace launches per sample stream (kernel_launches
                              also counts the shading, list-compaction and primary-hit kernels) */
  int32_t sample_streams;  /* concurrent sample-range renders the last frame was cut into (b200rt_opts.sample_streams) */
  uint64_t primary_rays;   /* rays of the primary-hit kernel; N sample streams trace them N times, `rays` counts them once */
} b200rt_stats;

void b200rt_default_opts(b200rt_opts *opts);

/* Context on CUDA device `device`.  Replaces cl.Context()/cl.CommandQueue()/Program.build()
 * (main.py:21-28, KernelLauncher.py:8-31). */
int b200rt_create(int device, b200rt_ctx **out_ctx);
void b200rt_destroy(b200rt_ctx *ctx);
const char *b200rt_last_error(const b200rt_ctx *ctx); /* ctx may be NULL: last create() error */

/* Geometry, materials and BVH in the layouts FileManager.py/BVH.py emit (SURVEY.md §8a); counts are
 * array lengths in ELEMENTS.  Replaces the nine cl.Buffer(COPY_HOST_PTR) uploads,
 * KernelLauncher.py:41-69.  light may be NULL/0 (the kernel never reads it).  Validates every index. */
int b200rt_set_scene(b200rt_ctx *ctx, const float *vertex_p, int64_t n_vertex_p, const float *vertex_n,
                     int64_t n_vertex_n, const float *vertex_uv, int64_t n_vertex_uv, const int32_t *face_data,
                     int64_t n_face_data, const float *material_data, int64_t n_material_data,
                     const int32_t *light_data, int64_t n_light_data, const float *bvh, int64_t n_bvh);

/* Only the material table (6 floats per material) — the UI edits materials between renders. */
int b200rt_set_materials(b200rt_ctx *ctx, const float *material_data, int64_t n_material_data);

/* RGBA8 environment map, row-major, top row first.  Replaces cl.Image(...), KernelLauncher.py:71-72. */
int b200rt_set_ibl(b200rt_ctx *ctx, const uint8_t *rgba, int width, int height);

/* The `Raytracing` kernel + blocking read-back, KernelLauncher.py:76-78.  cam = 10 floats, env = 5
 * floats (main.py:59-61,72-73).  width must equal (int)cam[6]; the frame has width*height work-items
 * (height == width in the reference).  out_rgb: width*height*3 floats on the HOST. */
int b200rt_render(b200rt_ctx *ctx, const float *cam, const float *env, int width, int height, int spp,
                  int max_bounce, const b200rt_opts *opts, float *out_rgb);

/* ---- opt-in adaptive sampling: a pixel stops taking samples once its estimated error is below a tolerance ----------
 * The rule, in binary32 with every operation rounded separately (no contraction), true division and a correctly
 * rounded sqrtf:
 *   - a sample's luminance is y = (0.2126f*r + 0.7152f*g) + 0.0722f*b of its final contribution (light-sampling term
 *     included);
 *   - per pixel (mean, m2) start at (0, 0); after the pixel's n-th sample (n counted from 1):
 *       delta = y - mean;  mean = mean + delta / (float)n;  m2 = m2 + delta * (y - mean);
 *   - after sample n with n >= min_spp, (n - min_spp) % check_every == 0 and n < spp:
 *       v = (m2 / (float)(n - 1)) / (float)n;  e = rel_error * fmaxf(fminf(mean, 1.0f), floor);
 *     the pixel stops iff v <= e * e (false for a NaN or Inf anywhere: such a pixel runs to spp);
 *   - a pixel that stopped after n samples is clamp01(sum / (float)n) of the same running sum a fixed-spp render
 *     keeps, i.e. the fixed-spp render of that pixel at spp = n; a pixel that reaches spp is what b200rt_render makes;
 *   - its standard error is sqrtf((m2 / (float)(n - 1)) / (float)n) with its final n;
 *   - pixels whose samples need no ray (primary miss or emitter) are not subject to the rule: they are rendered as
 *     b200rt_render renders them and report spp samples and a standard error of 0.
 * Stopping on a noisy estimate biases the image slightly (a pixel whose first samples happen to agree stops early);
 * rel_error bounds the noise, not that bias. */
typedef struct {
  int32_t min_spp;      /* samples every pixel takes before the rule is first evaluated; 2 <= min_spp <= spp */
  int32_t check_every;  /* evaluate after every check_every-th sample from min_spp on; >= 1 */
  float rel_error;      /* target standard error of the pixel's mean luminance, relative to max(min(mean,1), floor); finite, >= 0 */
  float floor;          /* finite, > 0: below this luminance the target is absolute (rel_error * floor) */
} b200rt_adaptive;

/* b200rt_render with a per-pixel sample count: spp is the maximum.  out_spp (int32 per pixel) and out_stderr
 * (float per pixel) may be NULL; entries of pixels outside the rendered set (pixel range / tile rows) are 0.
 * opts: output must be B200RT_OUT_FINAL over the whole sample range, sample_streams -1, 0 or 1 (the rule needs one
 * serial sequence of samples per pixel; -1 resolves to one stream and stats.sample_streams says 1); pixel ranges,
 * tile rows, both generators, every traversal and every sampling bit are allowed.  The launch loop stops once every
 * pixel has stopped: stats.samples, wave_iterations and kernel_launches report the work actually done. */
int b200rt_render_adaptive(b200rt_ctx *ctx, const float *cam, const float *env, int width, int height, int spp,
                           int max_bounce, const b200rt_opts *opts, const b200rt_adaptive *ad,
                           float *out_rgb, int32_t *out_spp, float *out_stderr);

/* ---- opt-in denoising: an edge-avoiding à-trous filter guided by a G-buffer of the primary hits --------------------
 * The G-buffer, per pixel i, from the primary hit of the render's own traversal mode and stack cap (so that `kind`
 * marks exactly the pixels whose samples need no ray, which the render finishes without tracing):
 *   - kind = -1 for a primary miss, 0 for an emissive material (type 0), 1 otherwise;
 *   - albedo = the material colour (material_data[6m + 1 .. 3]) for kind 1, (1, 1, 1) otherwise;
 *   - normal = normalize(first-vertex normal of the hit triangle) = n / sqrtf((n.x*n.x + n.y*n.y) + n.z*n.z): the
 *     reference's flat, unflipped normal; (0, 0, 0) if a component of it is not finite, and for a miss;
 *   - position = cam_pos + d * k per component (no FMA), d the camera direction of pixel i, k the hit distance;
 *     (0, 0, 0) for a miss.
 * The filter, in binary32 with every operation rounded separately (no contraction), true division, and no
 * transcendental function (so that a restatement can reproduce every bit of the ~10^9 weights of a 1080p frame):
 *   - a pixel with kind != 1 is output unchanged, bit for bit, and is never a tap of another pixel;
 *   - demodulate: c = I / fmaxf(a, 0.01f) per channel (I the input colour, a the albedo);
 *   - for pass l = 0 .. passes-1 with step h = 2^l:  c'_p = (sum_q w_pq * c_q) / (sum_q w_pq) per channel, over the
 *     taps q = p + h*(i, j) with j = -2..2 (rows, outer loop) and i = -2..2 (inner); every sum starts at 0.0f and adds
 *     in that order; a tap outside the frame or with kind_q != 1 is skipped;
 *   - weights, with k1 = {1/16, 1/4, 3/8, 1/4, 1/16} and f(d2, s) = 1.0f / (1.0f + d2 / s):
 *       the centre tap weighs exactly k1[2] * k1[2] (so the denominator is never 0);
 *       any other tap weighs w = (((k1[j+2] * k1[i+2]) * f(dc2, s_c)) * f(dn2, s_n)) * f(dx2, s_x), where
 *       d2 of a vector difference D = q - p is (D.x*D.x + D.y*D.y) + D.z*D.z, dc2 uses the current pass's c,
 *       s_c = (sigma_color * sigma_color) * 2^(-2l) (sigma_color halves every pass), s_n = sigma_normal * sigma_normal and
 *       s_x = sigma_position * sigma_position; a tap whose w is not > 0 (NaN, or 0 through underflow or an infinite
 *       distance) is skipped, so a NaN or infinite colour never reaches another pixel through a zero weight;
 *   - remodulate: out = clamp01(c' * fmaxf(a, 0.01f)), clamp01 being the reference's fmax(fmin(x, 1), 0) with NaN -> 1.
 * Known limits: a primary hit on pass-through glass describes the glass, not what is seen through it; reflections on
 * smooth glossy surfaces are blurred like texture.  The filter keeps the expectation of flat regions but not of
 * every pixel: it trades noise for a little blur. */
#define B200RT_DENOISE_PASSES 5
#define B200RT_DENOISE_SIGMA_COLOR 0.5f
#define B200RT_DENOISE_SIGMA_NORMAL 0.2f
typedef struct {
  int32_t passes;        /* 1..8; default B200RT_DENOISE_PASSES */
  float sigma_color;     /* finite, > 0: colour-distance scale of the first pass (demodulated units) */
  float sigma_normal;    /* finite, > 0: normal-distance scale */
  float sigma_position;  /* finite: > 0 world-distance scale; <= 0 automatic = 0.01f * the binary32 diagonal
                            sqrtf((dx*dx + dy*dy) + dz*dz) of the context's BVH root box (bvh[2..4] min, bvh[5..7] max) */
} b200rt_denoise_params;

/* The G-buffer of a frame: host outputs, 3 floats per pixel for albedo / normal / position and one int32 for kind; each
 * may be NULL.  opts: traversal and stack cap as for b200rt_render; pixel ranges and tile rows are refused. */
int b200rt_gbuffer(b200rt_ctx *ctx, const float *cam, int width, int height, const b200rt_opts *opts, float *albedo,
                   float *normal, float *position, int32_t *kind);

/* The filter on its own: host inputs (rgb / albedo / normal / position 3 floats per pixel, kind one int32 in {-1, 0, 1}),
 * host output, synchronous; out may be rgb.  An automatic sigma_position needs the context's scene. */
int b200rt_denoise(b200rt_ctx *ctx, const float *rgb, const float *albedo, const float *normal, const float *position,
                   const int32_t *kind, int width, int height, const b200rt_denoise_params *dn, float *out);

/* b200rt_render, then the G-buffer and the filter's passes on the device, then one read-back.  out_noisy (may be NULL)
 * receives the image b200rt_render makes.  opts: both generators, every traversal, every sampling bit and any
 * sample_streams; the filter needs the whole finalised frame, so B200RT_OUT_SUMS, a partial sample range, pixel ranges
 * and tile rows are refused.  stats: as b200rt_render, plus 2 + passes kernel launches and width*height camera rays in
 * rays and primary_rays (the G-buffer's); total_ms covers the render only. */
int b200rt_render_denoised(b200rt_ctx *ctx, const float *cam, const float *env, int width, int height, int spp,
                           int max_bounce, const b200rt_opts *opts, const b200rt_denoise_params *dn, float *out_rgb,
                           float *out_noisy);

/* Render + the 8-bit conversion of FileManager.saveImg (FileManager.py:334-338: `(data*255).astype('uint8')`, float32
 * product truncated toward zero) on the device, so that only width*height*3 BYTES cross to the host.  out_rgb8:
 * width*height*3 bytes on the HOST, row-major RGB — what PIL's Image.fromarray(..., 'RGB') takes. */
int b200rt_render_rgb8(b200rt_ctx *ctx, const float *cam, const float *env, int width, int height, int spp,
                       int max_bounce, const b200rt_opts *opts, uint8_t *out_rgb8);

/* Same, but out_rgb is a DEVICE pointer on the context's GPU and the call returns after the kernels
 * are enqueued on the context's stream (b200rt_sync waits).  Used by the multi-GPU path, whose
 * per-GPU partial sums are reduced over NVLink before they ever reach the host. */
int b200rt_render_device(b200rt_ctx *ctx, const float *cam, const float *env, int width, int height, int spp,
                         int max_bounce, const b200rt_opts *opts, float *d_out_rgb);

/* sums (B200RT_OUT_SUMS layout, device) -> clamp(sum / spp), device, in place allowed.  Raytracing.cl:211-219. */
int b200rt_finalize_device(b200rt_ctx *ctx, const float *d_sums, float *d_out_rgb, int64_t n_pixels, int spp);

/* Fused multi-GPU reduce + finalize: out = clamp((sum over n_parts partial-sum buffers) / spp).
 * d_parts[] may be peer-GPU pointers mapped into this process (NVLink P2P loads). */
int b200rt_reduce_finalize_device(b200rt_ctx *ctx, const float *const *d_parts, int n_parts, float *d_out_rgb,
                                  int64_t n_pixels, int spp);

int b200rt_sync(b200rt_ctx *ctx);

/* Run this context's kernels and copies on a caller-owned CUDA stream (cudaStream_t passed as void*),
 * e.g. the stream a torch.distributed / NCCL collective is enqueued on; NULL restores the context's own. */
int b200rt_set_stream(b200rt_ctx *ctx, void *cuda_stream);

/* Forget the content hashes of the cached scene / environment uploads: the next b200rt_set_scene and
 * b200rt_set_ibl copy host->device again even if the bytes are unchanged (what the reference does on
 * every render, KernelLauncher.py:38-72). */
int b200rt_invalidate(b200rt_ctx *ctx);

/* Parity artefact: the primary ray's kept triangle (-1 = miss) and hit distance per work-item. */
int b200rt_primary_hits(b200rt_ctx *ctx, const float *cam, int width, int height, const b200rt_opts *opts,
                        int32_t *tri_out, float *k_out);

/* Closest hit of n caller-supplied rays (6 floats each: origin, direction) — traversal on its own. */
int b200rt_trace_rays(b200rt_ctx *ctx, const float *rays, int64_t n, const b200rt_opts *opts, int32_t *tri_out,
                      float *k_out);

/* The `ImgProcessing` kernel + read-back, KernelLauncher.py:90-103: dst[i] = powr(min(src[i],1), 2.2)
 * for i < n, over `global` work-items (dst[i] untouched for n <= i < global). */
int b200rt_img_processing(b200rt_ctx *ctx, const float *src, float *dst, int64_t n, int64_t global);

int b200rt_get_stats(const b200rt_ctx *ctx, b200rt_stats *stats);

/* Device math used by the kernels, exposed so tests can compare it value by value with the oracle:
 * fn 0 sin, 1 cos, 2 acos, 3 asin, 4 atan2(a,b), 5 tan, 6 pow(a,b), 7 a/b, 8 sqrt, 9/10 the samplers' sincos,
 * 11/12 environment-map column of atan2(a,b) by the fast path / by the correctly rounded angle (8192 wide),
 * 13/14 the same for the row of asin(a) (4096 high). */
int b200rt_math_probe(b200rt_ctx *ctx, int fn, const float *a, const float *b, int64_t n, float *out);

/* Philox4x32-10 block of the device implementation (known-answer tests). */
int b200rt_philox_probe(b200rt_ctx *ctx, const uint32_t ctr[4], uint32_t key0, uint32_t key1, uint32_t out[4]);

/* Plain cudaMalloc / cudaFree on the context's GPU (zero-initialised).  Buffers that are exported with
 * b200rt_ipc_export must come from here: an IPC handle names a whole allocation, so a sub-range of a
 * framework's caching allocator cannot be shared. */
int b200rt_alloc(b200rt_ctx *ctx, int64_t bytes, void **d_ptr_out);
int b200rt_free(b200rt_ctx *ctx, void *d_ptr);

/* CUDA IPC handle (64 bytes) of a device buffer owned by this context's process, and the reverse —
 * lets one rank per GPU map its peers' partial-sum buffers for b200rt_reduce_finalize_device. */
int b200rt_ipc_export(b200rt_ctx *ctx, const void *d_ptr, uint8_t handle_out[64]);
int b200rt_ipc_open(b200rt_ctx *ctx, const uint8_t handle[64], void **d_ptr_out);
int b200rt_ipc_close(b200rt_ctx *ctx, void *d_ptr);

/* The reference's BVH.py, node for node, on the host cores (no context, no GPU involved): same splits (axis of
 * largest centroid variance, at the centroid mean, float64, NumPy's summation order), same node numbering, same
 * float32 boxes, same 9-float export (BVH.py:73-113,147-191).  Replaces `BVH(faceData, V_p).exportArray`
 * (FileManager.py:245).  bvh_out must hold (2 * n_triangles - 1) * 9 floats.  Returns B200RT_ERR_INVALID for an
 * input on which BVH.py itself does not terminate (every centroid of some node on one side of its mean). */
int b200rt_build_bvh(const float *vertex_p, int64_t n_vertex_p, const int32_t *face_data, int64_t n_face_data,
                     float *bvh_out, int64_t n_bvh_out, int32_t *depth_out);

/* ---- several GPUs of one NVSwitch box behind one handle (one host process) ---------------------------------------
 * What SURVEY.md 8b asks of the boundary: the call main.py makes (KernelLauncher.launch_Raytracing, KernelLauncher.py:33)
 * can own 1, 2, 4 or 8 GPUs.  Scene and environment are replicated; the frame is divided by contiguous sample ranges
 * with B200RT_RNG_PHILOX (image equal to the one-GPU image up to the order of the float additions) and by interleaved
 * rows of 8x4-pixel tiles with B200RT_RNG_REFERENCE (bit-identical); the per-GPU partial sums are read over NVLink by
 * one reduce + finalize kernel on the first GPU.  Same argument meaning as the single-GPU calls above; opts must leave
 * output, sample range and tile rows at their defaults.  b200rt_multi_context lends the per-GPU context (index 0 is
 * the GPU that holds the final image) for the calls that need no partition, e.g. b200rt_img_processing. */
typedef struct b200rt_multi b200rt_multi;
int b200rt_multi_create(const int *devices, int n_devices, b200rt_multi **out);
void b200rt_multi_destroy(b200rt_multi *m);
const char *b200rt_multi_last_error(const b200rt_multi *m); /* m may be NULL: last create error */
int b200rt_multi_device_count(const b200rt_multi *m);
b200rt_ctx *b200rt_multi_context(b200rt_multi *m, int index);
int b200rt_multi_set_scene(b200rt_multi *m, const float *vertex_p, int64_t n_vertex_p, const float *vertex_n,
                           int64_t n_vertex_n, const float *vertex_uv, int64_t n_vertex_uv, const int32_t *face_data,
                           int64_t n_face_data, const float *material_data, int64_t n_material_data,
                           const int32_t *light_data, int64_t n_light_data, const float *bvh, int64_t n_bvh);
int b200rt_multi_set_ibl(b200rt_multi *m, const uint8_t *rgba, int width, int height);
int b200rt_multi_invalidate(b200rt_multi *m);
int b200rt_multi_render(b200rt_multi *m, const float *cam, const float *env, int width, int height, int spp,
                        int max_bounce, const b200rt_opts *opts, float *out_rgb);
/* b200rt_multi_render, then b200rt_render_denoised's G-buffer (whole frame) and passes on the first GPU after the
 * reduce; same arguments and refusals as b200rt_multi_render, dn and out_noisy as b200rt_render_denoised. */
int b200rt_multi_render_denoised(b200rt_multi *m, const float *cam, const float *env, int width, int height, int spp,
                                 int max_bounce, const b200rt_opts *opts, const b200rt_denoise_params *dn, float *out_rgb,
                                 float *out_noisy);
/* rays / samples / launches summed over the GPUs (every GPU traces the frame's primary rays once); total_ms = the
 * slowest GPU, reduce included */
int b200rt_multi_get_stats(const b200rt_multi *m, b200rt_stats *stats);

/* Host-only view of what b200rt_set_scene uploads (no context, no GPU): validates the buffers exactly as
 * b200rt_set_scene does and writes the repacked interior-node records (8 x uint32 each, csrc/rt_trace.cuh "repacked
 * scene") to nodes_out (capacity in uint32 words; may be NULL to query).  The records hold the culling tree built over
 * the caller's leaf boxes (csrc/cull_tree.cpp), or the caller's own topology when B200RT_CULL_TREE=0 is set in the
 * environment.  info_out (24 floats): [0] interior nodes, [1] 16-byte units per node, [2] depth of the caller's tree,
 * [3] stack entries the reference-order walk needs, [4] canonical (fast traversal applies), [5] fast_ok, [6] cmax,
 * [7] cull_abs, [8..10] grid base, [11..13] grid pitch, [14..16] grid index of the root box's min planes, [17..19] of its
 * max planes, [20..22] host milliseconds of the three stages (triangles, tree walk, node records incl. the culling
 * tree), [23] depth of the tree in the records (level of its deepest leaf; sizes the traversal stacks).  rank_out (one
 * int32 per triangle, may be NULL): the triangle's position in the reference's visiting order, which breaks distance
 * ties.  Lets the CPU test-suite check that every quantised box encloses the exact one. */
int b200rt_repack_probe(const float *vertex_p, int64_t n_vertex_p, const float *vertex_n, int64_t n_vertex_n,
                        const int32_t *face_data, int64_t n_face_data, int64_t n_materials, const float *bvh,
                        int64_t n_bvh, uint32_t *nodes_out, int64_t n_nodes_out, int32_t *rank_out, float *info_out);

const char *b200rt_version(void);

/* CUDA devices visible to the process (0 without a usable driver / GPU). */
int b200rt_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200RT_H */
