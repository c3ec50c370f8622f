// Opt-in denoising (b200rt_render_denoised, b200rt_denoise, b200rt_gbuffer): the edge-avoiding à-trous filter that
// include/b200rt.h states, guided by a G-buffer of the primary hits.
//
//   k_gbuffer       one thread per pixel: from the tri / k of k_primary<..., PARITY = true, ...> (the hit the render's
//                   k_primary finds), the pixel's kind, normal, position and albedo as three float4 records, and the
//                   rendered colour as a float4 (when the frame comes from the device).
//   k_atrous<F, L>  one launch per pass, 2-D blocks so that a block's taps share L1 lines; ping-pong float4 colour.
//                   FIRST demodulates every tap it loads, LAST remodulates, clamps and writes the 3-float image.
// No transcendental, no contraction (the library is built with -fmad=false -prec-div=true): the code below is the
// header's statement in its order of operations, which is what makes it restatable bit for bit.
#pragma once
#include "rt_kernels.cuh"

namespace b200rt {

constexpr int kDnBlockX = 32, kDnBlockY = 4;
constexpr int kDnMaxPasses = 8;

// G-buffer records, one float4 each per pixel: gn = normal.xyz, kind;  gx = position.xyz, 0;  ga = albedo.xyz, 0
struct GBufferView {
  float4 *gn, *gx, *ga;
};

// SMOOTH (B200RT_SAMPLING_SMOOTH_NORMALS): the normal of a hit on a curved triangle is the normalised shading normal at
// the render's point cam_pos + unit(d) * k.  TEX (B200RT_SAMPLING_TEXTURES): the albedo of a type-1 or type-2 hit is
// surface_albedo at that point.
template <bool SMOOTH, bool TEX = false>
__global__ void __launch_bounds__(kBlock) k_gbuffer(const __grid_constant__ KernelArgs A, const int *__restrict__ tri,
                                                    const float *__restrict__ k, GBufferView G,
                                                    const float *__restrict__ rgb, float4 *__restrict__ col) {
  const int n = A.F.width * A.F.height;
  const int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  const SceneView &S = A.S;
  const int t = __ldg(tri + i);
  float kind = -1.0f;
  v3 nrm = mk3(0.0f, 0.0f, 0.0f), pos = mk3(0.0f, 0.0f, 0.0f), alb = mk3(1.0f, 1.0f, 1.0f);
  if (t >= 0) {
    const Material m = load_material(S.mats, tri_material(S, t));
    kind = m.type == 0 ? 0.0f : 1.0f;
    if (m.type != 0) alb = m.color;
    const float4 f0 = __ldg(S.frames + (size_t)kFrameVec * t);   // normalize(first-vertex normal), k_tri_frames
    if (isfinite(f0.x) && isfinite(f0.y) && isfinite(f0.z)) nrm = mk3(f0.x, f0.y, f0.z);
    const v3 d = camera_dir(A.F, i);
    if (SMOOTH) {
      const float4 nn = __ldg(S.normals + t);
      bool curved;
      const v3 n = shading_normal<true>(S, A.n_tris, t, mk3(nn.x, nn.y, nn.z), A.F.cam_pos + unit(d) * __ldg(k + i), &curved);
      if (curved) {
        const v3 un = unit(n);
        nrm = (isfinite(un.x) && isfinite(un.y) && isfinite(un.z)) ? un : mk3(0.0f, 0.0f, 0.0f);
      }
    }
    if (TEX && (m.type == 1 || m.type == 2))
      alb = surface_albedo(S, A.n_tris, t, tri_material(S, t), m.color, A.F.cam_pos + unit(d) * __ldg(k + i));
    pos = A.F.cam_pos + d * __ldg(k + i);
  }
  G.gn[i] = make_float4(nrm.x, nrm.y, nrm.z, kind);
  G.gx[i] = make_float4(pos.x, pos.y, pos.z, 0.0f);
  G.ga[i] = make_float4(alb.x, alb.y, alb.z, 0.0f);
  if (rgb) col[i] = make_float4(__ldg(rgb + 3 * (size_t)i), __ldg(rgb + 3 * (size_t)i + 1), __ldg(rgb + 3 * (size_t)i + 2), 0.0f);
}

struct AtrousArgs {
  const float4 *gn, *gx, *ga;   // G-buffer records (GBufferView)
  const float4 *cin;            // FIRST: the input colour I; else the previous pass's c (kind != 1: I, passed through)
  float4 *cout;                 // !LAST: this pass's c
  float *out;                   // LAST: the image, 3 floats per pixel
  int width, height, step;
  float s_c, s_n, s_x;          // this pass's scales (b200rt.h): sigma_color^2 * 2^-2l, sigma_normal^2, sigma_position^2
};

RT_DEV v3 demodulate(float4 I, float4 a) {
  return mk3(I.x / fmaxf(a.x, 0.01f), I.y / fmaxf(a.y, 0.01f), I.z / fmaxf(a.z, 0.01f));
}

RT_DEV float d2(v3 a, v3 b) {
  const v3 D = b - a;
  return (D.x * D.x + D.y * D.y) + D.z * D.z;
}

RT_DEV float edge_f(float d2v, float s) { return 1.0f / (1.0f + d2v / s); }

// __maxnreg__ instead of __launch_bounds__: left to itself ptxas keeps the FIRST instance at 40 registers around the
// true divisions' slow-path calls and spills; 64 still allows 8 blocks of 128 threads per SM
template <bool FIRST, bool LAST>
__global__ void __maxnreg__(64) k_atrous(const __grid_constant__ AtrousArgs P) {
  const int x = blockIdx.x * kDnBlockX + threadIdx.x, y = blockIdx.y * kDnBlockY + threadIdx.y;
  if (x >= P.width || y >= P.height) return;
  const int p = y * P.width + x;
  const float4 gp = __ldg(P.gn + p);
  const float4 cp4 = __ldg(P.cin + p);
  if (gp.w != 1.0f) {   // ray-free pixel: unchanged, bit for bit
    if (LAST) {
      P.out[3 * (size_t)p] = cp4.x; P.out[3 * (size_t)p + 1] = cp4.y; P.out[3 * (size_t)p + 2] = cp4.z;
    } else {
      P.cout[p] = cp4;
    }
    return;
  }
  const float4 ap = __ldg(P.ga + p);
  const float4 xp4 = __ldg(P.gx + p);
  const v3 np = mk3(gp.x, gp.y, gp.z), xp = mk3(xp4.x, xp4.y, xp4.z);
  const v3 cp = FIRST ? demodulate(cp4, ap) : mk3(cp4.x, cp4.y, cp4.z);
  const float k1[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
  float sx = 0.0f, sy = 0.0f, sz = 0.0f, sw = 0.0f;
#pragma unroll
  for (int j = -2; j <= 2; ++j) {
    const int yq = y + P.step * j;
#pragma unroll
    for (int i = -2; i <= 2; ++i) {
      const int xq = x + P.step * i;
      float w;
      v3 cq;
      if (i == 0 && j == 0) {
        w = k1[2] * k1[2];
        cq = cp;
      } else {
        if (xq < 0 || xq >= P.width || yq < 0 || yq >= P.height) continue;
        const int q = yq * P.width + xq;
        const float4 gq = __ldg(P.gn + q);
        if (gq.w != 1.0f) continue;
        const float4 cq4 = __ldg(P.cin + q);
        cq = FIRST ? demodulate(cq4, __ldg(P.ga + q)) : mk3(cq4.x, cq4.y, cq4.z);
        const float4 xq4 = __ldg(P.gx + q);
        w = (((k1[j + 2] * k1[i + 2]) * edge_f(d2(cp, cq), P.s_c)) * edge_f(d2(np, mk3(gq.x, gq.y, gq.z)), P.s_n)) *
            edge_f(d2(xp, mk3(xq4.x, xq4.y, xq4.z)), P.s_x);
        if (!(w > 0.0f)) continue;
      }
      sx = sx + w * cq.x;
      sy = sy + w * cq.y;
      sz = sz + w * cq.z;
      sw = sw + w;
    }
  }
  const v3 c = mk3(sx / sw, sy / sw, sz / sw);
  if (LAST) {
    float *o = P.out + 3 * (size_t)p;
    o[0] = clamp01(c.x * fmaxf(ap.x, 0.01f));
    o[1] = clamp01(c.y * fmaxf(ap.y, 0.01f));
    o[2] = clamp01(c.z * fmaxf(ap.z, 0.01f));
  } else {
    P.cout[p] = make_float4(c.x, c.y, c.z, 0.0f);
  }
}

}  // namespace b200rt
