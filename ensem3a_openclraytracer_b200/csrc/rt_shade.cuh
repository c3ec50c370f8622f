// Camera rays, direction sampling, BSDFs and the environment lookup of the b200rt kernels.
// Each function follows the reference statement by statement in rounding order
// (file:line given per function); see rt_math.cuh for the arithmetic contract.
#pragma once
#include "rt_math.cuh"

namespace b200rt {

// Everything that is constant over one frame.  The transcendental parts (camera / sun / environment
// rotations, focal distance) are evaluated once on the host by frame_setup() in b200rt_api.cu with
// the same correctly-rounded definitions; the reference re-derives them per ray.
struct FrameParams {
  int width, height;
  v3 cam_pos;
  float focal_off;  // 1 / (2 tan(fov/2)), Raytracing.cl:24
  float step;       // (float)(1.0 / cam[6]), Raytracing.cl:27
  rotor cam_rx, cam_ry, cam_rz;
  v3 sun_dir;       // Raytracing.cl:115-118
  float sun_power, ibl_power;
  rotor ibl_r1, ibl_r2;  // MathLib.cl:73-74
  int ibl_w, ibl_h;
  int spp, max_bounce;
  int s0, s1;
  int pixel_begin, pixel_end;
  int tile_row_mod, tile_row_rem;  // > 1: only tile rows with row % mod == rem (b200rt_opts)
  int out_mode;
  int rng_mode;
  uint32_t key0, key1;
  int sampling;     // B200RT_SAMPLING_*
};

struct Material {
  int type;
  v3 color;
  float roughness;
};

RT_DEV Material load_material(const float *mats, int idx) {  // Raytracing.cl:5-15
  const float *m = mats + 6 * idx;
  Material r;
  r.type = (int)__ldg(m);
  r.color = mk3(__ldg(m + 1), __ldg(m + 2), __ldg(m + 3));
  r.roughness = __ldg(m + 4);
  return r;
}

// Raytracing.cl:18-37: the camera direction through image-plane point (fx, fz), in pixels (column, row)
RT_DEV v3 camera_dir_at(const FrameParams &F, float fx, float fz) {
  v3 focal = mk3(F.cam_pos.x, F.cam_pos.y - F.focal_off, F.cam_pos.z);
  v3 pix = mk3(fx * F.step - 0.5f, 0.0f, 0.5f - fz * F.step);
  v3 d = unit((F.cam_pos + pix) - focal);
  d = apply_rotor(F.cam_rx, d);
  d = apply_rotor(F.cam_ry, d);
  d = apply_rotor(F.cam_rz, d);
  return d;
}

// the reference's camera ray of work-item i (column (i + 1) % width, its off-by-one included, Raytracing.cl:21-22)
RT_DEV v3 camera_dir(const FrameParams &F, int i) {
  int col = (i + 1) % F.width;
  int row = (i - col) / F.width;
  return camera_dir_at(F, (float)col, (float)row);
}

// opt-in pixel jitter (b200rt_opts.sampling bit 3): the ray through (col + ux - 0.5, row + uy - 0.5), a point of the
// one-pixel footprint centred on the reference's ray; (ux, uy) uniform in [0, 1)
RT_DEV v3 camera_dir_jittered(const FrameParams &F, int i, float ux, float uy) {
  int col = (i + 1) % F.width;
  int row = (i - col) / F.width;
  return camera_dir_at(F, (float)col + (ux - 0.5f), (float)row + (uy - 0.5f));
}

// uv * extent -> integer texel, exactly the reference's chain of binary32 roundings (MathLib.cl:78-80,87):
// RN(RN(a * inv) + 0.5) * extent, truncated, clamped by the sampler.  Monotone non-decreasing in a.
RT_DEV int texel_coord(float a, float inv, int extent) {
  const float u = a * inv + 0.5f;
  const int p = __float2int_rz(u * (float)extent);
  return max(0, min(p, extent - 1));
}

// The environment lookup needs atan2 / asin only to pick a texel.  CUDA documents the binary32 atan2f at 3 ulp and asinf
// at 2 ulp of the true value (measured around every texel boundary of 1x1 .. 8192x4096 maps, and within a few ulp of
// +-2^k: at most 2 and 1 ulp from the correctly rounded angle, tests/test_gpu_arith_exhaustive.py).  del = |a| 2^-21 is
// at least 4 ulp of a, so [a - del, a + del] holds the correctly rounded angle; texel_coord is monotone, so if both
// ends of that interval land in the same texel the texel is decided — otherwise (a lookup within ~1e-6 of a texel
// boundary) the correctly rounded binary64 path is taken.
RT_DEV int ibl_texel_u(float z, float x, int w) {
  const float a = atan2f(z, x);
  const float del = fabsf(a) * 4.76837158203125e-07f;  // 2^-21 >= 4 ulp of a
  int p = texel_coord(a - del, 0.1591f, w);
  if (p != texel_coord(a + del, 0.1591f, w)) p = texel_coord(cr_atan2(z, x), 0.1591f, w);
  return p;
}
RT_DEV int ibl_texel_v(float y, int h) {
  const float a = asinf(y);
  const float del = fabsf(a) * 4.76837158203125e-07f;
  int p = texel_coord(a - del, 0.3183f, h);
  if (p != texel_coord(a + del, 0.3183f, h)) p = texel_coord(cr_asin(y), 0.3183f, h);
  return p;
}

// MathLib.cl:72-90.  Integer texel coordinates through a clamp-to-edge sampler; UNORM8 -> b/255.
RT_DEV v3 ibl_lookup(const FrameParams &F, cudaTextureObject_t tex, v3 dir) {
  dir = apply_rotor(F.ibl_r1, dir);
  dir = apply_rotor(F.ibl_r2, dir);
  const int px = ibl_texel_u(dir.z, dir.x, F.ibl_w);
  const int py = ibl_texel_v(dir.y, F.ibl_h);
  uchar4 t = tex2D<uchar4>(tex, (float)px + 0.5f, (float)py + 0.5f);
  return mk3(__fdiv_rn((float)t.x, 255.0f), __fdiv_rn((float)t.y, 255.0f), __fdiv_rn((float)t.z, 255.0f)) * 1.0f;
}

// ---- per-triangle sampling frame ------------------------------------------------------------------------------
// Both samplers rotate a local +Z hemisphere direction onto the triangle's normal n (MathLib.cl:325-336 and
// :349-361): angle acos(n.z) about cross((0,0,1), n), through rotateVec — or, when |normalize(n).z| == 1, scale by
// n.z.  All of it depends on the triangle alone, so k_tri_frames evaluates it once per triangle at upload time with
// exactly the device code a per-sample evaluation would run:
//   f0 = normalize(n).xyz, z-aligned flag      f1,f2 = rotor of the cosine sampler (axis not normalised before
//   rotateVec)      f3,f4 = rotor of the uniform sampler (axis normalised first; rotateVec normalises again)
constexpr int kFrameVec = 5;  // float4 per triangle

struct TriFrame {
  v3 un;
  bool zal;
  rotor rot;
};

RT_DEV void make_tri_frame(v3 n, float4 *f) {
  const v3 zup = mk3(0.0f, 0.0f, 1.0f);
  const v3 un = unit(n);
  const bool zal = fabsf(dot(un, zup)) == 1.0f;
  const v3 axis = cross(zup, n);
  const float ang = cr_acos(dot(n, zup));
  float s, c;
  cr_sincos(ang * 0.5f, &s, &c);
  const rotor rc = make_rotor(c, s, axis);
  const rotor ru = make_rotor(c, s, unit(axis));
  f[0] = make_float4(un.x, un.y, un.z, zal ? 1.0f : 0.0f);
  f[1] = make_float4(rc.q.w, rc.q.x, rc.q.y, rc.q.z);
  f[2] = make_float4(rc.qi.w, rc.qi.x, rc.qi.y, rc.qi.z);
  f[3] = make_float4(ru.q.w, ru.q.x, ru.q.y, ru.q.z);
  f[4] = make_float4(ru.qi.w, ru.qi.x, ru.qi.y, ru.qi.z);
}

// which: 0 = unit normal only (glass), 1 = + cosine rotor, 2 = + uniform rotor
RT_DEV TriFrame load_tri_frame(const float4 *frames, int tri, int which) {
  const float4 *f = frames + (size_t)kFrameVec * tri;
  TriFrame T;
  const float4 f0 = __ldg(f);
  T.un = mk3(f0.x, f0.y, f0.z);
  T.zal = f0.w != 0.0f;
  if (which != 0) {
    const float4 a = __ldg(f + (which == 1 ? 1 : 3)), b = __ldg(f + (which == 1 ? 2 : 4));
    T.rot.q.w = a.x; T.rot.q.x = a.y; T.rot.q.y = a.z; T.rot.q.z = a.w;
    T.rot.qi.w = b.x; T.rot.qi.x = b.y; T.rot.qi.y = b.z; T.rot.qi.z = b.w;
  }
  return T;
}

// opt-in smooth shading (B200RT_SAMPLING_SMOOTH_NORMALS): load_tri_frame's result for a normal known only at the hit,
// make_tri_frame's statements in registers.  Glass (which 0) needs the unit normal alone.
RT_DEV TriFrame tri_frame_at(v3 n, int which) {
  TriFrame T;
  if (which == 0) {
    T.un = unit(n);
    T.zal = false;
    return T;
  }
  float4 f[kFrameVec];
  make_tri_frame(n, f);
  T.un = mk3(f[0].x, f[0].y, f[0].z);
  T.zal = f[0].w != 0.0f;
  const float4 a = which == 1 ? f[1] : f[3], b = which == 1 ? f[2] : f[4];
  T.rot.q.w = a.x; T.rot.q.x = a.y; T.rot.q.y = a.z; T.rot.q.z = a.w;
  T.rot.qi.w = b.x; T.rot.qi.x = b.y; T.rot.qi.y = b.z; T.rot.qi.z = b.w;
  return T;
}

// MathLib.cl:313-339
RT_DEV v3 sample_cosine(v3 n, const TriFrame &T, float u, float u2, float *inv_pdf) {
  float theta = u2 * 2.0f * 3.14f;
  float rad = sqrtf(u);
  float st, ct;
  cr_sincos(theta, &st, &ct);
  v3 local = mk3(rad * ct, rad * st, sqrtf(fmaxf(0.0f, 1.0f - u)));
  v3 l;
  if (T.zal) {
    l = local * n.z;
  } else {
    l = unit(apply_rotor(T.rot, local));
  }
  *inv_pdf = 3.14f / fmaxf(dot(l, n), 0.0f);
  return l;
}

// MathLib.cl:342-366
RT_DEV v3 sample_uniform(v3 n, const TriFrame &T, float u, float u2, float *inv_pdf) {
  float phi = 2.0f * 3.14f * u;
  float theta = cr_acos(1.0f - u2);
  float st, ct, sp, cp;
  cr_sincos(theta, &st, &ct);
  cr_sincos(phi, &sp, &cp);
  v3 local = mk3(cp * st, st * sp, ct);
  *inv_pdf = 2.0f * 3.14f;
  if (T.zal) return local * n.z;
  return apply_rotor(T.rot, local);
}

// ---- GGX microfacet pieces shared by the importance sampler of glossy surfaces and rough glass -------------------------
// orthonormal basis (T, B) around the unit vector N (Duff et al. 2017)
RT_DEV void basis_duff(v3 N, v3 *T, v3 *B) {
  const float sg = copysignf(1.0f, N.z);
  const float a = -1.0f / (sg + N.z);
  const float b = N.x * N.y * a;
  *T = mk3(1.0f + sg * N.x * N.x * a, sg * b, -sg * N.x);
  *B = mk3(b, sg + N.y * N.y * a, -N.y);
}

// A normal of the GGX distribution of visible normals [Heitz 2018] of roughness al around N (basis T, B from basis_duff)
// seen from the unit direction Vw, ndv = dot(N, Vw); (r, sp, cp) is the radius, sine and cosine of the polar point of
// the unit disc it is drawn with.  The importance sampler of glossy surfaces and rough glass share these statements.
RT_DEV v3 ggx_visible_normal(float al, v3 N, v3 T, v3 B, v3 Vw, float ndv, float r, float sp, float cp) {
  const v3 Vh = unit(mk3(al * dot(Vw, T), al * dot(Vw, B), ndv));
  const float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
  v3 T1 = mk3(1.0f, 0.0f, 0.0f);
  if (lensq > 0.0f) {
    const float inv = 1.0f / sqrtf(lensq);
    T1 = mk3(-Vh.y * inv, Vh.x * inv, 0.0f);
  }
  const v3 T2 = cross(Vh, T1);
  const float t1 = r * cp;
  float t2 = r * sp;
  const float s = 0.5f * (1.0f + Vh.z);
  t2 = (1.0f - s) * sqrtf(fmaxf(0.0f, 1.0f - t1 * t1)) + s * t2;
  const float t3 = sqrtf(fmaxf(0.0f, 1.0f - t1 * t1 - t2 * t2));
  const v3 Nh = ((T1 * t1) + (T2 * t2)) + (Vh * t3);
  const v3 hl = unit(mk3(al * Nh.x, al * Nh.y, fmaxf(0.0f, Nh.z)));
  return ((T * hl.x) + (B * hl.y)) + (N * hl.z);
}

// Smith's separable masking term of GGX for a direction at cosine c > 0 to the normal, a2 = alpha^2
RT_DEV float smith_g1(float a2, float c) { return (2.0f * c) / (c + sqrtf(a2 + (1.0f - a2) * c * c)); }

// ---- opt-in: refractive glass (b200rt_opts.sampling bit B200RT_SAMPLING_DIELECTRIC_GLASS) -------------------------------
constexpr float kGlassDefaultIor = 1.5f;  // B200RT_GLASS_DEFAULT_IOR: the ior of a glass material whose ior slot is 0

// the raw ior slot of material idx (materialData[6 idx + 5]), which the reference's extractMaterial never reads
RT_DEV float load_material_ior(const float *mats, int idx) { return __ldg(mats + 6 * idx + 5); }

// Fresnel's reflectance of unpolarised light at an interface of relative index eta, ci the cosine on the incident side,
// ct = sqrtf(k) the cosine of the refracted direction
RT_DEV float fresnel(float eta, float ci, float ct) {
  const float rs = (eta * ci - ct) / (eta * ci + ct);
  const float rp = (ci - eta * ct) / (ci + eta * ct);
  return 0.5f * (rs * rs + rp * rp);
}

// The smooth dielectric interface of b200rt.h: the next direction of a path that meets glass of index `ior` along d,
// un the unit normal, u one uniform.  Reflects with Fresnel's probability F (always on total internal reflection),
// refracts by Snell's law otherwise; *reflected tells which.  The caller keeps the throughput on a reflection and
// tints it by the colour on a refraction.
RT_DEV v3 scatter_dielectric(v3 d, v3 un, float ior, float u, bool *reflected) {
  const v3 w = unit(d);
  const float c = dot(w, un);
  const bool enter = c < 0.0f;
  const float eta = enter ? 1.0f / ior : ior;
  const float ci = enter ? -c : c;
  const v3 m = enter ? un : neg3(un);
  const float k = 1.0f - (eta * eta) * (1.0f - ci * ci);
  float ct = 0.0f;
  bool refl = true;
  if (k >= 0.0f) {
    ct = sqrtf(k);
    refl = !(u >= fresnel(eta, ci, ct));
  }
  *reflected = refl;
  if (refl) return w + m * (2.0f * ci);
  return w * eta + m * (eta * ci - ct);
}

// ---- opt-in: rough glass (b200rt_opts.sampling bit B200RT_SAMPLING_ROUGH_GLASS, on top of refractive glass) ------------
// The GGX microfacet interface of b200rt.h [Walter et al. 2007] with alpha = roughness > 0, met along d (un the unit
// normal, ior != 1): a microfacet normal h drawn from the visible normals seen from the incident side with (u1, u2), then
// scatter_dielectric's Fresnel choice at h with uf.  *reflected tells which; *weight is Smith's G1 of the outgoing
// direction, or 0 when that direction leaves on the wrong side of the surface.  c == 0, a non-finite c (un) or a
// non-finite h take scatter_dielectric with uf and weight 1.  The caller tints a refraction by the colour, then
// multiplies the throughput by the weight (a weight of 0 zeroes it).
RT_DEV v3 scatter_rough_dielectric(v3 d, v3 un, float ior, float al, float uf, float u1, float u2, bool *reflected,
                                   float *weight) {
  const float kTwoPi = 6.2831853f;
  const v3 w = unit(d);
  const float c = dot(w, un);
  const bool enter = c < 0.0f;
  const float eta = enter ? 1.0f / ior : ior;
  const v3 m = enter ? un : neg3(un);
  const v3 Vw = neg3(w);
  v3 T, B;
  basis_duff(m, &T, &B);
  float sp, cp;
  cr_sincos(kTwoPi * u2, &sp, &cp);
  const v3 h = ggx_visible_normal(al, m, T, B, Vw, dot(m, Vw), sqrtf(u1), sp, cp);
  *weight = 1.0f;
  if (c == 0.0f || !isfinite(c) || !isfinite(h.x) || !isfinite(h.y) || !isfinite(h.z))
    return scatter_dielectric(d, un, ior, uf, reflected);
  const float ch = dot(Vw, h);
  const float k = 1.0f - (eta * eta) * (1.0f - ch * ch);
  float ct = 0.0f;
  bool refl = true;
  if (k >= 0.0f) {
    ct = sqrtf(k);
    refl = !(uf >= fresnel(eta, ch, ct));
  }
  *reflected = refl;
  const v3 nd = refl ? w + h * (2.0f * ch) : w * eta + h * (eta * ch - ct);
  const float co = dot(nd, m);
  *weight = (refl ? co > 0.0f : co < 0.0f) ? smith_g1(al * al, fabsf(co)) : 0.0f;
  return nd;
}

// ---- opt-in: albedo textures (b200rt_opts.sampling bit B200RT_SAMPLING_TEXTURES) ---------------------------------------
// The bound textures (b200rt_set_textures) are read through the read-only data path.  The texture unit's bilinear filter
// is not used: its 8-bit fractional weights are not the float weights b200rt.h states.
struct TexView {
  const int4 *info;       // per texture: index of its first texel, w, h, -
  const uchar4 *texels;   // every texture's texels back to back, row-major, top row first
};

RT_DEV float lerpf(float a, float b, float t) { return a + (b - a) * t; }

RT_DEV v3 texel_value(const TexView &T, int base, int w, int x, int y) {
  const uchar4 c = __ldg(T.texels + base + y * w + x);
  return mk3(__fdiv_rn((float)c.x, 255.0f), __fdiv_rn((float)c.y, 255.0f), __fdiv_rn((float)c.z, 255.0f));
}

RT_DEV int wrap_index(int i, int n) {
  const int r = i % n;
  return r < 0 ? r + n : r;
}

// The texture factor f of b200rt.h at (u, v): repeat wrap, bilinear as lerps between the four texels around the point.
RT_DEV v3 texture_factor(const TexView &T, int tex, float u, float v) {
  if (!isfinite(u) || !isfinite(v)) return mk3(1.0f, 1.0f, 1.0f);
  const int4 info = __ldg(T.info + tex);
  const int w = info.y, h = info.z;
  const float fu = u - floorf(u), fv = v - floorf(v);
  const float tx = fu * (float)w - 0.5f, ty = (1.0f - fv) * (float)h - 0.5f;
  const int x0 = (int)floorf(tx), y0 = (int)floorf(ty);
  const float ax = tx - (float)x0, ay = ty - (float)y0;
  const int xa = wrap_index(x0, w), xb = wrap_index(x0 + 1, w), ya = wrap_index(y0, h), yb = wrap_index(y0 + 1, h);
  const v3 c00 = texel_value(T, info.x, w, xa, ya), c10 = texel_value(T, info.x, w, xb, ya);
  const v3 c01 = texel_value(T, info.x, w, xa, yb), c11 = texel_value(T, info.x, w, xb, yb);
  const v3 top = mk3(lerpf(c00.x, c10.x, ax), lerpf(c00.y, c10.y, ax), lerpf(c00.z, c10.z, ax));
  const v3 bot = mk3(lerpf(c01.x, c11.x, ax), lerpf(c01.y, c11.y, ax), lerpf(c01.z, c11.z, ax));
  return mk3(lerpf(top.x, bot.x, ay), lerpf(top.y, bot.y, ay), lerpf(top.z, bot.z, ay));
}

RT_DEV float ipow(float x, int n) {  // pown: repeated multiply from 1
  float r = 1.0f;
  for (int i = 0; i < n; ++i) r = r * x;
  return r;
}

// MathLib.cl:461-500
RT_DEV v3 bsdf_ggx(const Material &m, v3 v, v3 l, v3 n) {
  v3 h = unit(l + v);
  float a2 = ipow(m.roughness, 2);
  float D = a2 / (3.14f * ipow(ipow(fmaxf(dot(n, h), 0.0f), 2) * (a2 - 1.0f) + 1.0f, 2));
  float ndv = fmaxf(dot(n, v), 0.0f);
  float kk = m.roughness * sqrtf(2.0f / 3.14f);
  float g1 = ndv / (ndv * (1.0f - kk) + kk);
  float ndl = fmaxf(dot(n, l), 0.0f);
  float g2 = ndl / (ndl * (1.0f - kk) + kk);
  float G = g1 * g2;
  float F = 0.04f + (1.0f - 0.04f) * ipow(1.0f - fmaxf(dot(h, v), 0.0f), 5);
  float spec = (F * G * D) * (1.0f / fmaxf(4.0f * fmaxf(dot(v, n), 0.0f) * fmaxf(dot(l, n), 0.0f), 0.001f));
  float kd = (1.0f - F) * (1.0f - 0.5f);
  v3 diffuse = (m.color * kd) / 3.14f;
  return mk3(diffuse.x + spec, diffuse.y + spec, diffuse.z + spec);
}

// ---- opt-in: importance sampling of glossy surfaces (SURVEY.md 8f-4) ------------------------------------------------------
// The reference draws the next direction of a glossy surface uniformly over the hemisphere and carries BRDF_GGX as a
// weight (MathLib.cl:342-366, Raytracing.cl:63-66): at low roughness almost every sample misses the lobe.  This draws
// from a one-sample mixture of (a) the GGX distribution of visible normals [Heitz 2018] with alpha = roughness — the
// normal distribution BRDF_GGX itself uses (MathLib.cl:470-472) — reflected about the sampled normal, and (b) a
// cosine-weighted lobe for the BRDF's diffuse term, and returns 1 / pdf of the mixture, so the caller's
// BRDF_GGX * |cos| * inv_pdf is an estimator of the same integral.  u0 picks the lobe and is stretched back to [0, 1).
// A view direction below the surface (the reference does not flip normals) uses the cosine lobe alone.
// The test-side CPU restatement mirrors this statement order, so images stay bit-identical to it.
// density (per solid angle) with which sample_glossy_importance draws direction l; N, Vw unit vectors
RT_DEV float glossy_mix_pdf(float al, v3 N, v3 Vw, v3 l) {
  const float kPi = 3.14159265f;
  const float ndv = dot(N, Vw);
  const float ndl = dot(N, l);
  const float pdf_cos = fmaxf(ndl, 0.0f) / kPi;
  float pdf_spec = 0.0f;
  if (ndv > 0.0f && ndl > 0.0f) {
    const v3 h = unit(l + Vw);
    const float ndh = dot(N, h);
    const float a2 = al * al;
    const float dden = ndh * ndh * (a2 - 1.0f) + 1.0f;
    const float D = a2 / (kPi * dden * dden);
    const float G1 = smith_g1(a2, ndv);
    pdf_spec = (G1 * D) / (4.0f * ndv);
  }
  const float ps = ndv > 0.0f ? 0.5f : 0.0f;
  return ps * pdf_spec + (1.0f - ps) * pdf_cos;
}

RT_DEV v3 sample_glossy_importance(float roughness, v3 un, v3 d_in, float u0, float u1, float *inv_pdf) {
  const float kPi = 3.14159265f, kTwoPi = 6.2831853f;
  const v3 N = un;
  const v3 Vw = unit(neg3(d_in));
  const float ndv = dot(N, Vw);
  v3 T, B;
  basis_duff(N, &T, &B);
  const bool spec = ndv > 0.0f && u0 < 0.5f;
  const float u0r = u0 < 0.5f ? u0 * 2.0f : u0 * 2.0f - 1.0f;
  const float al = roughness;
  float sp, cp;
  cr_sincos(kTwoPi * u1, &sp, &cp);
  const float r = sqrtf(u0r);
  v3 l;
  if (spec) {
    const v3 h = ggx_visible_normal(al, N, T, B, Vw, ndv, r, sp, cp);
    l = (h * (2.0f * dot(Vw, h))) - Vw;
  } else {
    l = ((T * (r * cp)) + (B * (r * sp))) + (N * sqrtf(fmaxf(0.0f, 1.0f - u0r)));
  }
  const float pdf = glossy_mix_pdf(al, N, Vw, l);
  // the reference's uniform sampler weighs with 2 * 3.14 where the true density is 1 / (2 pi): its expectation is
  // 3.14 / pi times the integral.  Kept, so that both samplers converge to the same image.
  *inv_pdf = pdf > 0.0f ? (3.14f / kPi) / pdf : 0.0f;
  return l;
}

// ---- opt-in: direct sampling of the emitters (SURVEY.md 8f-4; b200rt_opts.sampling bit 1) ---------------------------------
// Not in the reference, whose kernel receives lightData and never reads it (Raytracing.cl:163); the author's intent is
// the dead sampleLight, MathLib.cl:404-454.  At every surface that scatters (types 1, 2) one emitter triangle is chosen
// uniformly and one point uniformly on it; a shadow ray decides visibility.  The emitter is then reachable two ways — by
// this light sample and by the surface's own direction sample happening to hit it — and both are kept with
// balance-heuristic weights p / (p_light + p_bsdf) (densities per solid angle), which keeps the estimate bounded next to
// a large emitter.  Same expectation as the reference's estimator: emission is the material's power (roughness slot,
// Raytracing.cl:105-109) from both faces, the diffuse factor is color / pi and the glossy one 3.14 / pi x BRDF_GGX, which
// is what the reference's samplers converge to.  The test-side CPU restatement mirrors the statement order.

// density per solid angle with which the light sampler reaches the point at squared distance dist2 along unit direction
// wi on emitter triangle (A, e1, e2); 0 when the triangle is seen edge-on
RT_DEV float light_pdf(v3 e1, v3 e2, int n_light, v3 wi, float dist2) {
  const v3 NL = cross(e1, e2);
  const float area2 = sqrtf(dot(NL, NL));
  const float cosL = fabsf(dot(NL, wi)) / area2;
  if (!(cosL > 0.0f) || !(area2 > 0.0f)) return 0.0f;
  return dist2 / ((cosL * ((float)n_light * 0.5f)) * area2);
}

// density per solid angle with which the surface's own sampler draws unit direction l (m.type 1 or 2)
RT_DEV float bsdf_pdf(const Material &m, int sampling, v3 un, v3 d_in, v3 l) {
  const float kPi = 3.14159265f;
  const float ndl = dot(un, l);
  if (m.type == 1) return fmaxf(ndl, 0.0f) / kPi;
  if (sampling & 1) return glossy_mix_pdf(m.roughness, un, unit(neg3(d_in)), l);
  return ndl > 0.0f ? 1.0f / (2.0f * kPi) : 0.0f;
}

// the weighted contribution of one light sample seen from surface point x (throughput `acc` before this surface's own
// factor); *w_out is the shadow ray's direction (y - x, so the emitter lies at parameter 1)
RT_DEV v3 sample_light(const Material &m, int sampling, v3 n, v3 un, v3 x, v3 d_in, v3 acc, v3 A, v3 e1, v3 e2, float Le,
                       int n_light, float ua, float ub, v3 *w_out) {
  const float kPi = 3.14159265f;
  if (ua + ub > 1.0f) { ua = 1.0f - ua; ub = 1.0f - ub; }
  const v3 y = (A + (e1 * ua)) + (e2 * ub);
  const v3 w = y - x;
  const float dist2 = dot(w, w);
  const float dist = sqrtf(dist2);
  const v3 wi = w / dist;
  const float cosS = dot(wi, un);
  v3 fr;
  if (m.type == 1) {
    fr = m.color * (1.0f / kPi);
  } else {
    fr = bsdf_ggx(m, neg3(d_in), wi, n) * (3.14f / kPi);
  }
  *w_out = w;
  if (!(cosS > 0.0f) || !(dist2 > 0.0f)) return mk3(0.0f, 0.0f, 0.0f);
  const float pl = light_pdf(e1, e2, n_light, wi, dist2);
  if (!(pl > 0.0f)) return mk3(0.0f, 0.0f, 0.0f);
  const float pb = bsdf_pdf(m, sampling, un, d_in, wi);
  return (acc * fr) * ((cosS * Le) / (pl + pb));
}

}  // namespace b200rt
