// rt_shade.cuh — per-lane shading: manual bilinear texture fetch, equirect
// environment lookup, normal mapping and the Disney-style diffuse + GGX-VNDF
// specular + sheen sampler.
//
// Behavioural contract (operation order included — results must equal the CPU
// oracle bit for bit): reference driver.c:49-104 (sampler, environment),
// :118-183 (hemisphere sample, normal map, frame, sheen), :200-348 (BRDF),
// :350-409 (material fetch and glue); common.h:82-88 (sRGB decode by pow only,
// AFTER filtering).  The reference reaches this code through a host function
// pointer per triangle; here it is a direct call with a material-table index.
// f32/f64 promotions follow the reference's literals (driver.c:119,214,220,
// 238,241-246,263,313): PI is a double.
#pragma once

#include "rt_device.cuh"

// Exact build (default): rt_math.h transcendentals and the reference's f64 promotions, bit-identical to the CPU oracle.
// RT_FAST build (rt_render_fast.cu, opt-in): hardware approximations (MUFU lg2/ex2/sin/cos), CUDA's f32 atan2/asin,
// f32 everywhere — a few ulp off per call, and one flipped lobe pick sends a path elsewhere, so the results are
// compared with the oracle statistically (bench.py --fast: parity key), not bit for bit.
#if defined(RT_FAST) && RT_FAST
typedef float rt_real;
#define RT_PI_R 3.14159265358979323846f
__device__ __forceinline__ float m_pow_positive(float x, float y) { return __powf(x, y); }
__device__ __forceinline__ float m_atan2(float y, float x) { return atan2f(y, x); }
__device__ __forceinline__ float m_asin(float x) { return asinf(x); }
__device__ __forceinline__ void  m_sincos(float a, float *s, float *c) { __sincosf(a, s, c); }
#else
typedef double rt_real;
#define RT_PI_R RT_PI
__device__ __forceinline__ float m_pow_positive(float x, float y) { return rt_powf_positive(x, y); }
__device__ __forceinline__ float m_atan2(float y, float x) { return rt_atan2f(y, x); }
__device__ __forceinline__ float m_asin(float x) { return rt_asinf(x); }
__device__ __forceinline__ void  m_sincos(float a, float *s, float *c) { rt_sincosf(a, s, c); }
#endif

// What is inlined where (measured on the helmet, 64-spp chunk, bounce-0 launches): shade_pbr inlined into the shade kernel
// (no ShadeIn / ShadeOut round trip through local memory) 2055 -> 1905 us; the environment lookup and ITS bilinear fetch
// inlined into the miss kernel 1727 -> 1647 us; the bilinear fetch inlined at the shade kernel's four call sites
// 2055 -> 2175 us (code size), so those share one out-of-line copy.
struct ShadeIn  { V3 dir, normal, normal_geo, tangent, bitangent; float u, v; };
struct ShadeOut { V3 dir, tint, emission; bool terminate; };

__device__ __forceinline__ float rnd(uint32_t &state) { return rt_rand_f32(&state); }

// driver.c:69-88: a texel byte b becomes (float)b / 255.999f.  Two instructions per channel, no table: PRMT drops the
// byte into the mantissa of 2^23 (the float 8388608 + b, exact), one fused multiply-add forms (2^23 + b) * k - 2^23 * k
// with k = RN(1 / 255.999f) — the exact sum is b * k, rounded once, and RN(b * k) equals the IEEE quotient for all 256
// bytes (tests/csrc/texel_scale_check.c).
__device__ __forceinline__ float texel_channel(unsigned rgba, unsigned selector) {
  const float k = 1.0f / 255.999f;
  return __fmaf_rn(__uint_as_float(__byte_perm(rgba, 0x4B000000u, selector)), k, -8388608.0f * k);
}
__device__ __forceinline__ V3 texel_rgb(const TextureDev &tex, int x, int y) {
  const unsigned t = __ldg(reinterpret_cast<const unsigned *>(tex.texels) + (x + tex.width * y));
  return mk3(texel_channel(t, 0x7650u), texel_channel(t, 0x7651u), texel_channel(t, 0x7652u));
}

// driver.c:49-93: negative wrap, fract, no half-texel offset, +1 neighbour clamped
__device__ __forceinline__ V3 sample_bilinear_inline(const TextureDev &tex, float u, float v) {
  if (u < 0) u += (float)(-(int)u + 1);
  if (v < 0) v += (float)(-(int)v + 1);
  u = u - floorf(u);
  v = v - floorf(v);
  float px = u * (float)tex.width;
  float py = v * (float)tex.height;
  int x0 = (int)px, y0 = (int)py;
  float a = px - (float)x0, b = py - (float)y0;
  int x1 = (x0 + 1 < tex.width)  ? x0 + 1 : x0;
  int y1 = (y0 + 1 < tex.height) ? y0 + 1 : y0;
  if (tex.texels_f32) {                 // the environment: texels already divided (rt_device.cuh)
    const float4 *row0 = tex.texels_f32 + (size_t)tex.width * y0, *row1 = tex.texels_f32 + (size_t)tex.width * y1;
    const float4 t00 = __ldg(row0 + x0), t10 = __ldg(row0 + x1), t01 = __ldg(row1 + x0), t11 = __ldg(row1 + x1);
    V3 top = lerp3(mk3(t00.x, t00.y, t00.z), mk3(t10.x, t10.y, t10.z), a);
    V3 bot = lerp3(mk3(t01.x, t01.y, t01.z), mk3(t11.x, t11.y, t11.z), a);
    return lerp3(top, bot, b);
  }
  V3 top = lerp3(texel_rgb(tex, x0, y0), texel_rgb(tex, x1, y0), a);
  V3 bot = lerp3(texel_rgb(tex, x0, y1), texel_rgb(tex, x1, y1), a);
  return lerp3(top, bot, b);
}

static __device__ __noinline__ V3 sample_bilinear(const TextureDev &tex, float u, float v) {
  return sample_bilinear_inline(tex, u, v);
}

// common.h:82-88.  The argument of the power is >= 0.055 / 1.055 (texel values are >= 0), so the
// case analysis of rt_powf can be skipped: rt_powf_positive is bit-identical there.
// x / 1.055f in three instructions instead of the general division's twelve: the quotient estimate x * r
// (r = RN(1 / 1.055f)), its exact residual by one fused multiply-add, one correction.  Equal to the IEEE quotient
// for EVERY binary32 x in [0.01, 4] (tests/csrc/div_const_check.c tries them all); the decode sees [0.055, 1.055].
__device__ __forceinline__ float div_1p055(float x) {
#if defined(RT_FAST) && RT_FAST
  return x * (1.0f / 1.055f);
#else
  const float r = 1.0f / 1.055f;
  const float q = x * r;
  return __fmaf_rn(__fmaf_rn(-1.055f, q, x), r, q);
#endif
}
__device__ __forceinline__ V3 decode_srgb(V3 c) {
  return mk3(m_pow_positive(div_1p055(c.x + 0.055f), 2.4f),
             m_pow_positive(div_1p055(c.y + 0.055f), 2.4f),
             m_pow_positive(div_1p055(c.z + 0.055f), 2.4f));
}

// driver.c:95-104 (asin argument clamped: DESIGN.md deviation list)
__device__ __forceinline__ V3 environment(const SceneDev &sc, V3 dir) {
  float inv_pi     = (float)(1.0f / RT_PI_R);
  float inv_two_pi = (float)(1.0f / (2.0f * RT_PI_R));
  float u = 0.5f + m_atan2(dir.z, dir.x) * inv_two_pi;
  float v = 0.5f - m_asin(clamp1(dir.y, -1.0f, 1.0f)) * inv_pi;
  return decode_srgb(sample_bilinear_inline(sc.textures[sc.env_texture], u, v));
}

__device__ __forceinline__ float luma(V3 c) { return dot3(c, mk3(0.2126f, 0.7152f, 0.0722f)); }

// driver.c:204-210
// pow_f32(x, 5) and pow_f32(x, 2) of the reference: rt_pow5f / x * x are what rt_powf returns for them
__device__ __forceinline__ float schlick1(float f0, float f90, float c) { return f0 + (f90 - f0) * rt_pow5f(1 - c); }

// driver.c:212-215
__device__ __forceinline__ float ggx_d(float roughness, float n_h) {       // k = 2 at both call sites
  float a2 = roughness * roughness;
  float b  = (n_h * n_h) * (a2 * a2 - 1) + 1;
  return (float)(a2 / (RT_PI_R * (b * b)));
}

// driver.c:217-221
__device__ __forceinline__ float smith_g1(float n_v, float alpha2) {
  float a = alpha2 * alpha2;
  float b = n_v * n_v;
  return (float)(((rt_real)2.0 * n_v) / (n_v + __fsqrt_rn(a + b - a * b)));
}

// driver.c:118-127
__device__ __forceinline__ V3 cosine_hemisphere(uint32_t &rng) {
  float angle  = (float)(rnd(rng) * 2 * RT_PI_R);
  float radius = __fsqrt_rn(rnd(rng));
  V3 d;
  float sn, cs;
  m_sincos(angle, &sn, &cs);
  d.x = sn * radius;
  d.y = cs * radius;
  d.z = __fsqrt_rn(1 - radius * radius);
  return d;
}

// driver.c:230-250
__device__ __forceinline__ V3 sample_vndf(V3 V, float ax, float ay, uint32_t &rng) {
  V3 Vh = normalize3(mk3(ax * V.x, ay * V.y, V.z));
  float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
  V3 T1 = lensq > 0 ? scale3(mk3(-Vh.y, Vh.x, 0), 1.0f / __fsqrt_rn(lensq)) : mk3(1, 0, 0);
  V3 T2 = cross3(Vh, T1);

  float r   = __fsqrt_rn(rnd(rng));
  float phi = (float)((rt_real)2.0 * RT_PI_R * rnd(rng));
  float sn, cs;
  m_sincos(phi, &sn, &cs);
  float t1  = r * cs;
  float t2  = r * sn;
  float s   = (float)((rt_real)0.5 * ((rt_real)1.0 + Vh.z));
  t2        = (float)(((rt_real)1.0 - s) * __fsqrt_rn((float)((rt_real)1.0 - t1 * t1)) + s * t2);

  rt_real rem = (rt_real)1.0 - t1 * t1 - t2 * t2;
  float   h   = __fsqrt_rn((float)((rt_real)0.0 > rem ? (rt_real)0.0 : rem));
  V3 Nh = add3(add3(scale3(T1, t1), scale3(T2, t2)), scale3(Vh, h));
  return normalize3(mk3(ax * Nh.x, ay * Nh.y, (0.0 > Nh.z ? 0.0f : Nh.z)));
}

// driver.c:166-183
__device__ __forceinline__ V3 sheen_term(float sheen, V3 base, float sheen_tint, float h_dot_l) {
  if (sheen <= 0.0f) return mk3(0, 0, 0);
  float lum = dot3(mk3(0.3f, 0.6f, 1.0f), base);
  V3 tint = (lum > 0.0f) ? scale3(base, 1.0f / lum) : mk3(1, 1, 1);
  float m = 1 - h_dot_l;
  float w = m * m * m * m * m;
  return scale3(lerp3(mk3(1, 1, 1), tint, sheen_tint), sheen * w);
}

// driver.c:129-153,350-367: the material fetch — what the BSDF receives at a surface: the shading normal (normal-mapped
// where the material has a map), the base colour after the albedo texture, roughness and metalness after their texture,
// clamp and rescale, and the emission.  No random numbers are drawn.  shade_pbr and the first-surface AOVs
// (rt_render.cu) both evaluate it here, so the AOVs are what the shader saw.
__device__ __forceinline__ void pbr_surface(const SceneDev &sc, const MaterialDev &mat, const ShadeIn &in, V3 &n, V3 &base,
                                            float &roughness, float &metalness, V3 &glow) {
  // driver.c:129-153
  n = in.normal;
  if (mat.tex_normal >= 0) {
    V3 s = sample_bilinear(sc.textures[mat.tex_normal], in.u, in.v);
    s = add3(scale3(s, 2.0f), mk3(-1, -1, -1));
    s.y *= -1;
    V3 t = in.tangent, b = in.bitangent;
    float k = mat.normal_strength;
    n = normalize3(mk3(k * (s.x * t.x + s.y * b.x + s.z * n.x) + n.x * (1 - k),
                       k * (s.x * t.y + s.y * b.y + s.z * n.y) + n.y * (1 - k),
                       k * (s.x * t.z + s.y * b.z + s.z * n.z) + n.z * (1 - k)));
  }

  base = mk3(mat.base[0], mat.base[1], mat.base[2]);
  if (mat.tex_albedo >= 0) base = mul3(base, decode_srgb(sample_bilinear(sc.textures[mat.tex_albedo], in.u, in.v)));

  roughness = mat.roughness; metalness = mat.metalness;
  if (mat.tex_mr >= 0) {
    V3 mr = sample_bilinear(sc.textures[mat.tex_mr], in.u, in.v);
    roughness *= mr.y;
    metalness *= mr.z;
  }
  roughness = clamp1(roughness, 0.001f, 1);
  if (metalness > 0.9f) metalness = 0.9f;
  metalness /= 0.9f;

  glow = mk3(mat.emission[0], mat.emission[1], mat.emission[2]);
  if (mat.tex_emission >= 0) {
    // emissive maps are mostly black, and a black bilinear tap decodes to one constant (common.h:82-88 has no linear toe:
    // pow(0.055 / 1.055, 2.4)) — sc.srgb_of_zero holds it, evaluated once by the same rt_math.h code, so a warp whose
    // taps are all black skips its three pow
    const V3 e = sample_bilinear(sc.textures[mat.tex_emission], in.u, in.v);
    const bool black = (e.x == 0.0f) & (e.y == 0.0f) & (e.z == 0.0f);
    const V3 lin = black ? mk3(sc.srgb_of_zero, sc.srgb_of_zero, sc.srgb_of_zero) : decode_srgb(e);
    glow = mul3(glow, lin);
  }
}

// driver.c:350-409 with :287-348 inlined
__device__ __forceinline__ void shade_pbr(const SceneDev &sc, int material, const ShadeIn &in, uint32_t &rng, ShadeOut &out) {
  const MaterialDev &mat = sc.materials[material];
  V3 n, base, glow;
  float roughness, metalness;
  pbr_surface(sc, mat, in, n, base, roughness, metalness, glow);
  out.emission = glow;
  out.terminate = false;
  out.tint = mk3(0, 0, 0);

  // driver.c:155-164
  V3 t, b;
  if (fabsf(dot3(n, in.dir)) < 0.9999f)             t = normalize3(cross3(n, in.dir));
  else if (fabsf(dot3(n, mk3(0, 1, 0))) < 0.9999f)  t = normalize3(cross3(n, mk3(0, 1, 0)));
  else                                              t = normalize3(cross3(n, mk3(1, 0, 0)));
  b = cross3(n, t);

  V3 minus_d = scale3(in.dir, -1);
  V3 wi = mk3(dot3(t, minus_d), dot3(b, minus_d), dot3(n, minus_d));

  // driver.c:287-348
  float aniso2  = mat.aniso * mat.aniso;
  float alpha_x = lerp1(roughness * roughness, 1, aniso2);
  float alpha_y = roughness * roughness;
  V3 h = sample_vndf(wi, alpha_x, alpha_y, rng);

  V3 f0 = lerp3(mk3(0.04f, 0.04f, 0.04f), base, metalness);
  float f90 = sel_min(1.0f, (1.0f / 0.04f) * luma(f0));
  V3 F = add3(f0, scale3(sub3(mk3(f90, f90, f90), f0), rt_pow5f(1 - dot3(wi, h))));

  float w_diff = 1 - metalness;
  float w_spec = luma(F);
  float inv_w  = 1 / (w_diff + w_spec);
  w_diff *= inv_w;
  w_spec *= inv_w;

  V3 wo;
  float fx = 0, fy = 0, fz = 0, fw = 0;
  if (rnd(rng) < w_diff) {
    wo = cosine_hemisphere(rng);
    h = normalize3(add3(wo, wi));
    float n_l = wo.z, n_v = wi.z;
    if (!(n_l <= 0 || n_v <= 0)) {
      float l_h = dot3(wo, h);
      float pdf = (float)(n_l / RT_PI_R);
      float fd90 = 0.5f + 2 * roughness * l_h * l_h;
      float fa = schlick1(1.0f, fd90, n_l);
      float fb = schlick1(1.0f, fd90, n_v);
      V3 diff = scale3(base, (float)(fa * fb / RT_PI_R));
      diff = mul3(diff, sub3(mk3(1, 1, 1), F));
      diff = add3(diff, sheen_term(mat.sheen, base, mat.sheen_tint, l_h));
      fx = diff.x * n_l; fy = diff.y * n_l; fz = diff.z * n_l;
      fw = w_diff * pdf;
    }
  } else {
    V3 mwi = scale3(wi, -1);
    wo = sub3(mwi, scale3(h, 2.0f * dot3(mwi, h)));
    float n_l = wo.z, n_v = wi.z;
    if (!(n_l <= 0 || n_v <= 0)) {
      n_l = sel_max(n_l, 0.001f);
      n_v = sel_max(n_v, 0.001f);
      float n_h = sel_min(h.z, 0.99f);
      float a2  = roughness * roughness;
      float pdf = (ggx_d(roughness, n_h) * smith_g1(n_v, a2)) / sel_max(0.00001f, 4.0f * n_v);
      float D = ggx_d(roughness, n_h);
      float G = smith_g1(n_v, a2) * smith_g1(n_l, a2);
      V3 spec = scale3(F, D * G / (4 * n_l * n_v));
      fx = spec.x * n_l; fy = spec.y * n_l; fz = spec.z * n_l;
      fw = w_spec * pdf;
    }
  }
  // the early `return vec4(0)` paths at driver.c:309-311,328-330 skip the final
  // normalize; the direction is unused then because the path terminates
  wo = normalize3(wo);

  out.dir = mk3(t.x * wo.x + b.x * wo.y + n.x * wo.z,
                t.y * wo.x + b.y * wo.y + n.y * wo.z,
                t.z * wo.x + b.z * wo.y + n.z * wo.z);
  if (fw > 0) out.tint = mk3(fx / fw, fy / fw, fz / fw);
  else        out.terminate = true;
}
