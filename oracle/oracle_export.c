/* oracle_export.c — TEST INFRASTRUCTURE.  Exported doors to header-only pieces
 * (rt_math.h, rt_seed.h) and to single steps of the oracle so unit tests can
 * pin them one at a time. */
#include "oracle.h"
#include "oracle_vec.h"
#include "rt_seed.h"
#include <immintrin.h>

f32 oracle_powf(f32 x, f32 y)    { return rt_powf(x, y); }
f32 oracle_sinf(f32 x)           { return rt_sinf(x); }
f32 oracle_cosf(f32 x)           { return rt_cosf(x); }
f32 oracle_atan2f(f32 y, f32 x)  { return rt_atan2f(y, x); }
f32 oracle_asinf(f32 x)          { return rt_asinf(x); }
u32 oracle_path_seed(u32 pixel, u32 sample, u32 user_seed) { return rt_path_seed(pixel, sample, user_seed); }
u32 oracle_rand_u32(u32 *state)  { return rt_rand_u32(state); }
f32 oracle_rand_f32(u32 *state)  { return rt_rand_f32(state); }

void oracle_powf_array(f32 const *x, f32 y, f32 *out, isize n) { for (isize i = 0; i < n; i++) out[i] = rt_powf(x[i], y); }
void oracle_powf_positive_array(f32 const *x, f32 y, f32 *out, isize n) { for (isize i = 0; i < n; i++) out[i] = rt_powf_positive(x[i], y); }
void oracle_pow5_array(f32 const *x, f32 *out, isize n) { for (isize i = 0; i < n; i++) out[i] = rt_pow5f(x[i]); }
void oracle_sincos_array(f32 const *x, f32 *s, f32 *c, isize n) { for (isize i = 0; i < n; i++) { s[i] = rt_sinf(x[i]); c[i] = rt_cosf(x[i]); } }
void oracle_sincos_fused_array(f32 const *x, f32 *s, f32 *c, isize n) { for (isize i = 0; i < n; i++) rt_sincosf(x[i], &s[i], &c[i]); }
void oracle_atan2_array(f32 const *y, f32 const *x, f32 *out, isize n) { for (isize i = 0; i < n; i++) out[i] = rt_atan2f(y[i], x[i]); }
void oracle_asin_array(f32 const *x, f32 *out, isize n) { for (isize i = 0; i < n; i++) out[i] = rt_asinf(x[i]); }

/* _mm256_rsqrt_ps, which raytracer.c:663 uses for primary rays: its bits are the CPU's choice, not IEEE's, so a
 * reference-seed-mode image recorded on one CPU holds on another only where this array comes out the same. */
void oracle_rsqrt_ps_array(f32 const *x, f32 *out, isize n) {
  for (isize i = 0; i < n; i += 8) {
    f32 in[8] = {1, 1, 1, 1, 1, 1, 1, 1}, res[8];
    for (isize k = 0; k < 8 && i + k < n; k++) in[k] = x[i + k];
    _mm256_storeu_ps(res, _mm256_rsqrt_ps(_mm256_loadu_ps(in)));
    for (isize k = 0; k < 8 && i + k < n; k++) out[i + k] = res[k];
  }
}

/* Primary ray of sample s at pixel (x, y): raytracer.c:644-677 with the exact
 * 1/sqrt (the form the parity mode uses on both sides). */
Ray oracle_primary_ray(Camera const *cam, isize width, isize height, isize x, isize y, isize s) {
  f32 inv_w = 1.0f / (f32)width, inv_h = 1.0f / (f32)height, aspect = (f32)width / (f32)height;
  f32 jit = oracle_hash12((f32)x * 50.0f + (f32)s, (f32)y);
  f32 ux = ((f32)x + jit - 0.5f) * 2.0f * inv_w - 1.0f;
  f32 uy = ((f32)y + jit - 0.5f) * 2.0f * inv_h - 1.0f;
  f32 cx = ux * aspect, cy = -uy, cz = -cam->focal_length;
  f32 inv_len = 1.0f / RT_SQRT_F32(cx * cx + cy * cy + cz * cz);
  f32 const (*m)[4] = cam->view_matrix.rows;
  Ray r;
  r.position  = v3(m[0][3], m[1][3], m[2][3]);
  r.direction = v3((m[0][0] * cx + m[0][1] * cy + m[0][2] * cz) * inv_len,
                   (m[1][0] * cx + m[1][1] * cy + m[1][2] * cz) * inv_len,
                   (m[2][0] * cx + m[2][1] * cy + m[2][2] * cz) * inv_len);
  return r;
}
