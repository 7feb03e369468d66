/* camera_rays.c — TEST INFRASTRUCTURE.  The renderer's camera ray of (pixel, sample), as rays a host would hand to
 * rt_gpu_cast_rays: the oracle's camera-ray lines (oracle/oracle_trace.c:335-374, the reference's raytracer.c:644-677
 * with rand_a == rand_b) restated one lane at a time with the exact 1/sqrt.
 *
 * Build: gcc -O2 -ffp-contract=off -shared -fPIC -I include (no contraction: every product and sum rounds separately,
 * as in the oracle's 8-wide code and on the GPU with -fmad=false).
 */
#include <math.h>

#include "raytracer.h"

/* raytracer.c:582-594, one lane of hash12x8 */
static inline f32 fractf(f32 v) { return v - floorf(v); }
static f32 hash12(f32 px, f32 py) {
  f32 a = fractf(px * 0.1031f);
  f32 b = fractf(py * 0.1031f);
  f32 c = fractf(px * 0.1031f);
  f32 k = 33.33f;
  f32 d = a * (b + k) + b * (c + k) + c * (a + k);
  return fractf((a + b + d * 2.0f) * (c + d));
}

/* out[(y * width + x) * 6 ..] = (eye, direction) of sample `sample` at pixel (x, y) of a width x height frame */
void camera_rays(Camera const *cam, isize width, isize height, isize sample, f32 *out) {
  f32 inv_width = 1.0f / (f32)width, inv_height = 1.0f / (f32)height, aspect = (f32)width / (f32)height;
  f32 const (*m)[4] = cam->view_matrix.rows;
  for (isize y = 0; y < height; y++) {
    for (isize x = 0; x < width; x++) {
      f32 jit = hash12((f32)x * 50.0f + (f32)sample, (f32)y);
      f32 ux = ((f32)x + jit - 0.5f) * 2.0f * inv_width - 1.0f;
      f32 uy = ((f32)y + jit - 0.5f) * 2.0f * inv_height - 1.0f;
      f32 cx = ux * aspect, cy = -uy, cz = -cam->focal_length;
      f32 inv_len = 1.0f / sqrtf(cx * cx + cy * cy + cz * cz);
      f32 *r = out + (y * width + x) * 6;
      r[0] = m[0][3]; r[1] = m[1][3]; r[2] = m[2][3];
      r[3] = (m[0][0] * cx + m[0][1] * cy + m[0][2] * cz) * inv_len;
      r[4] = (m[1][0] * cx + m[1][1] * cy + m[1][2] * cz) * inv_len;
      r[5] = (m[2][0] * cx + m[2][1] * cy + m[2][2] * cz) * inv_len;
    }
  }
}
