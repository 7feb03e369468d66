/* oracle.h — TEST INFRASTRUCTURE.  CPU restatement of the reference's hot path.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load liboracle.so.  Nothing under
 * raytracing_c_b200/ links or calls it.
 *
 * PARITY STATUS: the reference has no tests, fixtures or golden vectors
 * (SURVEY.md §4) and cannot be built as shipped (its stdlib "Codin" is not
 * vendored).  This oracle is pinned against the reference's own raytracer.c /
 * scene.c / denoiser.c / driver.c compiled unmodified, from where they lie
 * in a reference checkout (RT_REFERENCE_DIR), over a Codin shim (oracle/codin_shim, recipe
 * oracle/Makefile target `ref`, output oracle/_ref/libref.so) — see
 * tests/test_oracle_vs_ref.py and the committed fixtures under tests/golden/.
 * The shim itself carries the UNPINNED Codin choices listed in DESIGN.md.
 *
 * Each function cites the reference file:line it follows.
 */
#ifndef ORACLE_H
#define ORACLE_H

#include "raytracer.h"
#include "denoiser.h"
#include "rt_pbr.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- scene build (reference scene.c:78-242,311-426) ---- */
void oracle_scene_init(Scene *scene, Triangle_Slice src_triangles);
void oracle_scene_destroy(Scene *scene);

/* ---- shading callbacks (reference driver.c:49-409) ---- */
void   oracle_disney_shader_proc(rawptr data, Shader_Input const *in, Shader_Output *out);
Color3 oracle_sample_background(rawptr image, Vec3 direction);
Color3 oracle_sample_texture_bilinear(Image const *texture, Vec2 tex_coords);
/* The shader TU's thread-local generator state (reference common.h:13). */
u32   *oracle_shader_random_state(void);

/* ---- render (reference raytracer.c:443-720) ---- */
enum {
  ORACLE_SEED_REFERENCE = 0,  /* stream starts at 0 per thread, runs across pixels */
  ORACLE_SEED_PER_SAMPLE = 1, /* rt_path_seed(pixel, sample, user_seed) before each cast_ray */
};

typedef struct {
  i32   seed_mode;
  u32   user_seed;
  i32   approx_rsqrt;     /* 1 = _mm256_rsqrt_ps as raytracer.c:663; 0 = exact 1/sqrt */
  i32   sample_begin;     /* render samples [sample_begin, sample_end) of ctx->samples */
  i32   sample_end;       /* 0 = ctx->samples */
  f32  *accum;            /* optional W*H*3: sum over samples of cast_ray (pre-division) */
  f32  *per_sample;       /* optional W*H*(end-begin)*3 radiance of each sample */
  i32  *hit_ids;          /* optional W*H: padded slot of sample `sample_begin`'s primary hit, -1 = miss */
  u64   counters[8];      /* out: see ORACLE_CTR_* (summed over threads) */
  u8 const *pixel_mask;   /* optional W*H: only pixels with a non-zero byte are rendered (per-(pixel,sample) seeds make any
                           * subset independent: this is how full-size frames are spot-checked in seconds) */
} Oracle_Options;

enum {
  ORACLE_CTR_RAYS = 0, ORACLE_CTR_NODES, ORACLE_CTR_LEAVES, ORACLE_CTR_ACCEPTS,
  ORACLE_CTR_SHADES, ORACLE_CTR_MISSES, ORACLE_CTR_PASSTHROUGH, ORACLE_CTR_SAMPLES,
};

/* Runs the reference's chunk scheduler on n_threads OS threads and joins. */
void oracle_render(Rendering_Context *ctx, Oracle_Options *opt, i32 n_threads);

/* cast_ray (raytracer.c:505-558) for one ray with the shader generator in its current state. */
Color3 oracle_cast_ray(Scene const *scene, Ray ray, isize max_bounces);

/* ---- lightmap_bake (raytracer.c:722-784), see oracle_lightmap.c ---- */
typedef struct {
  i32  seed_mode;        /* ORACLE_SEED_* */
  u32  user_seed;
  u32  dir_state;        /* in/out (reference mode): raytracer.c's generator copy, feeds rand_vec3 */
  u32  shader_state;     /* in/out (reference mode): driver.c's generator copy, feeds the BSDF */
  f32 *values;           /* optional W*H*3: accumulated / samples of every written texel, before the u8 store */
  i32 *owner;            /* optional W*H: triangle slot that wrote the texel last (caller pre-fills with -1) */
  i64  texels_written;   /* out: stores, overlaps counted each time */
} Oracle_Lightmap_Options;
void oracle_lightmap_bake(Image const *lightmap, Scene const *scene, isize samples, Oracle_Lightmap_Options *opt);

/* One ray through the traversal only: returns padded slot or -1; *t_out = distance. */
i32 oracle_trace_ray(Scene const *scene, Ray ray, f32 *t_out);

/* hash12 jitter (reference raytracer.c:582-594), one lane. */
f32 oracle_hash12(f32 px, f32 py);

/* ---- denoiser (reference denoiser.c:12-149) ---- */
void oracle_denoise_image(Image const *src, Image const *dst, isize n_threads);

/* ---- film (reference raytracer.c:700-716, common.h:90-92) ---- */
void oracle_resolve(f32 const *accum, isize n_pixels, isize samples, u8 *rgb_out);

#ifdef __cplusplus
}
#endif
#endif
