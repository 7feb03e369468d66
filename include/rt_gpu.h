/* rt_gpu.h — additive C ABI of libraytracer_gpu.so (plain C, no Codin and no
 * torch types).  The five reference entry points live in raytracer.h and
 * denoiser.h; everything here is what a GPU back end needs in addition:
 * telling the library which host callbacks it replaces, uploading the scene
 * once, parity hooks, and a device-pointer level for hosts that own the device
 * memory themselves (bench.py wraps torch allocations and NCCL around it).
 *
 * Every call returns 0 on success, non-zero on failure, with the text in
 * rt_gpu_last_error().  There is no CPU fallback: without a CUDA device every
 * compute call fails.
 */
#ifndef RT_GPU_H
#define RT_GPU_H

#include "raytracer.h"
#include "denoiser.h"
#include "rt_pbr.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- lifecycle ----
 * One process drives one device (rt_gpu_init) or several (rt_gpu_init_devices): with N devices the
 * raytracer.h entry points split every frame over them (see RT_GPU_Options.split_mode), the per-device f32
 * accumulators are combined on devices[0] — by one fused reduce+resolve kernel that reads the peers'
 * buffers over NVLink, or by an NCCL reduce (RT_GPU_Options.reduce_mode) — and devices[0] resolves,
 * denoises and returns the image.  The reference has no counterpart: its driver starts N host threads
 * (driver.c:793-803); here `--gpus N` of the host program maps to this call. */
int         rt_gpu_init(int device);              /* = rt_gpu_init_devices(1, &device); idempotent per device */
int         rt_gpu_init_devices(int n_devices, int const *devices);   /* devices NULL = ordinals 0..n-1 */
int         rt_gpu_device_count(void);            /* devices this process drives (0 before init) */
int         rt_gpu_visible_devices(void);         /* CUDA devices visible to the process */
void        rt_gpu_shutdown(void);
char const *rt_gpu_last_error(void);
/* 0 = the most recent raytracer.h / denoiser.h entry-point call on this process succeeded; non-zero = it
 * failed (text in rt_gpu_last_error).  Those entry points return void (reference raytracer.h:51-56), so a
 * host checks this after rendering_context_finish / denoise_image. */
int         rt_gpu_last_status(void);
int         rt_gpu_sm_count(void);
/* Measured issue rate of non-fused FP32 multiply/add in lane-operations per second:
 * the roofline denominator for the trace kernel (csrc/rt_peak.cu). */
f64         rt_gpu_measure_fp32_issue(void);

/* Optional: allocate what a frame of this size needs (accumulators, path-queue workspace on every device) now, e.g.
 * on the thread that created the contexts while the model is still loading. */
int         rt_gpu_prepare_frame(isize width, isize height, isize samples, isize max_bounces);

/* ---- callbacks the device code internalises ----
 * Replaces the per-triangle Shader.proc indirect call (reference scene.h:30-35,
 * raytracer.c:535) and Scene.background.proc (scene.h:65-70, raytracer.c:554).
 * A triangle whose proc was not registered makes the upload fail. */
void rt_gpu_register_pbr_shader(Shader_Proc proc);      /* Shader.data is a PBR_Shader_Data*  */
void rt_gpu_register_background(Background_Proc proc);  /* Background.data is an Image* (equirect) */
/* Ready-made identities for hosts that have no CPU shader of their own; calling
 * them on the CPU aborts (there is no CPU path). */
void   rt_gpu_pbr_shader_proc(rawptr data, Shader_Input const *in, Shader_Output *out);
Color3 rt_gpu_background_proc(rawptr image, Vec3 direction);

/* ---- scene residency: upload once, keyed by the Scene pointer ----
 * The upload is asynchronous: nodes and triangles go first, textures and the environment follow on a copy
 * stream while the first primary trace already runs; host buffers in pinned memory (rt_gpu_host_alloc) are
 * DMA-read in place, pageable ones pass through a pinned staging ring.  The host buffers must stay alive
 * and unchanged until the next render of the scene has started or rt_gpu_scene_release was called.
 * A host that rebuilds a Scene at the same address (scene_init again) is detected by the buffer pointers
 * and sizes and re-uploaded; one that rewrites buffers in place must call rt_gpu_scene_upload again. */
int  rt_gpu_scene_upload(Scene const *scene);
/* pinned host memory for scene buffers and textures (plug into the host's allocator: H2D then needs no staging) */
void *rt_gpu_host_alloc(size_t bytes);
void  rt_gpu_host_free(void *p);
isize rt_gpu_scene_device_bytes(Scene const *scene);   /* bytes resident for this scene, 0 if absent */
isize rt_gpu_scene_upload_bytes(Scene const *scene);   /* bytes its upload copied host -> device */
void rt_gpu_scene_release(Scene const *scene);

/* ---- options for the raytracer.h entry points ---- */
enum { RT_GPU_SPLIT_AUTO = 0, RT_GPU_SPLIT_SAMPLES = 1, RT_GPU_SPLIT_CHUNKS = 2 };
enum { RT_GPU_REDUCE_P2P = 0, RT_GPU_REDUCE_NCCL = 1 };
typedef struct {
  u32   user_seed;        /* rt_seed.h; default 0 */
  i32   sample_begin;     /* render samples [begin, end) of ctx->samples.  With sample_range_set == 0, */
  i32   sample_end;       /* end 0 = all; with sample_range_set != 0 the range is taken literally (may be empty) */
  i32   slice_samples;    /* samples per progress slice of render_thread_proc (one wavefront chunk never spans
                           * slices); 0 (default) = as many as one chunk of path queues holds */
  i32   keep_hit_ids;     /* record the primary-hit slot of sample `sample_begin` */
  i32   sample_range_set;
  i32   split_mode;       /* N devices: RT_GPU_SPLIT_* — sample ranges in multiples of the 8-sample jitter batch
                           * (raytracer.c:641-697), or the reference's 32x32 chunks dealt round-robin
                           * (raytracer.c:619-637); AUTO = samples when the batches divide evenly, else chunks */
  i32   reduce_mode;      /* N devices: RT_GPU_REDUCE_* */
  i32   pixel_rank;       /* multi-PROCESS hosts: this process renders the 32x32 chunks congruent to */
  i32   pixel_world;      /* pixel_rank modulo pixel_world (<= 1: the whole image) */
  i32   fast_math;        /* 0 (default): every sample bit-identical to the reference arithmetic.  1: the bounce
                           * stages (trace of bounce >= 1, environment, BSDF) run FMA-contracted with hardware
                           * transcendentals (csrc/rt_render_fast.cu); primary-hit ids, ray generation and the film
                           * stay exact.  Faster, statistically equivalent, NOT bit-identical. */
} RT_GPU_Options;
void rt_gpu_set_options(RT_GPU_Options const *options);
void rt_gpu_get_options(RT_GPU_Options *options);

/* ---- parity hooks: results of the LAST render_thread_proc on this process ---- */
enum {
  RT_GPU_CTR_RAYS = 0, RT_GPU_CTR_NODES, RT_GPU_CTR_LEAVES, RT_GPU_CTR_ACCEPTS,
  RT_GPU_CTR_SHADES, RT_GPU_CTR_MISSES, RT_GPU_CTR_PASSTHROUGH, RT_GPU_CTR_SAMPLES,
};
int rt_gpu_read_accum(f32 *out, isize n_floats);       /* W*H*3 sums of cast_ray, pre-division */
int rt_gpu_read_hit_ids(i32 *out, isize n_pixels);     /* padded slot or -1 */
int rt_gpu_read_counters(u64 out[8]);
/* RGBA8 texels of texture `slot` of a resident scene (first device); out may be NULL to query the size */
int rt_gpu_read_texture(Scene const *scene, i32 slot, u8 *out, isize *width, isize *height);
/* the library's own 16-slot device counter block (first device): slots [0..8) as above, [8] rays whose whole walk
 * was the root-union test, [9] primary rays; pass it as d_counters to the device-level calls to get [8..16) filled */
int rt_gpu_counters_buffer(u64 **d_counters_out);
int rt_gpu_counters_reset(void);                       /* synchronises, then zeroes that block */
int rt_gpu_read_counters_ex(u64 out[16]);              /* all 16 slots, summed over the devices */
int rt_gpu_last_launches(void);                        /* kernels launched since the last entry-point call began */
f64 rt_gpu_last_kernel_ms(void);                       /* CUDA-event time of the last call's trace kernels */
/* wall-clock pieces of the last render_thread_proc: [0] scene upload issued inside the call (ms, 0 if resident),
 * [1] cross-device reduce + resolve (CUDA events), [2] image D2H + host copy, [3] split mode used */
void rt_gpu_last_frame_breakdown(f64 out[4]);

/* ---- lightmap_bake (raytracer.h:56, reference raytracer.c:722-784) with its parity hooks: values_out (optional, W*H*3 f32)
 * = accumulated / samples of every written texel before the u8 store; owner_out (optional, W*H i32) = the triangle slot
 * that owns each texel, -1 = untouched.  Seeds: rt_seed.h, per (texel, sample); RT_GPU_Options.user_seed applies. ---- */
int rt_gpu_lightmap_bake(Image const *lightmap, Scene const *scene, isize samples, f32 *values_out, i32 *owner_out);

/* ---- how a frame is split over `world` devices or processes (pure host arithmetic, no device needed) ----
 * Sample split: batches of 8 samples dealt as evenly as possible; ranks beyond the number of batches get an
 * empty range.  Returns the mode AUTO resolves to for this (samples, world). */
void rt_gpu_shard_samples(i32 rank, i32 world, i32 samples, i32 *begin, i32 *end);
i32  rt_gpu_shard_mode(i32 samples, i32 world, i32 requested_mode);
/* 32x32 chunks rank `rank` owns under the chunk split */
i32  rt_gpu_shard_chunks(i32 rank, i32 world, isize width, isize height);

/* ---- per-stage kernel timing (measurement harness): when enabled, every kernel of a render is
 *      bracketed by CUDA events on its launching stream; read = synchronise + sum since enable.
 *      Stages: 0 trace (closest hit), 1 miss (environment), 2 shade (BSDF), 3 accumulate. ---- */
void rt_gpu_stage_profile_enable(i32 on);
int  rt_gpu_stage_profile_read(f64 ms[4], i64 launches[4]);
/* the same split by bounce: slot = stage * 16 + min(bounce, 15) */
int  rt_gpu_stage_profile_read_bounces(f64 ms[64], i64 launches[64]);

/* ---- device-pointer level (all pointers are device memory; stream is a
 *      cudaStream_t passed as void*, NULL = the legacy default stream) ---- */
int rt_gpu_render_accum_device(Scene const *scene, isize width, isize height,
                               isize sample_begin, isize sample_end, isize max_bounces,
                               u32 user_seed, i32 accumulate,
                               f32 *d_accum,          /* W*H*3 */
                               f32 *d_per_sample,     /* optional W*H*(end-begin)*3 */
                               i32 *d_hit_ids,        /* optional W*H */
                               u64 *d_counters,       /* optional 8, atomically added */
                               void *stream);
/* The same for one shard of a frame split over `world` processes (one per GPU): the library picks the split
 * (RT_GPU_SPLIT_*; returns the mode used in *mode_used) and renders this rank's share of `samples` into d_accum,
 * which is zero outside the share, so the sum over ranks is the frame. */
int rt_gpu_render_shard_device(Scene const *scene, isize width, isize height, isize samples, isize max_bounces,
                               u32 user_seed, i32 rank, i32 world, i32 split_mode, i32 *mode_used,
                               f32 *d_accum, u64 *d_counters, void *stream);
/* Cross-process film: library-owned accumulator (cudaMalloc, exportable), CUDA-IPC handles, and the fused
 * reduce + resolve over peer-mapped accumulators (parts[0..n) summed in that order; d_sum_out and d_pixels optional). */
int rt_gpu_accum_buffer(isize width, isize height, f32 **d_accum_out);
int rt_gpu_ipc_export(void const *d_ptr, u8 handle_out[64]);
int rt_gpu_ipc_open(u8 const handle[64], void **d_ptr_out);
int rt_gpu_reduce_resolve_device(f32 const *const *d_parts, i32 n_parts, f32 *d_sum_out, isize width, isize height,
                                 isize samples, u8 *d_pixels, isize stride, i32 components, void *stream);
int rt_gpu_resolve_device(f32 const *d_accum, isize width, isize height, isize samples,
                          u8 *d_pixels, isize stride, i32 components, void *stream);
int rt_gpu_denoise_device(u8 const *d_src, u8 *d_dst, isize width, isize height,
                          isize src_stride, isize dst_stride, i32 components, void *stream);

/* ---- ray queries on a resident scene (csrc/rt_query.cu) ----
 * A query is the reference's ray_scene_hit (raytracer.c:443-503) with hit.distance set to t_max before the walk:
 *   - a ray is the reference's Ray (24 B, f32 alignment).  Directions are not normalised; t is in units of
 *     |direction|, as in the reference;
 *   - a triangle counts when it passes the Moller-Trumbore test of raytracer.c:115-159 with EPSILON <= t < t_max
 *     (strict).  t_max is per ray; a NULL t_max array means +inf for every ray.  A t_max that is NaN, negative or
 *     <= EPSILON gives a miss: that is what the reference's compares give, with no special case;
 *   - the walk visits nodes in the reference's order with its compares and tie rules, so the closest hit (ties
 *     included) is the reference's triangle slot.
 * Closest hit: t, the barycentrics u, v of the hit and the padded triangle slot (the numbering of rt_gpu_read_hit_ids:
 * scene->triangles.aos[slot] is the triangle).  A miss is t = +inf, u = v = 0, slot = -1.  The optional surface
 * record is raytracer.c:164-182 in the f32 expressions the renderer uses: point = o + d * t, the interpolated
 * shading normal (not normalised, as in the reference), the geometric normal and the interpolated texture
 * coordinates; all zero for a miss.
 * Occlusion: one byte per ray, 1 = some triangle counts.  It is the same ordered walk, stopped at the first leaf
 * that accepts a triangle.  Until that acceptance hit.distance is still t_max, so the occlusion walk is a prefix of
 * the closest-hit walk with the same t_max: occluded[i] == (closest hit of ray i has slot >= 0) exactly, and its
 * node, leaf and accept counts never exceed those of the closest-hit query.
 * Queries are always exact: RT_GPU_Options.fast_math does not apply to them.
 * They run on the first device, do not wait for the scene's textures (only for its geometry), and do not serialise
 * against renders; two queries on one device are serialised by the library (they share a work counter). */
typedef struct { f32 t, u, v; i32 slot; } RT_GPU_Hit;                                   /* 16 B */
typedef struct { Vec3 point, normal, normal_geo; Vec2 tex_coords; } RT_GPU_Surface;     /* 44 B */
/* device pointers, stream-ordered (stream: cudaStream_t as void*, NULL = the legacy default stream).  d_hits must be
 * 16-byte aligned; d_t_max, d_surface and d_counters are optional.  d_counters: four u64, atomically added, as
 * RT_GPU_CTR_RAYS / NODES / LEAVES / ACCEPTS.  n_rays in [0, INT32_MAX]; 0 is a no-op. */
int rt_gpu_closest_hit_device(Scene const *scene, Ray const *d_rays, f32 const *d_t_max, isize n_rays,
                              RT_GPU_Hit *d_hits, RT_GPU_Surface *d_surface, u64 *d_counters, void *stream);
int rt_gpu_occluded_device(Scene const *scene, Ray const *d_rays, f32 const *d_t_max, isize n_rays,
                           u8 *d_occluded, u64 *d_counters, void *stream);
/* host memory: staged through library-owned device buffers, queried, copied back; returns when the results are in
 * place.  t_max and surface are optional. */
int rt_gpu_closest_hit(Scene const *scene, Ray const *rays, f32 const *t_max, isize n_rays,
                       RT_GPU_Hit *hits, RT_GPU_Surface *surface);
int rt_gpu_occluded(Scene const *scene, Ray const *rays, f32 const *t_max, isize n_rays, u8 *occluded);

/* ---- radiance for caller rays on a resident scene (csrc/rt_render.cu) ----
 * The reference's cast_ray (raytracer.c:505-558) for a batch of n_rays rays, each traced for `samples` samples with
 * sample indices sample_begin + s, s in [0, samples):
 *   - a ray is the reference's Ray (24 B, f32 alignment), as for the queries.  Directions are used as given: the
 *     renderer normalises its camera rays, cast_ray itself does not;
 *   - path (i, s) is cast_ray(scene, ray_i, max_bounces) with the shader generator seeded to
 *     rt_path_seed(key_i, sample_begin + s, user_seed) just before the call (rt_seed.h, the renderer's rule).  key_i is
 *     keys[i], or i when keys is NULL.  Results therefore depend neither on the order of the batch nor on how it is
 *     split into calls; a host that passes the renderer's camera ray of (pixel p, sample s) with key p gets the
 *     renderer's radiance of that sample bit for bit;
 *   - radiance[i] (3 f32) is the sum over the samples in sample order, before any division (the meaning of
 *     rt_gpu_read_accum).  With accumulate != 0 the sums continue from what the buffer holds, so samples [0, k) then
 *     [k, n) equal [0, n) bit for bit.  With samples == 0 nothing is traced: radiance is zeroed unless accumulate
 *     is set, in which case it is left as it is (as rt_gpu_render_accum_device does with an empty range);
 *   - per_sample (optional, [n_rays][samples][3] f32) receives each path's radiance, as the renderer's per-sample output;
 *   - d_counters (optional, 8 u64, atomically added) as RT_GPU_CTR_*; SAMPLES grows by n_rays * samples;
 *   - NaN radiance is summed as the renderer sums it (there is no film here, so the film's NaN -> 0 does not apply);
 *   - max_bounces = 0 gives zero radiance for every path, as cast_ray does.
 * Always exact: RT_GPU_Options.fast_math does not apply.  First device only.  The call shades, so it waits for the
 * scene's texels as well as its geometry; it uses the device's path-queue workspace, so it is serialised with renders
 * and lightmap bakes on that device (not with ray queries).  A batch larger than one workspace chunk is split over rays
 * and samples inside the call.
 * Refused before any launch: n_rays outside [0, INT32_MAX], samples < 0, sample_begin < 0,
 * sample_begin + samples > INT32_MAX, max_bounces < 0, NULL rays or radiance with n_rays > 0, a scene that is not
 * resident (rt_gpu_scene_upload).  n_rays = 0 is a no-op. */
int rt_gpu_cast_rays_device(Scene const *scene, Ray const *d_rays, u32 const *d_keys, isize n_rays, isize sample_begin,
                            isize samples, isize max_bounces, u32 user_seed, i32 accumulate,
                            f32 *d_radiance,          /* n_rays*3 */
                            f32 *d_per_sample,        /* optional n_rays*samples*3 */
                            u64 *d_counters,          /* optional 8 */
                            void *stream);
/* host memory: staged through library-owned device buffers; returns when the results are in place */
int rt_gpu_cast_rays(Scene const *scene, Ray const *rays, u32 const *keys, isize n_rays, isize sample_begin, isize samples,
                     isize max_bounces, u32 user_seed, i32 accumulate, f32 *radiance, f32 *per_sample);

/* ---- first-surface AOVs of the renderer's camera samples on a resident scene (csrc/rt_render.cu) ----
 * Per-pixel buffers aligned with the beauty image: what surface each sample of the renderer's path (pixel p, sample s)
 * shades first, for s in [sample_begin, sample_end), with max_bounces:
 *   1. the camera ray of (p, s) is the one the renderer traces, from the scene's current camera as a render reads it;
 *   2. while the hit is a back face (dot(ng, d) > 0 || dot(normal, d) > 0, raytracer.c:516-522) and fewer than
 *      max_bounces walks have been made, the walk continues from point + d * EPSILON, as the renderer's path does;
 *   3. the first front-face hit within max_bounces walks is the sample's surface: where the path runs its first shader.
 *      A sample that escapes, or uses up its walks on back faces, has no surface.
 * Values at the surface are the renderer's f32 expressions:
 *   albedo    the base colour the BSDF receives: base_color times the sRGB-decoded albedo texel where there is one;
 *   normal    the shading normal handed to the BSDF: the normalised interpolated normal, normal-mapped where the
 *             material has a normal map;
 *   position  o + d * t of the last walk (the shaded point);
 *   depth     sqrt((position - eye) . (position - eye)), eye the camera origin: three products summed left to right,
 *             one IEEE square root;
 *   emission  the emission the shader returns (emission times the decoded emissive texel);
 *   roughness, metalness  after their texture, the clamp and min(., 0.9) / 0.9;
 *   coverage  1.
 * A sample with no surface adds nothing to any field.  Nothing random happens before a path's first shade (the jitter
 * is a hash of pixel and sample, the back-face step is deterministic, the material fetch draws no random numbers), so
 * every record is exact per (pixel, sample), with no seed; NaN values (a degenerate interpolated normal) are summed as
 * they come.
 * aov[y * width + x] holds the SUMS over the samples in sample order, before any division (the meaning of
 * rt_gpu_read_accum): divide by coverage for the mean over covered samples, or by the sample count.  With
 * accumulate != 0 the sums continue from what the buffer holds, so [0, k) then [k, n) equals [0, n) bit for bit.  With
 * an empty range or max_bounces = 0 nothing is traced: the records are zeroed unless accumulate is set, in which case
 * they are left as they are, and the counters are not touched.
 * d_counters (optional, 8 u64, atomically added) as RT_GPU_CTR_*: RAYS, NODES, LEAVES, ACCEPTS of every walk; SHADES =
 * samples with a surface; MISSES = walks that escaped; PASSTHROUGH = back-face hits; SAMPLES = W * H * (end - begin).
 * Always exact: RT_GPU_Options.fast_math does not apply, and pixel_rank / pixel_world do not either (the call covers the
 * whole image).  First device only.  The call reads texels, so it waits for the scene's texels as well as its geometry;
 * it uses the device's path-queue workspace and rewrites the camera-relative scene copies, so it is serialised with
 * renders, lightmap bakes and cast_rays on that device.
 * Refused before any launch: width or height < 1, or an image whose one sample per pixel exceeds 2^31 path ids;
 * sample_begin < 0, sample_end < sample_begin, sample_end > INT32_MAX; max_bounces < 0; a NULL record buffer, or
 * (device form) one that is not 16-byte aligned; a scene that is not resident (rt_gpu_scene_upload). */
typedef struct {
  Vec3 albedo;   f32 coverage;
  Vec3 normal;   f32 depth;
  Vec3 position; f32 roughness;
  Vec3 emission; f32 metalness;
} RT_GPU_AOV;                                   /* 64 B: four 16-byte vectors per pixel */
int rt_gpu_render_aov_device(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                             isize max_bounces, i32 accumulate,
                             RT_GPU_AOV *d_aov,       /* W*H, 16-byte aligned */
                             u64 *d_counters,         /* optional 8 */
                             void *stream);
/* host memory: staged through a library-owned device buffer, from zero; returns when the records are in place */
int rt_gpu_render_aov(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                      isize max_bounces, RT_GPU_AOV *aov);

/* ---- adaptive sampling: masked sample passes and a film for per-pixel sample counts (csrc/rt_render.cu) ----
 * rt_gpu_render_masked_device renders samples [sample_begin, sample_end) of the pixels d_mask selects, by the
 * renderer's own camera paths.  The library supplies the mechanism; the host keeps the policy (which pixels have
 * converged, how many samples a pass takes, when to stop).
 *   - mask: W*H bytes, row-major; non-zero = render the pixel.  NULL = every pixel.
 *   - radiance: for a selected pixel p and sample s the path is the renderer's path (p, s): the same camera ray, the
 *     seed rt_path_seed(p, s, user_seed) and the same per-sample radiance as rt_gpu_render_accum_device.  d_accum[p]
 *     (3 f32) is the sum in sample order, before any division.
 *   - second moment (d_accum_sq, optional, W*H*3 f32): the per-channel sum of v * v in sample order; the product is
 *     rounded, then the add (IEEE f32 without contraction: numpy float32 reproduces it).
 *   - accumulate = 0: every pixel of d_accum, and of d_accum_sq if given, is written: selected pixels get their sums
 *     from zero, the others 0 (as the shard call is zero outside its share).  accumulate != 0: selected pixels continue
 *     from the buffers, the others are not touched.
 *   - an empty range or max_bounces = 0 is handled as the renderer handles it: nothing is traced or counted, and the
 *     buffers are zeroed unless accumulate is set, in which case they are left as they are.
 *   - d_counters (optional, 8 u64, atomically added) as RT_GPU_CTR_*, over the selected paths only: SAMPLES grows by
 *     (selected pixels) * (end - begin).
 *   - RT_GPU_Options.fast_math applies exactly as it does to rt_gpu_render_accum_device: the call is the renderer with
 *     a mask.  pixel_rank / pixel_world do not apply (the call covers the whole image).  First device only.
 * Key property: because every path is seeded per (pixel, sample) and the sums continue in sample order, after passes
 * that cover samples [0, n_p) of pixel p, chained with accumulate, d_accum[p] and d_accum_sq[p] equal a uniform render
 * of [0, n_p) at that pixel bit for bit, whatever the passes in between selected elsewhere.
 * Ordering: the call uses the device's path-queue workspace and rewrites the camera-relative scene copies, so it is
 * serialised with renders, lightmap bakes, cast_rays and AOV calls on that device; like a render it waits for the
 * scene's geometry before its primary trace and for its texels after it.
 * Refused before any launch: width or height < 1, or an image whose one sample per pixel exceeds 2^31 path ids;
 * sample_begin < 0, sample_end < sample_begin, sample_end > INT32_MAX; max_bounces < 0; a NULL d_accum; a scene that
 * is not resident (rt_gpu_scene_upload). */
int rt_gpu_render_masked_device(Scene const *scene, isize width, isize height,
                                u8 const *d_mask,        /* optional W*H, row-major: non-zero = render; NULL = every pixel */
                                isize sample_begin, isize sample_end, isize max_bounces, u32 user_seed, i32 accumulate,
                                f32 *d_accum,            /* W*H*3 */
                                f32 *d_accum_sq,         /* optional W*H*3 */
                                u64 *d_counters,         /* optional 8 */
                                void *stream);
/* The film with a sample count per pixel: reference raytracer.c:700-716 with samples = d_samples[pixel].  Each channel
 * is sum * (1.0f / (f32)n), clamped, sRGB-encoded and truncated to u8, as rt_gpu_resolve_device does; a count <= 0
 * gives 0 bytes and a NaN sum gives 0.  With every count equal to n the bytes equal rt_gpu_resolve_device(..., n, ...).
 * Refused: a NULL d_samples, components < 3. */
int rt_gpu_resolve_counts_device(f32 const *d_accum, i32 const *d_samples, isize width, isize height,
                                 u8 *d_pixels, isize stride, i32 components, void *stream);

/* ---- many views of a resident scene in one call (csrc/rt_render.cu) ----
 * rt_gpu_render_views_device renders samples [sample_begin, sample_end) of n_views whole images of one scene, view v
 * from cameras[v], into slice v of d_accum ([n_views][H][W][3] f32).  After its primary trace a path no longer depends
 * on the camera it came from, so each view runs its own primary trace (with the camera-relative copies and sky tiles
 * of its camera) and every bounce launch is shared by the views: the renderer's fixed cost per call (launches, the
 * tails of the late bounces) is paid once per call rather than once per view.
 * Key property: slice v of d_accum equals, bit for bit,
 *   rt_gpu_render_accum_device(scene, width, height, sample_begin, sample_end, max_bounces,
 *                              user_seeds ? user_seeds[v] : 0, accumulate, ...)
 * called with scene->camera = cameras[v], whatever the other views are, their number and order, and however the call is
 * split into chunks inside.  The counters gain the sum of those per-view calls' counters, the extended slots [8..16)
 * included when the library's own block (rt_gpu_counters_buffer) is passed.
 *   - cameras: a host array; only the fields the renderer reads are used, rows 0..2 of view_matrix and focal_length.
 *     scene->camera is neither read nor written by the call: a render after it uses scene->camera as before.
 *   - seeds: view v's path (p, s) is seeded rt_path_seed(p, s, user_seeds[v]), the renderer's rule; NULL user_seeds =
 *     0 for every view.  Pass distinct seeds for views whose noise should not be correlated.
 *   - accumulate behaves per view as for a render: the sums continue from each slice, so [0, k) then [k, n) equals
 *     [0, n).  An empty range or max_bounces = 0 traces and counts nothing and zeroes every slice unless accumulate is
 *     set.  n_views = 0 is a no-op.
 *   - RT_GPU_Options.fast_math applies as it does to a render (each view equals the fast single render); pixel_rank /
 *     pixel_world do not apply (each view is a whole image).  First device only.
 * Ordering: like a render, the call uses the device's path-queue workspace and rewrites the camera-relative scene
 * copies, so it is serialised with renders, lightmap bakes, cast_rays and AOV calls on that device; it waits for the
 * scene's geometry before its first primary trace and for its texels after it.
 * Refused before any launch: width or height < 1, or an image whose one sample per pixel exceeds 2^31 path ids;
 * sample_begin < 0, sample_end < sample_begin, sample_end > INT32_MAX; max_bounces < 0; n_views < 0; NULL cameras with
 * n_views > 0; a NULL d_accum (device form) or both outputs NULL (host form); a scene that is not resident
 * (rt_gpu_scene_upload).  No camera a render accepts is refused. */
/* device pointers on the first device, ordered on `stream` (cudaStream_t as void*, NULL = the legacy default stream) */
int rt_gpu_render_views_device(Scene const *scene, i32 n_views,
                               Camera const *cameras,   /* host array [n_views] */
                               u32 const *user_seeds,   /* optional host array [n_views]; NULL = 0 for every view */
                               isize width, isize height, isize sample_begin, isize sample_end, isize max_bounces,
                               i32 accumulate,
                               f32 *d_accum,            /* [n_views][H][W][3] */
                               u64 *d_counters,         /* optional 8 (16 with the library's own block) */
                               void *stream);
/* host memory: staged through the device's staging block, from zero; accum ([n_views][H][W][3] f32) and pixels
 * ([n_views][H][W][3] u8, the film of rt_gpu_resolve_device with samples = sample_end - sample_begin; black when the
 * range is empty) are each optional, but not both NULL; returns when the results are in place */
int rt_gpu_render_views(Scene const *scene, i32 n_views, Camera const *cameras, u32 const *user_seeds,
                        isize width, isize height, isize sample_begin, isize sample_end, isize max_bounces,
                        f32 *accum, u8 *pixels);

/* ---- moving geometry on a resident scene: refit the BVH and triangle records on the device (csrc/rt_refit.cu) ----
 * A refit keeps the topology scene_init chose (which triangle sits in which slot, which child is which) and recomputes,
 * from new vertex positions, everything that depends on them, with host/scene_build.c's f32 expressions:
 *   - per occupied slot: the vertex arrays, the edges, the geometric normal, tangent and bitangent (pack_leaf), and the
 *     vertex normals when given; UVs and materials are kept;
 *   - per node child: the union of the subtree's triangle boxes inflated by EPSILON, exactly as scene_init computes it;
 *     a child with no triangle keeps its all-zero box;
 *   - the root-union box the renderer's sky tiles and root shortcut use.
 * So refitting unchanged positions reproduces scene_init's bytes, and every render, query, AOV call and lightmap bake
 * afterwards equals the same call on a host Scene built with the new positions under the same topology.  The boxes are
 * exact, but under large motion they overlap more and tracing slows down: when to rebuild with scene_init is the host's
 * choice.
 * Occupancy is the upload's: a slot is a triangle when its Triangle_AOS had a shader at upload.  Inputs of padding
 * slots are ignored; those slots stay zero.
 * Ordering: the refit waits on the device for every earlier render, lightmap bake, cast_rays, AOV, masked pass and
 * query of the scene, and every later one waits for the refit; no caller needs a synchronisation of its own.  With
 * several devices the peers receive the result over NVLink.
 * The call SYNCHRONISES with the host before it returns (it reads back a validation flag and the root node).
 * Refused, with the resident scene unchanged: a scene that is not resident (rt_gpu_scene_upload), NULL positions, a
 * non-finite coordinate in an occupied slot. */
/* device pointers on the first device, ordered on `stream` (cudaStream_t as void*, NULL = the legacy default stream).
 * d_positions: f32[9][n_slots], the Scene's own block order x0 x1 x2 y0 y1 y2 z0 z1 z2; d_normals (optional):
 * f32[n_slots][3][3], normal_a, normal_b, normal_c of each slot (Triangle_AOS order), NULL = keep.  The host buffers are
 * not touched: a later rt_gpu_scene_upload, or the re-upload of a Scene whose buffers changed, replaces a device-only
 * refit with what the host buffers hold. */
int rt_gpu_scene_refit_device(Scene const *scene, f32 const *d_positions, f32 const *d_normals, void *stream);
/* host form: the host has rewritten scene->triangles.x/y/z (and, with refit_normals, aos[s].normal_a/b/c) in slot
 * order.  They are staged as the upload stages them (pinned memory in place, pageable through the staging ring), refit
 * on the device, and the refit node boxes and each occupied slot's normal, tangent and bitangent are written back into
 * scene->bvh.nodes.data and scene->triangles.aos; padding slots' positions (and normals) are zeroed.  Afterwards the host
 * Scene is exactly what the device holds, for a CPU reference, a scene-cache save or a later re-upload. */
int rt_gpu_scene_refit(Scene *scene, i32 refit_normals);
/* parity hook: the node bytes resident on the first device (n_internal * 192 B into out) */
int rt_gpu_read_nodes(Scene const *scene, BVH_Node *out);

#ifdef __cplusplus
}
#endif
#endif
