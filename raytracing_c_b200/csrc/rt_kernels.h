// rt_kernels.h — launch wrappers shared between the kernel translation units and
// the C-ABI layer (rt_cabi.cu).  Each returns a cudaError_t value as int.
#pragma once

#include <cuda_runtime.h>
#include "rt_device.cuh"

// wavefront render of samples [p.sample_begin, p.sample_end) into p.accum; `workspace` holds the path queues
// (rt_render_workspace_bytes; a smaller one only means more, smaller chunks).  *n_launches += kernels launched.
// With p.pixel_mask and/or p.accum_sq the primary trace and the accumulate run their masked builds: only the selected
// pixels are rendered (the others are zeroed without p.accumulate, untouched with it) and the second moments are summed.
size_t rt_render_workspace_bytes(int width, int height, int n_samples, int max_bounces, int split_world);
int rt_render_chunk_samples(int width, int height, int split_world);
unsigned rt_render_tiles(int width, int height, int split_rank, int split_world);
int rt_launch_render(const RenderParams &p, int sm_count, void *workspace, size_t workspace_bytes,
                     cudaStream_t stream, int *n_launches);
// lightmap_bake (raytracer.c:722-784) on the wavefront: see rt_render.cu.  `scratch` holds rt_lightmap_workspace_bytes,
// `workspace` the path queues: rt_lightmap_paths_workspace_bytes for n_texels * samples paths at the preferred chunk
// size, or with `floor` the smallest one the bake asks for (one sample of every texel)
size_t rt_lightmap_workspace_bytes(int width, int height);
size_t rt_lightmap_paths_workspace_bytes(size_t n_texels, int samples, int max_bounces, bool floor);
int rt_launch_lightmap(const SceneDev &scene, int width, int height, int samples, int max_bounces, uint32_t user_seed,
                       unsigned char *d_pixels, int stride, int components, float *d_values, int *d_owner_out,
                       void *scratch, int sm_count, void *workspace, size_t workspace_bytes, cudaStream_t stream,
                       int *n_launches, unsigned *n_jobs_out);
// cast_ray (raytracer.c:505-558) for caller rays on the wavefront, samples [sample_begin, sample_begin + samples) of each
// ray summed into radiance (see rt_render.cu); `workspace` holds the path queues: rt_cast_rays_workspace_bytes for
// n_rays * samples paths at the preferred chunk size, or with `floor` the smallest one the launch accepts
size_t rt_cast_rays_workspace_bytes(size_t n_paths, int max_bounces, bool floor);
int rt_launch_cast_rays(const SceneDev &scene, const float *rays, const unsigned *keys, int n_rays, int sample_begin,
                        int samples, int max_bounces, uint32_t user_seed, int accumulate, float *radiance, float *per_sample,
                        unsigned long long *counters, int sm_count, void *workspace, size_t workspace_bytes,
                        cudaStream_t stream, int *n_launches);
// first-surface AOVs of the renderer's camera samples [sample_begin, sample_end), whole image, summed per pixel into aov
// (W*H records of 16 floats, 16-byte aligned; see rt_render.cu).  The workspace is the renderer's
// (rt_render_workspace_bytes with split_world 1)
int rt_launch_aov(const SceneDev &scene, int width, int height, int sample_begin, int sample_end, int max_bounces,
                  int accumulate, float *aov, unsigned long long *counters, int sm_count, void *workspace,
                  size_t workspace_bytes, cudaStream_t stream, int *n_launches);
int rt_launch_resolve(const float *accum, int width, int height, int samples, unsigned char *pixels,
                      int stride, int components, cudaStream_t stream);
// the film with a sample count per pixel (samples[W*H]; a count <= 0 gives 0 bytes)
int rt_launch_resolve_counts(const float *accum, const int *samples, int width, int height, unsigned char *pixels,
                             int stride, int components, cudaStream_t stream);
// sum of parts.n accumulators (own + peer-mapped) in rank order, optional copy of the sum, optional resolve to u8
int rt_launch_reduce_resolve(const ReduceParts &parts, float *sum_out, int width, int height, int samples,
                             unsigned char *pixels, int stride, int components, cudaStream_t stream);
int rt_launch_denoise(const unsigned char *src, unsigned char *dst, int width, int height,
                      int src_stride, int dst_stride, int components, cudaStream_t stream);
int rt_render_blocks_per_sm(void);
// RGB8 / RGBA8 rows (stride in pixels) -> tightly packed RGBA8 texels
int rt_launch_texel_repack(const unsigned char *src, int width, int height, int stride, int components,
                           uchar4 *dst, cudaStream_t stream);
// RGBA8 texels -> float4 (r, g, b, 0) / 255.999f: the environment's second copy (TextureDev.texels_f32)
int rt_launch_texel_expand(const uchar4 *src, size_t n, float4 *dst, cudaStream_t stream);
// tri_pos / tri_rec from the host's vertex arrays, Triangle_AOS records and per-slot material indices (rt_denoise.cu)
int rt_launch_scene_pack(const float *soa, const float4 *aos, const int *mat_index, int n_slots, float4 *tri_pos, float4 *tri_rec,
                         cudaStream_t stream);
// ray queries (rt_query.cu): closest hit (any = false: hits, optional surface) or occlusion (any = true: occluded)
// of n_rays rays at their own index; `fetch` is a zeroed work counter no other launch uses at the same time
struct QueryParams {
  SceneDev  scene;
  const float *rays;                     // [n_rays][6]: the reference's Ray (position, direction)
  const float *t_max;                    // optional [n_rays], NULL = +inf
  unsigned  n_rays;
  float4   *hits;                        // [n_rays] (t, u, v, slot bits)
  float    *surface;                     // optional [n_rays][11]: point, normal, normal_geo, tex_coords
  unsigned char *occluded;               // [n_rays]
  unsigned *fetch;
  unsigned long long *counters;          // optional 4: rays, nodes, leaves, accepts
};
int rt_launch_query(const QueryParams &p, bool any, int sm_count, cudaStream_t stream);
// per-stage CUDA-event timing of rt_launch_render's kernels (off by default)
// slot = stage * RT_STAGE_BOUNCES + min(bounce, RT_STAGE_BOUNCES - 1)
enum { RT_STAGE_TRACE = 0, RT_STAGE_MISS, RT_STAGE_SHADE, RT_STAGE_ACCUMULATE, RT_N_STAGES, RT_STAGE_BOUNCES = 16 };
void rt_stage_profile_enable(int on, int device);
int  rt_stage_profile_read(double ms[RT_N_STAGES * RT_STAGE_BOUNCES], long long launches[RT_N_STAGES * RT_STAGE_BOUNCES]);
