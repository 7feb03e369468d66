// rt_render.cu — the path-tracing kernels for sm_100a, wavefront form.
//
// Replaces render_thread_proc's pixel loop and everything under it (reference
// raytracer.c:443-558 traversal + cast_ray, :582-594 jitter hash, :596-720 chunk
// loop, camera, film) — see DESIGN.md for the mapping.
//
// Execution model.  cast_ray's bounce loop (raytracer.c:512-556) is unrolled over
// KERNELS instead of running inside one thread, so every kernel is small enough
// for the instruction cache and runs one kind of work with full warps:
//
//   chunk of S samples x all pixels = N paths, path id = ((tile*S + s)*32 + pixel-in-8x4-tile)
//   trace<primary>   generate camera ray (raytracer.c:644-677), closest hit  -> HIT queue | MISS queue
//   for bounce b = 0 .. max_bounces-1:
//     trace          (b > 0) RAY queue -> closest hit                         -> HIT queue | MISS queue
//     miss           environment * tint + emission (raytracer.c:554)          -> rad[path]
//     shade          back-face pass-through (:516-522) or BSDF (:524-552)     -> RAY queue | rad[path]
//   accumulate       accum[pixel] += rad[path(pixel, s)] in sample order      (raytracer.c:696-700)
//
// Queues are structure-of-float4 arrays in HBM; a record moves WITH its path
// (warp-aggregated atomic append), so every stage reads and writes coalesced
// 16-byte vectors and rays stay compacted.  Queue lengths live on the device: all
// launches of a chunk are enqueued back to back without a host round trip, each
// kernel is a persistent grid that strides over "whatever the previous stage produced".
// Queue ORDER is not deterministic, results are: a path's arithmetic depends only on
// its own record, and the per-pixel sum is taken afterwards in sample order, so the f32
// accumulator equals the sequential CPU loop bit for bit.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <vector>

#include "rt_stages.cuh"
#include "rt_kernels.h"

// rt_render_fast.cu: the same bounce-stage kernels compiled with FMA contraction and hardware transcendentals
void rt_fast_launch_trace(const StageParams &P, unsigned grid, size_t smem, cudaStream_t stream, bool wide);
void rt_fast_launch_miss(const StageParams &P, unsigned grid, cudaStream_t stream);
void rt_fast_launch_shade(const StageParams &P, unsigned grid, cudaStream_t stream);
void rt_fast_launch_sky(const StageParams &P, unsigned grid, cudaStream_t stream);
int  rt_fast_trace_setup(size_t level_bytes, int *wide_blocks_per_sm);

// ------------------------------------------------------------ camera-relative scene
// All primary rays start at the camera origin o (raytracer.c:612).  Everything in the slab and
// triangle tests that depends on o but not on the direction — (plane - o) per node, and per triangle
// tv = o - p0, qv = tv x e1, e2 . qv (raytracer.c:123-135) — is evaluated here once per render with the
// same f32 expressions the per-ray code uses, so the primary trace reads constants instead.
__global__ void rt_camera_relative_kernel(const SceneDev sc) {
  const float ox = sc.view[0][3], oy = sc.view[1][3], oz = sc.view[2][3];
  const int n_node_floats = sc.n_internal * 48;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_node_floats + sc.n_slots; i += gridDim.x * blockDim.x) {
    if (i < n_node_floats) {
      const int row = (i % 48) / 8;                     // rows: min x y z, max x y z
      const float o = (row % 3 == 0) ? ox : (row % 3 == 1) ? oy : oz;
      sc.nodes_rel[i] = sc.nodes[i] - o;
    } else {
      const int slot = i - n_node_floats;
      const float4 A = sc.tri_pos[3 * slot], B = sc.tri_pos[3 * slot + 1], C = sc.tri_pos[3 * slot + 2];
      const float e1x = A.w, e1y = B.x, e1z = B.y, e2x = B.z, e2y = B.w, e2z = C.x;
      const float tvx = ox - A.x, tvy = oy - A.y, tvz = oz - A.z;
      const float qvx = tvy * e1z - tvz * e1y, qvy = tvz * e1x - tvx * e1z, qvz = tvx * e1y - tvy * e1x;
      sc.tri_rel[4 * slot + 0] = make_float4(tvx, tvy, tvz, e1x);
      sc.tri_rel[4 * slot + 1] = B;
      sc.tri_rel[4 * slot + 2] = make_float4(e2z, qvx, qvy, qvz);
      sc.tri_rel[4 * slot + 3] = make_float4(e2x * qvx + e2y * qvy + e2z * qvz, 0, 0, 0);
    }
  }
}

// ----------------------------------------------------------------- accumulate
// raytracer.c:696-700: color += cast_ray(...) in sample order, one thread per pixel.  MASKED (a masked pass, or one with
// second moments): a pixel P.pixel_mask does not select is written 0 when the call does not accumulate and is left as
// it is otherwise; P.accum_sq (optional) gains v * v per sample alongside the sum (product rounded, then the add).
// With P.tiles: the traced tiles only (the sky kernel sums the others).
template <bool MASKED>
__device__ __forceinline__ void accumulate_pixels(const StageParams &P) {
  const unsigned n = (P.tiles ? P.tiles[0] : P.n_tiles) * 32u;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned tile = i >> 5, in_tile = i & 31u;
    int x0, y0;
    tile_origin(P, P.tiles ? P.tiles[2 + tile] : tile, x0, y0);
    const int px = x0 + (int)(in_tile & 7u), py = y0 + (int)(in_tile >> 3);
    if (px >= P.width || py >= P.height) continue;
    const int pixel = py * P.width + px;
    if (MASKED && P.pixel_mask && !P.pixel_mask[pixel]) {
      if (!P.accumulate) {
        P.accum[3 * pixel + 0] = 0; P.accum[3 * pixel + 1] = 0; P.accum[3 * pixel + 2] = 0;
        if (P.accum_sq) { P.accum_sq[3 * pixel + 0] = 0; P.accum_sq[3 * pixel + 1] = 0; P.accum_sq[3 * pixel + 2] = 0; }
      }
      continue;
    }
    V3 sum = P.accumulate ? mk3(P.accum[3 * pixel], P.accum[3 * pixel + 1], P.accum[3 * pixel + 2]) : mk3(0, 0, 0);
    V3 sq = mk3(0, 0, 0);
    if (MASKED && P.accum_sq && P.accumulate) sq = mk3(P.accum_sq[3 * pixel], P.accum_sq[3 * pixel + 1], P.accum_sq[3 * pixel + 2]);
#if RT_PATH_LAYOUT == 1
    const float4 *r = P.q.rad + (size_t)i * (size_t)P.n_samples;
    const size_t r_step = 1;
#else
    const float4 *r = P.q.rad + ((size_t)tile * (size_t)P.n_samples) * 32 + in_tile;
    const size_t r_step = 32;
#endif
    for (int s = 0; s < P.n_samples; s++) {
      const float4 v = r[(size_t)s * r_step];
      sum = add3(sum, mk3(v.x, v.y, v.z));
      if (MASKED && P.accum_sq) sq = add3(sq, mul3(mk3(v.x, v.y, v.z), mk3(v.x, v.y, v.z)));
      if (P.per_sample) {
        float *dst = P.per_sample + ((size_t)pixel * (size_t)P.per_sample_stride + (size_t)(P.per_sample_offset + s)) * 3;
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z;
      }
    }
    P.accum[3 * pixel + 0] = sum.x;
    P.accum[3 * pixel + 1] = sum.y;
    P.accum[3 * pixel + 2] = sum.z;
    if (MASKED && P.accum_sq) { P.accum_sq[3 * pixel + 0] = sq.x; P.accum_sq[3 * pixel + 1] = sq.y; P.accum_sq[3 * pixel + 2] = sq.z; }
  }
}

__global__ void __launch_bounds__(256)
rt_accumulate_kernel(const __grid_constant__ StageParams P) { accumulate_pixels<false>(P); }

__global__ void __launch_bounds__(256)
rt_accumulate_masked_kernel(const __grid_constant__ StageParams P) { accumulate_pixels<true>(P); }

// ----------------------------------------------------------------------- film
// raytracer.c:700-716 + common.h:90-92: /spp, clamp, sRGB OETF, *255.999, truncate.
__device__ __forceinline__ unsigned char film_u8(float sum, float inv_samples) {
  float v = sum * inv_samples;
  if (v != v) v = 0;
  v = clamp1(v, 0, 1);
  v = (v <= 0.0031308f) ? (12.92f * v) : (1.055f * rt_powf(v, 1.0f / 2.4f) - 0.055f);
  v = v * 255.999f;
  return (unsigned char)v;
}

__global__ void rt_resolve_kernel(const float *__restrict__ accum, int width, int height, float inv_samples,
                                  unsigned char *__restrict__ pixels, int stride, int components) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= width * height) return;
  int x = i % width, y = i / width;
  unsigned char *dst = pixels + (size_t)components * (size_t)(x + y * stride);
  #pragma unroll
  for (int c = 0; c < 3; c++) dst[c] = film_u8(accum[3 * i + c], inv_samples);
}

// the film of a pixel with its own sample count: 1 / samples[i] taken per pixel, a count <= 0 gives 0 bytes
__global__ void rt_resolve_counts_kernel(const float *__restrict__ accum, const int *__restrict__ samples, int width,
                                         int height, unsigned char *__restrict__ pixels, int stride, int components) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= width * height) return;
  int x = i % width, y = i / width;
  const int n = samples[i];
  const float inv_samples = 1.0f / (float)n;
  unsigned char *dst = pixels + (size_t)components * (size_t)(x + y * stride);
  #pragma unroll
  for (int c = 0; c < 3; c++) dst[c] = n > 0 ? film_u8(accum[3 * i + c], inv_samples) : 0;
}

// Multi-GPU film: the per-device accumulators are combined and resolved by ONE kernel on the device that owns
// the image.  parts[k] are device pointers — this device's own buffer and its peers' buffers mapped over NVLink
// (cudaDeviceEnablePeerAccess inside one process, cudaIpcOpenMemHandle across processes) — read with 16-byte loads
// and summed in fixed rank order ((p0 + p1) + p2 ...), so the frame does not depend on which GPU finished first.
// Replaces an ncclReduce into a staging buffer followed by rt_resolve_kernel: no round trip through HBM, no second launch.
// One thread = four pixels = three float4 per part.
__global__ void __launch_bounds__(256)
rt_reduce_resolve_kernel(const ReduceParts parts, float *__restrict__ sum_out, int width, int height, float inv_samples,
                         unsigned char *__restrict__ pixels, int stride, int components) {
  const int n_pixels = width * height;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int first = g * 4;
  if (first >= n_pixels) return;
  float v[12];
  const int n_here = n_pixels - first < 4 ? n_pixels - first : 4;
  if (n_here == 4) {
    #pragma unroll
    for (int q = 0; q < 3; q++) {
      // every part's vector is requested before the first add (a peer's accumulator is a ~2 us round trip over NVLink:
      // the loop over parts, left rolled, waited for each in turn); the sum itself stays in rank order
      float4 t[RT_MAX_PARTS];
      #pragma unroll
      for (int k = 0; k < RT_MAX_PARTS; k++)
        if (k < parts.n) t[k] = reinterpret_cast<const float4 *>(parts.part[k])[3 * g + q];
      float4 s = t[0];
      #pragma unroll
      for (int k = 1; k < RT_MAX_PARTS; k++)
        if (k < parts.n) { s.x += t[k].x; s.y += t[k].y; s.z += t[k].z; s.w += t[k].w; }
      v[4 * q] = s.x; v[4 * q + 1] = s.y; v[4 * q + 2] = s.z; v[4 * q + 3] = s.w;
      if (sum_out) reinterpret_cast<float4 *>(sum_out)[3 * g + q] = s;
    }
  } else {
    for (int j = 0; j < 3 * n_here; j++) {
      float s = parts.part[0][3 * first + j];
      for (int k = 1; k < parts.n; k++) s += parts.part[k][3 * first + j];
      v[j] = s;
      if (sum_out) sum_out[3 * first + j] = s;
    }
  }
  if (!pixels) return;
  for (int j = 0; j < n_here; j++) {
    const int i = first + j, x = i % width, y = i / width;
    unsigned char *dst = pixels + (size_t)components * (size_t)(x + y * stride);
    #pragma unroll
    for (int c = 0; c < 3; c++) dst[c] = film_u8(v[3 * j + c], inv_samples);
  }
}

// ------------------------------------------------------------------- launchers
#define RT_PATH_BYTES ((2 + 3 + 1 + 2) * sizeof(float4))       // ray + hit + miss records and the tint / emission(=rad) state of one path
#define RT_CHUNK_PATHS_MAX (512u << 20)
#define RT_CAST_RAYS_MIN_CHUNK (1u << 16)                      // paths of the smallest workspace a cast_rays call accepts

// queue lengths of bounces 0 .. max_bounces (at least one bounce's worth)
static size_t counts_bytes(int max_bounces) {
  size_t b = (size_t)((max_bounces > 0 ? max_bounces : 1) + 1) * Q_STRIDE * sizeof(unsigned);
  return (b + 255) & ~(size_t)255;
}

// Paths per wavefront chunk.  Every chunk pays a fixed cost: the late bounces hold a few 10^4..10^5 rays and their
// kernels last as long as their slowest warp whatever the chunk's size.  Measured on helmet 1080p x 1024 spp with the
// final kernels of round 2 (128 B per path): 7.00 / 7.16 / 7.25 Gsamples/s at 128 / 256 / 512 Mi paths.  Default
// 512 Mi paths = 69 GB of the 180 GB on the device (a 1080p frame: 256 samples of every pixel per chunk); a device
// that cannot spare it gets smaller chunks (rt_cabi.cu halves the request until it fits).  Path ids are 32-bit: 2^31
// is the ceiling.  RT_GPU_CHUNK_PATHS overrides it (tuning / tests).
static size_t chunk_paths_max() {
  if (const char *e = getenv("RT_GPU_CHUNK_PATHS")) {
    unsigned long long v = strtoull(e, nullptr, 10);
    if (v > (1ull << 31)) v = 1ull << 31;          // path ids and queue lengths are 32-bit
    if (v > 0) return (size_t)v;
  }
  return RT_CHUNK_PATHS_MAX;
}

// samples of every pixel per chunk (n_samples > 0: at most that many)
static size_t chunk_samples(size_t per_sample, int n_samples) {
  size_t s = chunk_paths_max() / per_sample;
  if (s < 1) s = 1;
  if (n_samples > 0 && s > (size_t)n_samples) s = (size_t)n_samples;
  return s;
}

// paths a workspace holds past its queue lengths, at per_path bytes each
static size_t path_capacity(size_t workspace_bytes, int max_bounces, size_t per_path) {
  const size_t cb = counts_bytes(max_bounces);
  return workspace_bytes < cb ? 0 : (workspace_bytes - cb) / per_path;
}

// job tiles (8x4 pixels) one render covers: the whole image, or the 32x32 chunks congruent to split_rank
unsigned rt_render_tiles(int width, int height, int split_rank, int split_world) {
  if (split_world <= 1) return (unsigned)((width + 7) / 8) * (unsigned)((height + 3) / 4);
  const long chunks = (long)((width + 31) / 32) * (long)((height + 31) / 32);
  const long owned = chunks > split_rank ? (chunks - split_rank + split_world - 1) / split_world : 0;
  return (unsigned)owned * 32u;
}

// samples of every pixel one wavefront chunk holds at the preferred queue size
int rt_render_chunk_samples(int width, int height, int split_world) {
  size_t per_sample = (size_t)rt_render_tiles(width, height, 0, split_world) * 32;
  if (per_sample < 32) per_sample = 32;
  return (int)chunk_samples(per_sample, 0);
}

// the tile lists of a render (StageParams.tiles): two counts and one id per job tile
static size_t tile_list_bytes(unsigned n_tiles) { return ((2 + (size_t)n_tiles) * sizeof(unsigned) + 255) & ~(size_t)255; }

size_t rt_render_workspace_bytes(int width, int height, int n_samples, int max_bounces, int split_world) {
  const unsigned tiles = rt_render_tiles(width, height, 0, split_world);
  size_t per_sample = (size_t)tiles * 32;
  if (per_sample < 32) per_sample = 32;
  return tile_list_bytes(tiles) + counts_bytes(max_bounces) + chunk_samples(per_sample, n_samples) * per_sample * RT_PATH_BYTES;
}

// Views per chunk of a many-view call: as many as one sample of each fits the preferred chunk size and `paths` (what the
// workspace holds), at least one.  per_view: the paths of one sample of one view.
static size_t view_group(int n_views, size_t per_view, size_t paths) {
  size_t g = chunk_paths_max() / per_view;
  if (g > paths / per_view) g = paths / per_view;
  if (g < 1) g = 1;
  return g < (size_t)n_views ? g : (size_t)n_views;
}

// The workspace of a many-view call: the views' tile lists, then one chunk of n_samples samples of a group of views at the
// preferred size, or with `floor` one sample of one view.  n_views = 1 is rt_render_workspace_bytes.
size_t rt_render_views_workspace_bytes(int width, int height, int n_views, int n_samples, int max_bounces, bool floor) {
  const unsigned tiles = rt_render_tiles(width, height, 0, 1);
  size_t per_view = (size_t)tiles * 32;
  if (per_view < 32) per_view = 32;
  const size_t per_sample = floor ? per_view : view_group(n_views, per_view, SIZE_MAX) * per_view;
  return tile_list_bytes(tiles) * (size_t)n_views + counts_bytes(max_bounces) +
         chunk_samples(per_sample, floor ? 1 : n_samples) * per_sample * RT_PATH_BYTES;
}

// trace kernels' blocks per SM at the level-store size they were measured for, per device (cudaFuncSetAttribute is per device)
struct TraceOccupancy { size_t level_bytes; int primary, generic, wide, fast, fast_wide, masked, based; };
static TraceOccupancy g_occupancy[RT_MAX_DEVICES];

// what a launcher needs of trace_launch_setup: the device, the level store, and the trace kernels' persistent grids
// (one wave: blocks per SM x SMs)
struct TraceLaunch { int dev; size_t level_bytes; unsigned primary, generic, wide, fast, fast_wide, masked, based; };

// ---- optional per-stage timing (bench.py's roofline leg): CUDA events around every launch, on the
// launching stream; read back and summed by rt_stage_profile_read
struct StageEvent { cudaEvent_t a, b; int stage; };
static bool g_profile = false;
static int  g_profile_device = 0;        // launches on other devices of a multi-device frame are not timed
static std::vector<StageEvent> g_stage_events;
static std::vector<cudaEvent_t> g_event_pool;

static cudaEvent_t pooled_event() {
  if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

struct StageTimer {
  cudaStream_t st; bool on; StageEvent ev;
  StageTimer(int stage, cudaStream_t s, int device) : st(s), on(g_profile && device == g_profile_device) {
    if (on) { ev.a = pooled_event(); ev.b = pooled_event(); ev.stage = stage; cudaEventRecord(ev.a, st); }
  }
  ~StageTimer() { if (on) { cudaEventRecord(ev.b, st); g_stage_events.push_back(ev); } }
};

void rt_stage_profile_enable(int on, int device) {
  g_profile = on != 0;
  g_profile_device = device;
  for (StageEvent &e : g_stage_events) { g_event_pool.push_back(e.a); g_event_pool.push_back(e.b); }
  g_stage_events.clear();
}

int rt_stage_profile_read(double ms[RT_N_STAGES * RT_STAGE_BOUNCES], long long launches[RT_N_STAGES * RT_STAGE_BOUNCES]) {
  for (int i = 0; i < RT_N_STAGES * RT_STAGE_BOUNCES; i++) { ms[i] = 0; launches[i] = 0; }
  for (StageEvent &e : g_stage_events) {
    cudaError_t err = cudaEventSynchronize(e.b);
    if (err != cudaSuccess) return (int)err;
    float t = 0;
    cudaEventElapsedTime(&t, e.a, e.b);
    ms[e.stage] += t;
    launches[e.stage] += 1;
    g_event_pool.push_back(e.a); g_event_pool.push_back(e.b);
  }
  g_stage_events.clear();
  return 0;
}

// the queue lengths, then eight arrays of `paths` records; returns the end of the last array
static char *bind_queues(PathQueues &q, void *workspace, int max_bounces, size_t paths) {
  char *w = static_cast<char *>(workspace);
  q.counts = reinterpret_cast<unsigned *>(w); w += counts_bytes(max_bounces);
  float4 **arrays[] = { &q.ray_a, &q.ray_b, &q.hit_a, &q.hit_b, &q.hit_h, &q.miss_a, &q.tint, &q.emis };
  for (float4 **a : arrays) { *a = reinterpret_cast<float4 *>(w); w += paths * sizeof(float4); }
  q.rad = q.emis;
  return w;
}

// Chunk fitting of a call that runs paths_per_sample paths per sample and n_samples samples: as many samples per chunk
// as the preferred chunk size and the workspace allow, each path taking RT_PATH_BYTES + extra_bytes.  Binds the queues
// for one chunk, points *extra (if given) at the chunk's extra bytes, and returns the samples per chunk, or 0 when one
// sample does not fit.
static int fit_chunk(StageParams &P, size_t paths_per_sample, int n_samples, size_t extra_bytes, void *workspace,
                     size_t workspace_bytes, char **extra) {
  const size_t cap = path_capacity(workspace_bytes, P.max_bounces, RT_PATH_BYTES + extra_bytes);
  if (cap < paths_per_sample) return 0;
  size_t fit = chunk_samples(paths_per_sample, n_samples);
  if (fit > cap / paths_per_sample) fit = cap / paths_per_sample;
  char *end = bind_queues(P.q, workspace, P.max_bounces, fit * paths_per_sample);
  if (extra) *extra = end;
  return (int)fit;
}

// Dynamic shared memory opt-in and occupancy of the trace kernels on the current device (once per device and depth).
static int trace_launch_setup(const SceneDev &scene, int sm_count, TraceLaunch &t) {
  const size_t level_bytes = level_store_bytes(scene.depth);
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= RT_MAX_DEVICES) return (int)cudaErrorInvalidDevice;
  TraceOccupancy &o = g_occupancy[dev];
  if (o.generic == 0 || level_bytes != o.level_bytes) {
    o.primary = level_store_blocks_per_sm((const void *)rt_trace_kernel<true>, level_bytes);
    o.generic = level_store_blocks_per_sm((const void *)rt_trace_kernel<false>, level_bytes);
    o.wide = level_store_blocks_per_sm((const void *)rt_trace_kernel<false, RT_TRACE_MIN_BLOCKS_WIDE>, level_bytes);
    o.fast = rt_fast_trace_setup(level_bytes, &o.fast_wide);
    o.masked = level_store_blocks_per_sm((const void *)rt_trace_kernel<true, RT_TRACE_MIN_BLOCKS_PRIMARY, true>, level_bytes);
    o.based = level_store_blocks_per_sm((const void *)rt_trace_kernel<true, RT_TRACE_MIN_BLOCKS_PRIMARY, false, true>, level_bytes);
    o.level_bytes = level_bytes;
  }
  t = TraceLaunch{dev, level_bytes, (unsigned)(sm_count * o.primary), (unsigned)(sm_count * o.generic),
                  (unsigned)(sm_count * o.wide), (unsigned)(sm_count * o.fast), (unsigned)(sm_count * o.fast_wide),
                  (unsigned)(sm_count * o.masked), (unsigned)(sm_count * o.based)};
  return 0;
}

// grid-stride kernels (miss, shade, accumulate): blocks per SM by queue length.  The items of a queue cost unevenly
// (texture taps, lobe picks), so the long queues of the first bounces want many short-lived blocks to even out the
// last wave (bounce-0 miss 2073 / 1950 / 1889 / 1864 / 1856 us at 8 / 16 / 32 / 64 / 128 blocks per SM), the short late
// queues want few (every block builds its texel table first: bounce-7 shade 23 / 31 / 41 us at 8 / 64 / 128).
static unsigned flat_grid(int sm_count) { return (unsigned)(sm_count * 8); }
static unsigned miss_grid(int sm_count, int b) { return (unsigned)sm_count * (b == 0 ? 64u : b == 1 ? 32u : 8u); }
static unsigned shade_grid(int sm_count, int b) { return (unsigned)sm_count * (b == 0 ? 64u : 8u); }

// the trace of bounce P.bounce's RAY queue, exact or fast: the wide build for the long queues of the first bounces, the
// generic one after.  The lightmap bake launches its own (the generic build at every bounce).
static void launch_bounce_trace(const StageParams &P, const TraceLaunch &t, bool fast, cudaStream_t stream) {
  const bool wide = P.bounce <= RT_TRACE_WIDE_BOUNCES;
  if (fast)      rt_fast_launch_trace(P, wide ? t.fast_wide : t.fast, t.level_bytes, stream, wide);
  else if (wide) rt_trace_kernel<false, RT_TRACE_MIN_BLOCKS_WIDE><<<t.wide, RT_BLOCK, t.level_bytes, stream>>>(P);
  else           rt_trace_kernel<false><<<t.generic, RT_BLOCK, t.level_bytes, stream>>>(P);
}

// The camera frame of a render or AOV call: job tiles, the split's share of them, fastdiv magic.
static StageParams camera_frame(const SceneDev &scene, int width, int height, int split_rank, int split_world, int max_bounces) {
  StageParams P{};
  P.scene = scene;
  P.width = width; P.height = height;
  P.tiles_x = (width + 7) / 8; P.tiles_y = (height + 3) / 4;
  P.split_rank = split_rank; P.split_world = split_world > 1 ? split_world : 1;
  P.chunks_x = (width + 31) / 32;
  P.n_tiles = rt_render_tiles(width, height, P.split_rank, P.split_world);
  // a path id is at most n_paths (32-bit), so a tile id is below 2^27 and a chunk id below tiles/32 * world + world
  P.div_tiles_x = rt_fastdiv_make((uint32_t)P.tiles_x, 0xffffffffu >> 5);
  P.div_chunks_x = rt_fastdiv_make((uint32_t)P.chunks_x, 0xffffffffu);
  P.max_bounces = max_bounces;
  return P;
}

// The header of a camera-path chunk: samples [s0, s0 + chunk) clipped to sample_end of every pixel, the accumulator
// continued or not, empty queues.
static void camera_chunk(StageParams &P, int s0, int sample_end, int chunk, bool continues, cudaStream_t stream) {
  const int S = (sample_end - s0 < chunk) ? sample_end - s0 : chunk;
  P.sample0 = s0; P.n_samples = S;
  P.n_paths = (unsigned)((size_t)P.n_tiles * 32 * (size_t)S);
  P.div_samples = rt_fastdiv_make((uint32_t)S, P.n_paths);
  P.accumulate = continues ? 1 : 0;
  cudaMemsetAsync(P.q.counts, 0, counts_bytes(P.max_bounces), stream);
}

// ------------------------------------------------------------------ sky tiles
// A job tile is sky when no jittered camera ray of its pixels can reach the root-union box: every such ray would end
// its walk at walk_misses_root and its path at the bounce-0 miss kernel, and rt_sky_kernel renders it without the path
// queues.  The argument is made in f64 on an inflated box and an enlarged footprint (DESIGN.md, "Sky tiles"), so a
// tile is classified sky only when the f32 ray generation and slab test cannot disagree.
#define RT_SKY_MARGIN 1e-3          // box inflation and zero-direction guard, relative
#define RT_SKY_PIXELS 2.0           // footprint enlargement, pixels

// Continuous pixel coordinates (u, v): pixel (px, py) casts its rays through u in [px - 0.5, px + 0.5] and v in
// [py - 0.5, py + 0.5] (jitter in [0, 1], raytracer.c:644-677).  `rect` bounds the projection of the inflated box;
// rot, aspect and focal give the camera-space direction of (u, v), whose components must keep one sign per tile.
struct SkyFrame { double rect[4]; double rot[3][3]; double aspect, focal, width, height; };

// The frame of a render, or false when no tile may be sky: a box corner at or behind the camera plane (this also
// covers a camera inside the box), an empty or non-finite box, or a camera matrix without a finite inverse.
static bool sky_frame(const SceneDev &sc, int width, int height, SkyFrame &f) {
  double r[3][3], o[3], lo[3], hi[3], scale = 0, diag = 0;
  for (int a = 0; a < 3; a++) {
    for (int b = 0; b < 3; b++) r[a][b] = sc.view[a][b];
    o[a] = sc.view[a][3]; lo[a] = sc.root_lo[a]; hi[a] = sc.root_hi[a];
    if (!(lo[a] <= hi[a]) || !std::isfinite(lo[a]) || !std::isfinite(hi[a]) || !std::isfinite(o[a])) return false;
    scale = std::fmax(scale, std::fmax(std::fabs(o[a]), std::fmax(std::fabs(lo[a]), std::fabs(hi[a]))));
    diag += (hi[a] - lo[a]) * (hi[a] - lo[a]);
  }
  const double m = RT_SKY_MARGIN * (scale + std::sqrt(diag));
  // inverse of the camera's 3x3 (camera space -> world is r, so world -> camera is its inverse)
  const double det = r[0][0] * (r[1][1] * r[2][2] - r[1][2] * r[2][1]) - r[0][1] * (r[1][0] * r[2][2] - r[1][2] * r[2][0]) +
                     r[0][2] * (r[1][0] * r[2][1] - r[1][1] * r[2][0]);
  double inv[3][3];
  for (int a = 0; a < 3; a++)
    for (int b = 0; b < 3; b++) {
      const int a1 = (b + 1) % 3, a2 = (b + 2) % 3, b1 = (a + 1) % 3, b2 = (a + 2) % 3;
      inv[a][b] = (r[a1][b1] * r[a2][b2] - r[a1][b2] * r[a2][b1]) / det;
      if (!std::isfinite(inv[a][b])) return false;
    }
  const double aspect = (double)((float)width / (float)height), focal = sc.focal_length;
  if (!(focal > 0) || !std::isfinite(focal)) return false;
  double u0 = INFINITY, u1 = -INFINITY, v0 = INFINITY, v1 = -INFINITY;
  for (int c = 0; c < 8; c++) {
    double w[3], p[3];
    for (int a = 0; a < 3; a++) w[a] = ((c >> a) & 1 ? hi[a] + m : lo[a] - m) - o[a];
    for (int a = 0; a < 3; a++) p[a] = inv[a][0] * w[0] + inv[a][1] * w[1] + inv[a][2] * w[2];
    if (!(p[2] < 0)) return false;                          // camera looks down -z: the corner is not in front
    // the camera-space direction (cx, cy, -focal) through the corner; cx = (2u / W - 1) * aspect, cy = 1 - 2v / H
    const double cx = p[0] * (-focal / p[2]), cy = p[1] * (-focal / p[2]);
    const double u = (cx / aspect + 1) * 0.5 * width, v = (1 - cy) * 0.5 * height;
    if (!std::isfinite(u) || !std::isfinite(v)) return false;
    u0 = std::fmin(u0, u); u1 = std::fmax(u1, u); v0 = std::fmin(v0, v); v1 = std::fmax(v1, v);
  }
  f = SkyFrame{{u0, u1, v0, v1}, {{r[0][0], r[0][1], r[0][2]}, {r[1][0], r[1][1], r[1][2]}, {r[2][0], r[2][1], r[2][2]}},
               aspect, focal, (double)width, (double)height};
  return true;
}

// tile sky? Its footprint, enlarged by RT_SKY_PIXELS, lies outside f.rect, and no direction component changes sign on it
// or comes within RT_SKY_MARGIN of zero relative to its terms: a zero component makes the ray non-regular (WALK_REG),
// whose walk does not take the root-union shortcut.  Tiles without pixels are sky (nothing renders them).
__device__ bool sky_tile(const StageParams &P, const SkyFrame &f, unsigned tile) {
  int x0, y0;
  tile_origin(P, tile, x0, y0);
  if (x0 >= P.width || y0 >= P.height) return true;
  const double ua = x0 - 0.5 - RT_SKY_PIXELS, ub = x0 + 7.5 + RT_SKY_PIXELS;
  const double va = y0 - 0.5 - RT_SKY_PIXELS, vb = y0 + 3.5 + RT_SKY_PIXELS;
  if (!(ub < f.rect[0] || ua > f.rect[1] || vb < f.rect[2] || va > f.rect[3])) return false;
  for (int a = 0; a < 3; a++) {
    double g_min = INFINITY, g_max = -INFINITY, terms = 0;
    for (int c = 0; c < 4; c++) {
      const double cx = ((c & 1 ? ub : ua) * 2 / f.width - 1) * f.aspect, cy = 1 - (c & 2 ? vb : va) * 2 / f.height;
      const double g = f.rot[a][0] * cx + f.rot[a][1] * cy - f.rot[a][2] * f.focal;
      g_min = fmin(g_min, g); g_max = fmax(g_max, g);
      terms = fmax(terms, fabs(f.rot[a][0] * cx) + fabs(f.rot[a][1] * cy) + fabs(f.rot[a][2] * f.focal));
    }
    if (!(g_min > RT_SKY_MARGIN * terms || g_max < -RT_SKY_MARGIN * terms)) return false;
  }
  return true;
}

// One block: the traced tiles to P.tiles[2 ..] ascending, the sky tiles from the end, the two counts to [0] and [1].
__global__ void __launch_bounds__(1024)
rt_sky_tiles_kernel(const __grid_constant__ StageParams P, const SkyFrame f, unsigned *tiles) {
  __shared__ unsigned warp_sky[32];
  __shared__ unsigned base_sky;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, lt = (1u << lane) - 1u;
  if (threadIdx.x == 0) base_sky = 0;
  for (unsigned t0 = 0; t0 < P.n_tiles; t0 += blockDim.x) {
    const unsigned tile = t0 + threadIdx.x;
    const bool sky = tile < P.n_tiles && sky_tile(P, f, tile);
    const unsigned m = __ballot_sync(RT_FULL, sky);
    if (lane == 0) warp_sky[warp] = __popc(m);
    __syncthreads();
    unsigned before = base_sky;
    for (unsigned w = 0; w < warp; w++) before += warp_sky[w];
    const unsigned sky_rank = before + __popc(m & lt);
    if (tile < P.n_tiles) {
      if (sky) tiles[2 + P.n_tiles - 1 - sky_rank] = tile;
      else     tiles[2 + tile - sky_rank] = tile;                 // tiles before it that are traced
    }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) base_sky = sky_rank + (sky ? 1u : 0u);
    __syncthreads();
  }
  if (threadIdx.x == 0) { tiles[0] = P.n_tiles - base_sky; tiles[1] = base_sky; }
}

// The scene as view v of a render sees it: the scene's own camera, or (many views) cameras[v] on a copy.
static SceneDev view_scene(const RenderParams &p, int v) {
  SceneDev sc = p.scene;
  if (p.cameras) {
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) sc.view[r][c] = p.cameras[v].view[r][c];
    sc.focal_length = p.cameras[v].focal_length;
  }
  return sc;
}

// Many views (p.cameras): each view is exactly the render it replaces.  A chunk covers a group of views and a sample
// range; view v of the group owns the path ids [base_v, base_v + n_tiles * 32 * S), base_v = (v - v0) * n_tiles * 32 * S
// (sky tiles leave holes, so the host knows every base).  Per view: the camera-relative copies (one copy, rewritten when
// the view changes: stream order makes that safe), the primary trace with the view's camera, seed and tile list, and on
// its first chunk the sky kernel; the bounce launches are shared by the group; then one accumulate per view.  A render is
// one view with the scene's camera and enqueues what it always has.
int rt_launch_render(const RenderParams &p, int sm_count, void *workspace, size_t workspace_bytes,
                     cudaStream_t stream, int *n_launches) {
  const int n_views = p.cameras ? p.n_views : 1;
  const size_t image_bytes = (size_t)p.width * p.height * 3 * sizeof(float);
  if (n_views < 1) return (int)cudaGetLastError();
  const int n_total = p.sample_end - p.sample_begin;
  if (n_total <= 0 || p.max_bounces < 1) {
    // no samples, or cast_ray's loop body never runs (raytracer.c:512,557): the sum gains nothing
    if (!p.accumulate) {
      for (int v = 0; v < n_views; v++) cudaMemsetAsync(p.accum + (size_t)v * p.view_stride, 0, image_bytes, stream);
      if (p.accum_sq) cudaMemsetAsync(p.accum_sq, 0, image_bytes, stream);
    }
    return (int)cudaGetLastError();
  }
  TraceLaunch t;
  if (int e = trace_launch_setup(p.scene, sm_count, t)) return e;

  StageParams P = camera_frame(p.scene, p.width, p.height, p.split_rank, p.split_world, p.max_bounces);
  P.user_seed = p.user_seed;
  P.accum = p.accum;
  P.per_sample = p.per_sample;
  P.per_sample_stride = n_total;
  P.counters = p.counters;
  P.counters_ex = p.counters_ex;
  P.pixel_mask = p.pixel_mask;
  P.accum_sq = p.accum_sq;
  const bool masked_sum = p.pixel_mask || p.accum_sq;      // the MASKED accumulate: mask, second moments or both

  // chunking: as many samples of every pixel (of a group of views) per chunk as the workspace holds paths
  const size_t per_sample = (size_t)P.n_tiles * 32;
  if (P.split_world > 1 && !p.accumulate)      // the pixels of other ranks stay zero (the cross-rank sum adds them)
    cudaMemsetAsync(p.accum, 0, image_bytes, stream);
  if (per_sample == 0) return (int)cudaGetLastError();
  // the tile lists first (one per view), then the path queues
  const size_t list_bytes = tile_list_bytes(P.n_tiles), lists_bytes = list_bytes * (size_t)n_views;
  if (workspace_bytes < lists_bytes) return (int)cudaErrorMemoryAllocation;
  const size_t queue_bytes = workspace_bytes - lists_bytes;
  const int group = (int)view_group(n_views, per_sample, path_capacity(queue_bytes, P.max_bounces, RT_PATH_BYTES));
  const int chunk = fit_chunk(P, (size_t)group * per_sample, n_total, 0, static_cast<char *>(workspace) + lists_bytes,
                              queue_bytes, nullptr);
  if (chunk == 0) return (int)cudaErrorMemoryAllocation;

  rt_camera_relative_kernel<<<(unsigned)sm_count, 256, 0, stream>>>(view_scene(p, 0));
  int launches = 1, relative_view = 0;          // the view the camera-relative copies hold
  std::vector<const unsigned *> tiles((size_t)n_views, nullptr);
  for (int v = 0; v < n_views; v++) {
    SkyFrame sky;
    unsigned *list = reinterpret_cast<unsigned *>(static_cast<char *>(workspace) + (size_t)v * list_bytes);
    if (sky_frame(view_scene(p, v), p.width, p.height, sky)) {
      rt_sky_tiles_kernel<<<1, 1024, 0, stream>>>(P, sky, list);
      tiles[(size_t)v] = list;
      launches++;
    }
  }
  P.tiles = tiles[0];
  bool shading_waited = false;
  for (int v0 = 0; v0 < n_views; v0 += group) {
    const int v1 = v0 + group < n_views ? v0 + group : n_views;
    for (int s0 = p.sample_begin; s0 < p.sample_end; s0 += chunk) {
      P.per_sample_offset = s0 - p.sample_begin;
      P.hit_ids = (s0 == p.sample_begin) ? p.hit_ids : nullptr;
      camera_chunk(P, s0, p.sample_end, chunk, p.accumulate || s0 > p.sample_begin || P.split_world > 1, stream);
      P.bounce = 0;
      for (int v = v0; v < v1; v++) {
        // view v's primary trace: its camera, seed and tile list, its paths from base_v; the HIT / MISS appends continue
        StageParams Pv = P;
        Pv.scene = view_scene(p, v);
        Pv.user_seed = p.user_seeds ? p.user_seeds[v] : p.user_seed;
        Pv.tiles = tiles[(size_t)v];
        Pv.accum = p.accum + (size_t)v * p.view_stride;
        Pv.path_base = (unsigned)(v - v0) * P.n_paths;
        if (v != relative_view) {
          rt_camera_relative_kernel<<<(unsigned)sm_count, 256, 0, stream>>>(Pv.scene);
          relative_view = v;
          launches++;
        }
        if (v > v0) cudaMemsetAsync(&P.q.counts[Q_FETCH], 0, sizeof(unsigned), stream);
        {
          StageTimer st(RT_STAGE_TRACE * RT_STAGE_BOUNCES, stream, t.dev);
          if (p.pixel_mask)   rt_trace_kernel<true, RT_TRACE_MIN_BLOCKS_PRIMARY, true><<<t.masked, RT_BLOCK, t.level_bytes, stream>>>(Pv);
          else if (p.cameras) rt_trace_kernel<true, RT_TRACE_MIN_BLOCKS_PRIMARY, false, true><<<t.based, RT_BLOCK, t.level_bytes, stream>>>(Pv);
          else                rt_trace_kernel<true><<<t.primary, RT_BLOCK, t.level_bytes, stream>>>(Pv);
        }
        launches++;
        // textures and the environment may still be in flight on the upload's copy stream: the primary trace reads
        // nodes and triangles only, everything after the call's first one waits here (rt_scene.cu)
        if (!shading_waited && p.shading_ready) cudaStreamWaitEvent(stream, p.shading_ready, 0);
        shading_waited = true;
        if (s0 == p.sample_begin && Pv.tiles) {
          // every sample of the view's sky tiles in one launch, timed as a bounce-0 miss stage
          StageParams S = Pv;
          S.sample0 = p.sample_begin; S.n_samples = n_total;
          S.per_sample_offset = 0;
          S.hit_ids = p.hit_ids;
          StageTimer st(RT_STAGE_MISS * RT_STAGE_BOUNCES, stream, t.dev);
          if (p.fast) rt_fast_launch_sky(S, flat_grid(sm_count) * 4, stream);
          else        rt_sky_kernel<<<flat_grid(sm_count) * 4, 256, 0, stream>>>(S);
          launches++;
        }
      }
      for (int b = 0; b < p.max_bounces; b++) {
        P.bounce = b;
        const int bslot = b < RT_STAGE_BOUNCES ? b : RT_STAGE_BOUNCES - 1;
        if (b > 0) {
          StageTimer st(RT_STAGE_TRACE * RT_STAGE_BOUNCES + bslot, stream, t.dev);
          launch_bounce_trace(P, t, p.fast, stream);
          launches++;
        }
        {
          StageTimer st(RT_STAGE_MISS * RT_STAGE_BOUNCES + bslot, stream, t.dev);
          if (p.fast) rt_fast_launch_miss(P, miss_grid(sm_count, b), stream);
          else        rt_miss_kernel<<<miss_grid(sm_count, b), 256, 0, stream>>>(P);
        }
        {
          StageTimer st(RT_STAGE_SHADE * RT_STAGE_BOUNCES + bslot, stream, t.dev);
          if (p.fast) rt_fast_launch_shade(P, shade_grid(sm_count, b), stream);
          else        rt_shade_kernel<<<shade_grid(sm_count, b), 256, 0, stream>>>(P);
        }
        launches += 2;
      }
      for (int v = v0; v < v1; v++) {
        // view v's sums from its own paths: rad from base_v, its tile list, its accumulator
        StageParams A = P;
        A.tiles = tiles[(size_t)v];
        A.accum = p.accum + (size_t)v * p.view_stride;
        A.q.rad = P.q.rad + (size_t)(v - v0) * P.n_paths;
        StageTimer st(RT_STAGE_ACCUMULATE * RT_STAGE_BOUNCES, stream, t.dev);
        if (masked_sum) rt_accumulate_masked_kernel<<<flat_grid(sm_count) * 4, 256, 0, stream>>>(A);
        else            rt_accumulate_kernel<<<flat_grid(sm_count) * 4, 256, 0, stream>>>(A);
        launches++;
      }
    }
  }
  if (n_launches) *n_launches += launches;
  return (int)cudaGetLastError();
}

// ===================================================================== lightmap_bake
// Reference raytracer.c:722-784: every triangle, in slot order, rasterises its UV footprint into the lightmap; each
// covered texel gets `samples` cosine-weighted cast_ray estimates from the interpolated surface point; a texel covered by
// several triangles keeps the LAST one's value.  Here: (1) an ownership pass finds that last triangle per texel
// (atomicMax over slots — same coverage arithmetic, f32, no contraction), (2) owned texels are compacted into jobs,
// (3) every (job, sample) is a path of the same wavefront as the renderer — its first ray comes from the texel instead
// of the camera — and (4) the cosine-weighted sum is taken per job in sample order.  Per-(texel, sample) seeds
// (rt_seed.h) replace the reference's two sequential generator streams, as for the renderer.
struct LightmapParams {
  int      width, height, samples;
  int     *owner;          // [W*H] slot of the last covering triangle, -1 = none
  unsigned *jobs;          // [n_jobs] texel index
  unsigned *n_jobs;
  float   *sums;           // [n_jobs][3] running cosine-weighted sums
  float   *cosw;           // [path] cosine of the sample's first direction (0: no direction found)
};

// barycentric weights of texel (x, y) in UV triangle `slot` exactly as raytracer.c:733-745 computes them
__device__ __forceinline__ bool lightmap_weights(const SceneDev &sc, int slot, float W, float H, float px, float py,
                                                 float &w0, float &w1, float &w2) {
  const float4 r4 = __ldg(sc.tri_rec + (size_t)slot * 7 + 4), r5 = __ldg(sc.tri_rec + (size_t)slot * 7 + 5);
  const float p0x = r4.z * W, p0y = r4.w * H, p1x = r5.x * W, p1y = r5.y * H, p2x = r5.z * W, p2y = r5.w * H;
  const float denom = (p1y - p2y) * (p0x - p2x) + (p2x - p1x) * (p0y - p2y);
  w0 = ((p1y - p2y) * (px - p2x) + (p2x - p1x) * (py - p2y)) / denom;
  w1 = ((p2y - p0y) * (px - p2x) + (p0x - p2x) * (py - p2y)) / denom;
  w2 = 1.0f - w0 - w1;
  return w0 >= -RT_EPS && w1 >= -RT_EPS && w2 >= -RT_EPS;
}

// one block per triangle slot: the texels of its UV bounding box (raytracer.c:728-731: float products truncated to i32)
__global__ void __launch_bounds__(128)
rt_lightmap_owner_kernel(const SceneDev sc, const LightmapParams L) {
  const int slot = blockIdx.x;
  const float W = (float)L.width, H = (float)L.height;
  const float4 r4 = __ldg(sc.tri_rec + (size_t)slot * 7 + 4), r5 = __ldg(sc.tri_rec + (size_t)slot * 7 + 5);
  const float ax = r4.z, ay = r4.w, bx = r5.x, by = r5.y, cx = r5.z, cy = r5.w;
  const int min_x = (int)(sel_min(ax, sel_min(bx, cx)) * W), max_x = (int)(sel_max(ax, sel_max(bx, cx)) * W);
  const int min_y = (int)(sel_min(ay, sel_min(by, cy)) * H), max_y = (int)(sel_max(ay, sel_max(by, cy)) * H);
  // texels outside the lightmap are not stored (the reference writes out of bounds): clip the box
  const int x0 = min_x < 0 ? 0 : min_x, x1 = max_x >= L.width ? L.width - 1 : max_x;
  const int y0 = min_y < 0 ? 0 : min_y, y1 = max_y >= L.height ? L.height - 1 : max_y;
  if (x1 < x0 || y1 < y0) return;
  const int bw = x1 - x0 + 1, n = bw * (y1 - y0 + 1);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int x = x0 + i % bw, y = y0 + i / bw;
    float w0, w1, w2;
    if (lightmap_weights(sc, slot, W, H, (float)x, (float)y, w0, w1, w2)) atomicMax(&L.owner[y * L.width + x], slot);
  }
}

__global__ void __launch_bounds__(256)
rt_lightmap_jobs_kernel(const LightmapParams L) {
  const unsigned n = (unsigned)(L.width * L.height), lane = threadIdx.x & 31u;
  const unsigned n_round = (n + 31u) & ~31u;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
    const bool owned = i < n && L.owner[i] >= 0;
    const unsigned pos = warp_append(L.n_jobs, owned, lane);
    if (owned) L.jobs[pos] = i;
  }
}

// common.h:30-42 with the generator state in a register; the final scale is a DOUBLE division narrowed to f32
__device__ __forceinline__ V3 lightmap_rand_vec3(uint32_t &state) {
  for (;;) {
    V3 p;
    p.x = rt_rand_f32(&state) * 2.0f + -1.0f;
    p.y = rt_rand_f32(&state) * 2.0f + -1.0f;
    p.z = rt_rand_f32(&state) * 2.0f + -1.0f;
    const float lensq = dot3(p, p);
    if (RT_EPS < lensq && lensq <= 1) return scale3(p, (float)(1.0 / (double)__fsqrt_rn(lensq)));
  }
}

// first ray of path (job, sample): raytracer.c:747-772
__global__ void __launch_bounds__(256)
rt_lightmap_raygen_kernel(const __grid_constant__ StageParams P, const LightmapParams L, unsigned n_jobs) {
  const SceneDev &sc = P.scene;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned n = n_jobs * (unsigned)P.n_samples, n_round = (n + 31u) & ~31u;
  const float W = (float)L.width, H = (float)L.height;
  for (unsigned path = blockIdx.x * blockDim.x + threadIdx.x; path < n_round; path += gridDim.x * blockDim.x) {
    bool shoot = false;
    V3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    uint32_t rng = 0;
    if (path < n) {
      const unsigned job = path / (unsigned)P.n_samples;
      const int s = P.sample0 + (int)(path - job * (unsigned)P.n_samples);
      const unsigned texel = L.jobs[job];
      const int slot = L.owner[texel];
      const int x = (int)(texel % (unsigned)L.width), y = (int)(texel / (unsigned)L.width);
      float w0, w1, w2;
      lightmap_weights(sc, slot, W, H, (float)x, (float)y, w0, w1, w2);
      const float *soa = sc.tri_soa + slot;
      const size_t N = (size_t)sc.n_slots;
      const V3 position = mk3(soa[0] * w0 + soa[N] * w1 + soa[2 * N] * w2,
                              soa[3 * N] * w0 + soa[4 * N] * w1 + soa[5 * N] * w2,
                              soa[6 * N] * w0 + soa[7 * N] * w1 + soa[8 * N] * w2);
      const float4 *rec = sc.tri_rec + (size_t)slot * 7;
      const float4 r0 = __ldg(rec), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
      // rec_normal's expressions (rt_device.cuh), written out: through the call one instruction of this kernel is
      // scheduled one slot later
      const V3 normal = mk3(r0.w * w0 + r1.z * w1 + r2.y * w2, r1.x * w0 + r1.w * w1 + r2.z * w2, r1.y * w0 + r2.x * w1 + r2.w * w2);
      o = add3(position, scale3(normal, RT_EPS));
      uint32_t dir_state = rt_path_seed(texel, (uint32_t)s, P.user_seed ^ RT_LIGHTMAP_DIR_SALT);
      rng = rt_path_seed(texel, (uint32_t)s, P.user_seed);
      float cosine = 0;
      for (int tries = 0; tries < RT_LIGHTMAP_MAX_TRIES; tries++) {
        d = lightmap_rand_vec3(dir_state);
        cosine = dot3(d, normal);
        if (cosine > 0) break;
        cosine = 0;
      }
      shoot = cosine > 0;
      L.cosw[path] = cosine;
      if (!shoot) P.q.rad[path] = make_float4(0, 0, 0, 0);
    }
    const unsigned pos = warp_append(&P.q.counts[Q_RAYS], shoot, lane);
    if (shoot) {
      P.q.ray_a[pos] = make_float4(o.x, o.y, o.z, d.x);
      P.q.ray_b[pos] = make_float4(d.y, d.z, __uint_as_float(path), __uint_as_float(rng));
    }
  }
}

// raytracer.c:773: accumulated += cast_ray(...) * cos, in sample order
__global__ void __launch_bounds__(256)
rt_lightmap_accumulate_kernel(const __grid_constant__ StageParams P, const LightmapParams L, unsigned n_jobs, int first_chunk) {
  for (unsigned job = blockIdx.x * blockDim.x + threadIdx.x; job < n_jobs; job += gridDim.x * blockDim.x) {
    V3 sum = first_chunk ? mk3(0, 0, 0) : mk3(L.sums[3 * job], L.sums[3 * job + 1], L.sums[3 * job + 2]);
    const size_t base = (size_t)job * (size_t)P.n_samples;
    for (int s = 0; s < P.n_samples; s++) {
      const float c = L.cosw[base + s];
      if (!(c > 0)) continue;
      const float4 v = P.q.rad[base + s];
      sum = add3(sum, scale3(mk3(v.x, v.y, v.z), c));
    }
    L.sums[3 * job] = sum.x; L.sums[3 * job + 1] = sum.y; L.sums[3 * job + 2] = sum.z;
  }
}

// raytracer.c:777-779: the UN-SCALED f32 goes into the u8 (saturating here; C leaves out-of-range undefined)
__global__ void __launch_bounds__(256)
rt_lightmap_store_kernel(const LightmapParams L, unsigned n_jobs, unsigned char *pixels, int stride, int components, float *values) {
  for (unsigned job = blockIdx.x * blockDim.x + threadIdx.x; job < n_jobs; job += gridDim.x * blockDim.x) {
    const unsigned texel = L.jobs[job];
    const int x = (int)(texel % (unsigned)L.width), y = (int)(texel / (unsigned)L.width);
    unsigned char *dst = pixels + (size_t)components * (size_t)(x + y * stride);
    for (int c = 0; c < 3; c++) {
      const float v = L.sums[3 * job + c] / (float)L.samples;
      if (values) values[3 * (size_t)texel + c] = v;
      dst[c] = !(v == v) ? 0 : (v <= 0 ? 0 : (v >= 255 ? 255 : (unsigned char)v));
    }
  }
}

size_t rt_lightmap_workspace_bytes(int width, int height) {
  const size_t n = (size_t)width * (size_t)height;
  return ((n * (sizeof(int) + sizeof(unsigned) + 3 * sizeof(float)) + 256 + 255) & ~(size_t)255);
}

// `scratch` holds owner / jobs / sums (rt_lightmap_workspace_bytes), `workspace` the path queues plus one f32 per path.
int rt_launch_lightmap(const SceneDev &scene, int width, int height, int samples, int max_bounces, uint32_t user_seed,
                       unsigned char *d_pixels, int stride, int components, float *d_values, int *d_owner_out,
                       void *scratch, int sm_count, void *workspace, size_t workspace_bytes, cudaStream_t stream,
                       int *n_launches, unsigned *n_jobs_out) {
  TraceLaunch t;
  if (int e = trace_launch_setup(scene, sm_count, t)) return e;
  const size_t n_texels = (size_t)width * (size_t)height;
  LightmapParams L{};
  L.width = width; L.height = height; L.samples = samples;
  char *sp = static_cast<char *>(scratch);
  L.n_jobs = reinterpret_cast<unsigned *>(sp); sp += 256;
  L.owner = reinterpret_cast<int *>(sp);       sp += n_texels * sizeof(int);
  L.jobs = reinterpret_cast<unsigned *>(sp);   sp += n_texels * sizeof(unsigned);
  L.sums = reinterpret_cast<float *>(sp);
  cudaMemsetAsync(L.n_jobs, 0, 256, stream);
  cudaMemsetAsync(L.owner, 0xff, n_texels * sizeof(int), stream);
  const unsigned flat = flat_grid(sm_count);
  rt_lightmap_owner_kernel<<<(unsigned)scene.n_slots, 128, 0, stream>>>(scene, L);
  rt_lightmap_jobs_kernel<<<flat, 256, 0, stream>>>(L);
  int launches = 2;
  unsigned n_jobs = 0;
  cudaMemcpyAsync(&n_jobs, L.n_jobs, sizeof n_jobs, cudaMemcpyDeviceToHost, stream);
  if (cudaError_t e = cudaStreamSynchronize(stream)) return (int)e;
  if (n_jobs_out) *n_jobs_out = n_jobs;
  if (d_owner_out) cudaMemcpyAsync(d_owner_out, L.owner, n_texels * sizeof(int), cudaMemcpyDeviceToDevice, stream);
  if (n_jobs == 0 || samples < 1 || max_bounces < 1) { if (n_launches) *n_launches += launches; return (int)cudaGetLastError(); }

  StageParams P{};
  P.scene = scene;
  P.width = width; P.height = height;
  P.max_bounces = max_bounces;
  P.user_seed = user_seed;
  char *cosw = nullptr;
  const int chunk = fit_chunk(P, n_jobs, samples, sizeof(float), workspace, workspace_bytes, &cosw);
  if (chunk == 0) return (int)cudaErrorMemoryAllocation;
  L.cosw = reinterpret_cast<float *>(cosw);
  for (int s0 = 0; s0 < samples; s0 += chunk) {
    const int S = samples - s0 < chunk ? samples - s0 : chunk;
    P.sample0 = s0; P.n_samples = S;
    P.n_paths = n_jobs * (unsigned)S;
    cudaMemsetAsync(P.q.counts, 0, counts_bytes(max_bounces), stream);
    rt_lightmap_raygen_kernel<<<flat, 256, 0, stream>>>(P, L, n_jobs);
    launches++;
    // the generic trace and flat grids at every bounce, not the camera path's per-bounce shapes
    for (int b = 0; b < max_bounces; b++) {
      P.bounce = b;
      rt_trace_kernel<false><<<t.generic, RT_BLOCK, t.level_bytes, stream>>>(P);
      rt_miss_kernel<<<flat, 256, 0, stream>>>(P);
      rt_shade_kernel<<<flat, 256, 0, stream>>>(P);
      launches += 3;
    }
    rt_lightmap_accumulate_kernel<<<flat, 256, 0, stream>>>(P, L, n_jobs, s0 == 0);
    launches++;
  }
  rt_lightmap_store_kernel<<<flat, 256, 0, stream>>>(L, n_jobs, d_pixels, stride, components, d_values);
  launches++;
  if (n_launches) *n_launches += launches;
  return (int)cudaGetLastError();
}

// ===================================================================== cast_rays
// Reference raytracer.c:505-558 for caller-supplied rays: path (ray i, sample s) is cast_ray(scene, ray_i, max_bounces)
// with the shader generator seeded to rt_path_seed(key_i, s, user_seed) (rt_seed.h) just before the call.  The first ray
// of a path is the caller's, as given (not normalised); the bounces run on the renderer's unchanged stage kernels, and
// the per-ray sum is taken in sample order.  A chunk holds R rays x S samples, path id = ray_in_chunk * S + s: a warp is
// consecutive samples of one ray, as in the renderer's layout.
struct CastRaysParams {
  const float    *rays;          // [n_rays][6]: the reference's Ray (position, direction)
  const unsigned *keys;          // optional [n_rays]: seed key of each ray, NULL = its index
  unsigned  ray0, n_rays;        // this chunk: rays [ray0, ray0 + n_rays)
  float    *radiance;            // [n_rays total][3] running sums
  float    *per_sample;          // optional [n_rays total][per_sample_stride][3], this chunk at +per_sample_offset
  int       per_sample_stride, per_sample_offset;
};

// first ray of path (ray, sample): the caller's ray and the path's seed, appended to the RAY queue of bounce 0.  Without
// bounces (max_bounces = 0) cast_ray returns its zero emission: the path ends here with radiance 0 and counts as a sample
// (otherwise the miss or shade kernel that ends it counts it).
__global__ void __launch_bounds__(256)
rt_cast_rays_raygen_kernel(const __grid_constant__ StageParams P, const CastRaysParams C) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned S = (unsigned)P.n_samples, n = P.n_paths, n_round = (n + 31u) & ~31u;
  unsigned c_samples = 0;
  for (unsigned path = blockIdx.x * blockDim.x + threadIdx.x; path < n_round; path += gridDim.x * blockDim.x) {
    bool shoot = false;
    float4 a = make_float4(0, 0, 0, 0), b = make_float4(0, 0, 0, 0);
    if (path < n) {
      const unsigned r = path / S, ray = C.ray0 + r;
      const int s = P.sample0 + (int)(path - r * S);
      const float *src = C.rays + (size_t)ray * 6;
      const uint32_t key = C.keys ? C.keys[ray] : ray;
      const uint32_t rng = rt_path_seed(key, (uint32_t)s, P.user_seed);
      shoot = P.max_bounces > 0;
      a = make_float4(src[0], src[1], src[2], src[3]);
      b = make_float4(src[4], src[5], __uint_as_float(path), __uint_as_float(rng));
      if (!shoot) { P.q.rad[path] = make_float4(0, 0, 0, 0); c_samples++; }
    }
    const unsigned pos = warp_append(&P.q.counts[Q_RAYS], shoot, lane);
    if (shoot) { P.q.ray_a[pos] = a; P.q.ray_b[pos] = b; }
  }
  if (P.counters) add_counter(P.counters, 7, c_samples);
}

// raytracer.c:696-700 per ray: radiance += cast_ray(...) in sample order, from zero on the first chunk of a call without
// `accumulate`, else from the buffer
__global__ void __launch_bounds__(256)
rt_cast_rays_accumulate_kernel(const __grid_constant__ StageParams P, const CastRaysParams C) {
  for (unsigned r = blockIdx.x * blockDim.x + threadIdx.x; r < C.n_rays; r += gridDim.x * blockDim.x) {
    const size_t ray = (size_t)C.ray0 + r;
    float *dst = C.radiance + 3 * ray;
    V3 sum = P.accumulate ? mk3(dst[0], dst[1], dst[2]) : mk3(0, 0, 0);
    const float4 *rad = P.q.rad + (size_t)r * (size_t)P.n_samples;
    for (int s = 0; s < P.n_samples; s++) {
      const float4 v = rad[s];
      sum = add3(sum, mk3(v.x, v.y, v.z));
      if (C.per_sample) {
        float *ps = C.per_sample + (ray * (size_t)C.per_sample_stride + (size_t)(C.per_sample_offset + s)) * 3;
        ps[0] = v.x; ps[1] = v.y; ps[2] = v.z;
      }
    }
    dst[0] = sum.x; dst[1] = sum.y; dst[2] = sum.z;
  }
}

size_t rt_cast_rays_workspace_bytes(size_t n_paths, int max_bounces, bool floor) {
  size_t paths = floor ? (size_t)RT_CAST_RAYS_MIN_CHUNK : chunk_paths_max();
  if (paths > n_paths) paths = n_paths;
  if (paths < 1) paths = 1;
  return counts_bytes(max_bounces) + paths * RT_PATH_BYTES;
}

size_t rt_lightmap_paths_workspace_bytes(size_t n_texels, int samples, int max_bounces, bool floor) {
  // a path's records and its cosine, plus slack: the queue lengths' share of a 32-path tile and 16 B (156 B at 8 bounces)
  const size_t per_path = RT_PATH_BYTES + sizeof(float) + counts_bytes(max_bounces) / 32 + 16;
  const size_t chunk = chunk_samples(32, 0) * 32;
  size_t paths = floor ? n_texels : n_texels * (size_t)samples;
  if (paths > chunk) paths = chunk;
  if (paths < n_texels) paths = n_texels;
  return paths * per_path + 4096;
}

int rt_launch_cast_rays(const SceneDev &scene, const float *rays, const unsigned *keys, int n_rays, int sample_begin,
                        int samples, int max_bounces, uint32_t user_seed, int accumulate, float *radiance, float *per_sample,
                        unsigned long long *counters, int sm_count, void *workspace, size_t workspace_bytes,
                        cudaStream_t stream, int *n_launches) {
  if (n_rays <= 0) return (int)cudaGetLastError();
  if (samples <= 0) {
    // no samples: the sums gain nothing (as rt_launch_render)
    if (!accumulate) cudaMemsetAsync(radiance, 0, (size_t)n_rays * 3 * sizeof(float), stream);
    return (int)cudaGetLastError();
  }
  TraceLaunch t;
  if (int e = trace_launch_setup(scene, sm_count, t)) return e;

  StageParams P{};
  P.scene = scene;
  P.width = 1; P.height = 1;                 // no camera: the bounce trace does not use them
  P.max_bounces = max_bounces;
  P.user_seed = user_seed;
  P.counters = counters;
  CastRaysParams C{};
  C.rays = rays; C.keys = keys; C.radiance = radiance; C.per_sample = per_sample;
  C.per_sample_stride = samples;

  // chunking: R rays x S samples per chunk, at most `cap` paths.  Every sample of every ray when they fit; otherwise
  // samples of a ray stay together up to a warp's worth (or all of them, if the rays are few) and the rays are split
  size_t cap = path_capacity(workspace_bytes, max_bounces, RT_PATH_BYTES);
  if (cap < 1) return (int)cudaErrorMemoryAllocation;
  if (cap > chunk_paths_max()) cap = chunk_paths_max();
  size_t S = (size_t)samples, R = (size_t)n_rays;
  if (R * S > cap) {
    const size_t warp = cap < 32 ? cap : 32;
    S = cap / R > warp ? cap / R : warp;
    if (S > (size_t)samples) S = (size_t)samples;
    R = cap / S;
    if (R > (size_t)n_rays) R = (size_t)n_rays;
  }
  bind_queues(P.q, workspace, max_bounces, R * S);

  // the renderer's per-bounce launch shapes (rt_launch_render); bounce 0 is a generic trace of a long queue
  int launches = 0;
  for (size_t r0 = 0; r0 < (size_t)n_rays; r0 += R) {
    C.ray0 = (unsigned)r0;
    C.n_rays = (unsigned)((size_t)n_rays - r0 < R ? (size_t)n_rays - r0 : R);
    for (int s0 = sample_begin; s0 < sample_begin + samples; s0 += (int)S) {
      const int n_s = sample_begin + samples - s0 < (int)S ? sample_begin + samples - s0 : (int)S;
      P.sample0 = s0; P.n_samples = n_s;
      P.n_paths = C.n_rays * (unsigned)n_s;
      P.accumulate = (accumulate || s0 > sample_begin) ? 1 : 0;
      C.per_sample_offset = s0 - sample_begin;
      cudaMemsetAsync(P.q.counts, 0, counts_bytes(max_bounces), stream);
      rt_cast_rays_raygen_kernel<<<flat_grid(sm_count), 256, 0, stream>>>(P, C);
      launches++;
      for (int b = 0; b < max_bounces; b++) {
        P.bounce = b;
        launch_bounce_trace(P, t, false, stream);
        rt_miss_kernel<<<miss_grid(sm_count, b), 256, 0, stream>>>(P);
        rt_shade_kernel<<<shade_grid(sm_count, b), 256, 0, stream>>>(P);
        launches += 3;
      }
      rt_cast_rays_accumulate_kernel<<<flat_grid(sm_count) * 4, 256, 0, stream>>>(P, C);
      launches++;
    }
  }
  if (n_launches) *n_launches += launches;
  return (int)cudaGetLastError();
}

// ===================================================================== first-surface AOVs
// What surface the renderer's path (pixel, sample) shades first: its camera ray (the unchanged primary trace), walked
// through back faces as shade_hit steps through them (raytracer.c:516-522), to the first front face within max_bounces
// walks.  Nothing random happens before that shade, so the record is exact per (pixel, sample).  The surface kernel
// keeps, per path id, (point.xyz, slot) in `tint` and (u, v) in `emis` (path state the trace kernel never touches;
// slot -1 = no surface); the accumulate kernel evaluates the material there (pbr_surface, as shade_pbr does) and sums
// per pixel in sample order.

// the HIT queue of bounce b: a back face goes on to the RAY queue of b + 1 while walks remain; a front face is the path's
// surface.  Misses have no kernel (their record stays "no surface"): their count comes from the queue length.
__global__ void __launch_bounds__(256)
rt_aov_surface_kernel(const __grid_constant__ StageParams P) {
  const SceneDev &sc = P.scene;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned n = P.q.counts[P.bounce * Q_STRIDE + Q_HITS];
  unsigned *next_rays = &P.q.counts[(P.bounce + 1) * Q_STRIDE + Q_RAYS];
  const unsigned n_round = (n + 31u) & ~31u;          // whole warps stay in the loop for the collective append
  unsigned c_shades = 0, c_pass = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
    bool cont = false;
    float4 ra = make_float4(0, 0, 0, 0), rb = make_float4(0, 0, 0, 0);
    if (i < n) {
      const float4 a = P.q.hit_a[i], b = P.q.hit_b[i], h = P.q.hit_h[i];
      const V3 o = mk3(a.x, a.y, a.z), d = mk3(a.w, b.x, b.y);
      const unsigned path = __float_as_uint(b.z);
      const int slot = __float_as_int(h.w);
      // shade_hit's point, interpolated normal and back-face test (rt_stages.cuh)
      const float4 *rec = sc.tri_rec + (size_t)slot * 7;
      const float4 r0 = __ldg(rec + 0), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
      const V3 ng = rec_normal_geo(r0);
      const float w1 = h.y, w2 = h.z, w0 = 1 - w1 - w2;
      const V3 point = hit_point(o, d, h.x);
      const V3 normal = rec_normal(r0, r1, r2, w0, w1, w2);
      if (hit_back_face(ng, normal, d)) {
        c_pass++;
        cont = P.bounce + 1 < P.max_bounces;
        const V3 next = add3(point, scale3(d, RT_EPS));
        ra = make_float4(next.x, next.y, next.z, d.x);
        rb = make_float4(d.y, d.z, b.z, b.w);
      } else {
        c_shades++;
        P.q.tint[path] = make_float4(point.x, point.y, point.z, h.w);
        P.q.emis[path] = make_float4(w1, w2, 0, 0);
      }
    }
    const unsigned pos = warp_append(next_rays, cont, lane);
    if (cont) { P.q.ray_a[pos] = ra; P.q.ray_b[pos] = rb; }
  }
  if (P.counters) {
    add_counter(P.counters, 4, c_shades);
    add_counter(P.counters, 6, c_pass);
    if (blockIdx.x == 0 && threadIdx.x == 0)
      atomicAdd(&P.counters[5], (unsigned long long)P.q.counts[P.bounce * Q_STRIDE + Q_MISSES]);
  }
}

// per pixel: the records of its samples in sample order, each sample's material evaluated at its surface, summed into
// aov[pixel] = (albedo, coverage) (normal, depth) (position, roughness) (emission, metalness) — from zero on the first
// chunk of a call without `accumulate`, else from the buffer
__global__ void __launch_bounds__(256)
rt_aov_accumulate_kernel(const __grid_constant__ StageParams P, float4 *__restrict__ aov) {
  const SceneDev &sc = P.scene;
  const float ex = sc.view[0][3], ey = sc.view[1][3], ez = sc.view[2][3];          // the camera origin (raytracer.c:612)
  const unsigned n = P.n_tiles * 32u;
  unsigned c_samples = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned tile = i >> 5, in_tile = i & 31u;
    int x0, y0;
    tile_origin(P, tile, x0, y0);
    const int px = x0 + (int)(in_tile & 7u), py = y0 + (int)(in_tile >> 3);
    if (px >= P.width || py >= P.height) continue;
    float4 *dst = aov + 4 * ((size_t)py * (size_t)P.width + (size_t)px);
    float4 s0 = make_float4(0, 0, 0, 0), s1 = s0, s2 = s0, s3 = s0;
    if (P.accumulate) { s0 = dst[0]; s1 = dst[1]; s2 = dst[2]; s3 = dst[3]; }
    const size_t first = (size_t)i * (size_t)P.n_samples;            // RT_PATH_LAYOUT 1: path id = pixel * S + s
    for (int s = 0; s < P.n_samples; s++) {
      const float4 surf = P.q.tint[first + s];
      const int slot = __float_as_int(surf.w);
      if (slot < 0) continue;
      const float4 bary = P.q.emis[first + s];
      // shade_hit's shading input (rt_stages.cuh) at the recorded surface
      const float4 *rec = sc.tri_rec + (size_t)slot * 7;
      const float4 r0 = __ldg(rec + 0), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2), r3 = __ldg(rec + 3);
      const float4 r4 = __ldg(rec + 4), r5 = __ldg(rec + 5), r6 = __ldg(rec + 6);
      const float w1 = bary.x, w2 = bary.y, w0 = 1 - w1 - w2;
      const V3 normal = rec_normal(r0, r1, r2, w0, w1, w2);
      // the material fetch does not read the direction
      const ShadeIn in = shade_input(mk3(0, 0, 0), normal, rec_normal_geo(r0), r3, r4, r5, w0, w1, w2);
      V3 nrm, base, glow;
      float roughness, metalness;
      pbr_surface(sc, sc.materials[rec_material(r6)], in, nrm, base, roughness, metalness, glow);
      const float dx = surf.x - ex, dy = surf.y - ey, dz = surf.z - ez;
      const float depth = __fsqrt_rn(dx * dx + dy * dy + dz * dz);
      s0.x += base.x; s0.y += base.y; s0.z += base.z; s0.w += 1.0f;
      s1.x += nrm.x;  s1.y += nrm.y;  s1.z += nrm.z;  s1.w += depth;
      s2.x += surf.x; s2.y += surf.y; s2.z += surf.z; s2.w += roughness;
      s3.x += glow.x; s3.y += glow.y; s3.z += glow.z; s3.w += metalness;
    }
    dst[0] = s0; dst[1] = s1; dst[2] = s2; dst[3] = s3;
    c_samples += (unsigned)P.n_samples;
  }
  if (P.counters) add_counter(P.counters, 7, c_samples);
}

int rt_launch_aov(const SceneDev &scene, int width, int height, int sample_begin, int sample_end, int max_bounces,
                  int accumulate, float *aov, unsigned long long *counters, int sm_count, void *workspace,
                  size_t workspace_bytes, cudaStream_t stream, int *n_launches) {
  const int n_total = sample_end - sample_begin;
  if (n_total <= 0 || max_bounces < 1) {
    // no samples, or no walk: no sample has a surface (as rt_launch_render)
    if (!accumulate) cudaMemsetAsync(aov, 0, (size_t)width * (size_t)height * 16 * sizeof(float), stream);
    return (int)cudaGetLastError();
  }
  TraceLaunch t;
  if (int e = trace_launch_setup(scene, sm_count, t)) return e;

  // the renderer's frame and chunking (rt_launch_render, whole image)
  StageParams P = camera_frame(scene, width, height, 0, 1, max_bounces);
  P.counters = counters;
  const int chunk = fit_chunk(P, (size_t)P.n_tiles * 32, n_total, 0, workspace, workspace_bytes, nullptr);
  if (chunk == 0) return (int)cudaErrorMemoryAllocation;

  rt_camera_relative_kernel<<<(unsigned)sm_count, 256, 0, stream>>>(scene);
  int launches = 1;
  for (int s0 = sample_begin; s0 < sample_end; s0 += chunk) {
    camera_chunk(P, s0, sample_end, chunk, accumulate || s0 > sample_begin, stream);
    cudaMemsetAsync(P.q.tint, 0xff, (size_t)P.n_paths * sizeof(float4), stream);    // slot -1: no surface yet
    P.bounce = 0;
    rt_trace_kernel<true><<<t.primary, RT_BLOCK, t.level_bytes, stream>>>(P);
    launches++;
    for (int b = 0; b < max_bounces; b++) {
      P.bounce = b;
      if (b > 0) {
        launch_bounce_trace(P, t, false, stream);
        launches++;
      }
      rt_aov_surface_kernel<<<shade_grid(sm_count, b), 256, 0, stream>>>(P);     // in place of miss and shade
      launches++;
    }
    rt_aov_accumulate_kernel<<<flat_grid(sm_count) * 4, 256, 0, stream>>>(P, reinterpret_cast<float4 *>(aov));
    launches++;
  }
  if (n_launches) *n_launches += launches;
  return (int)cudaGetLastError();
}

int rt_launch_resolve(const float *accum, int width, int height, int samples, unsigned char *pixels,
                      int stride, int components, cudaStream_t stream) {
  int n = width * height;
  float inv_samples = 1.0f / (float)samples;
  rt_resolve_kernel<<<(n + 255) / 256, 256, 0, stream>>>(accum, width, height, inv_samples, pixels, stride, components);
  return (int)cudaGetLastError();
}

int rt_launch_resolve_counts(const float *accum, const int *samples, int width, int height, unsigned char *pixels,
                             int stride, int components, cudaStream_t stream) {
  int n = width * height;
  rt_resolve_counts_kernel<<<(n + 255) / 256, 256, 0, stream>>>(accum, samples, width, height, pixels, stride, components);
  return (int)cudaGetLastError();
}

int rt_launch_reduce_resolve(const ReduceParts &parts, float *sum_out, int width, int height, int samples,
                             unsigned char *pixels, int stride, int components, cudaStream_t stream) {
  const int groups = (width * height + 3) / 4;
  const float inv_samples = 1.0f / (float)samples;
  rt_reduce_resolve_kernel<<<(groups + 255) / 256, 256, 0, stream>>>(parts, sum_out, width, height, inv_samples, pixels, stride, components);
  return (int)cudaGetLastError();
}

int rt_render_blocks_per_sm(void) {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < RT_MAX_DEVICES ? g_occupancy[dev].generic : 0;
}
