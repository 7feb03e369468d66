// rt_stages.cuh — the wavefront stage kernels (trace, miss, shade) and the records they exchange.
//
// Compiled twice: by rt_render.cu as written — IEEE f32 in the reference's operation order, no FMA contraction,
// rt_math.h transcendentals: the parity path — and by rt_render_fast.cu with RT_FAST=1 (FMA contraction on, hardware
// transcendentals, f32 where the reference's unsuffixed literals promote to f64): the opt-in fast mode
// (RT_GPU_Options.fast_math).  RT_KN() gives the second copy its own kernel names.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>

#include "rt_device.cuh"
#include "rt_fastdiv.h"
#include "rt_trace.cuh"
#include "rt_shade.cuh"

#if defined(RT_FAST) && RT_FAST
#define RT_KN(name) name##_fast
#else
#define RT_KN(name) name
#endif

#ifndef RT_TRACE_MIN_BLOCKS
#define RT_TRACE_MIN_BLOCKS 3
#endif
#ifndef RT_TRACE_MIN_BLOCKS_PRIMARY
#define RT_TRACE_MIN_BLOCKS_PRIMARY 4
#endif
#ifndef RT_TRACE_MIN_BLOCKS_WIDE
#define RT_TRACE_MIN_BLOCKS_WIDE 4       // bounce rays of the first RT_TRACE_WIDE_BOUNCES bounces
#endif
#ifndef RT_TRACE_WIDE_BOUNCES
#define RT_TRACE_WIDE_BOUNCES 2
#endif
#ifndef RT_EMIT_ONE_ATOMIC
#define RT_EMIT_ONE_ATOMIC 1
#endif

// counts[bounce][...]: queue lengths written by one stage and read by the next
// (HITS and MISSES share one aligned 64-bit word: the trace kernel reserves both with one atomic)
enum { Q_RAYS = 0, Q_FETCH = 1, Q_HITS = 2, Q_MISSES = 3, Q_STRIDE = 4 };

struct PathQueues {
  // queue records, compacted (a record moves with its ray): what the traversal needs and nothing else
  float4 *ray_a, *ray_b;                            // (o.xyz, d.x) (d.yz, path, rng)
  float4 *hit_a, *hit_b, *hit_h;                    // the same two + (t, u, v, slot)
  float4 *miss_a;                                   // (d.xyz, path)
  // path state, indexed by path id (touched by exactly one thread per stage: no ordering hazard): the running
  // tint and emission of cast_ray (raytracer.c:507-510,537,544).  The trace kernel neither reads nor writes them.
  // When a path ends, its radiance replaces the emission — `rad` IS `emis`.
  float4 *tint, *emis;
  float4 *rad;                                      // [path] radiance of the finished sample (alias of emis)
  unsigned *counts;                                 // [max_bounces + 1][Q_STRIDE]
};

struct __align__(16) StageParams {
  SceneDev   scene;
  PathQueues q;
  int        width, height, tiles_x, tiles_y;
  // pixel-space split (multi-GPU at low spp, SURVEY 8e): split_world > 1 = this render owns the reference's
  // 32x32 chunks (raytracer.c:619-637) whose row-major id is congruent to split_rank; a chunk is 4 x 8 job tiles
  int        split_rank, split_world, chunks_x;
  unsigned   n_tiles;                 // job tiles (8x4 pixels) this render covers
  int        sample0, n_samples;      // this chunk: samples [sample0, sample0 + n_samples)
  int        bounce, max_bounces;
  uint32_t   user_seed;
  unsigned   n_paths;                 // tiles * n_samples * 32
  RT_FastDiv div_samples, div_tiles_x, div_chunks_x;   // magic pairs of the three per-launch divisors (rt_fastdiv.h)
  int        accumulate;
  float     *accum;
  float     *per_sample;              // optional [pixel][per_sample_stride][3], this chunk at +per_sample_offset
  int        per_sample_stride, per_sample_offset;
  int       *hit_ids;                 // optional, written by the primary trace for sample `sample0`
  unsigned long long *counters;
  unsigned long long *counters_ex;    // optional 8 more: [0] rays whose walk was the root-union test alone, [1] primary rays
  // masked passes (rt_gpu_render_masked_device), last so that the fields above keep their offsets
  const unsigned char *pixel_mask;    // optional [pixel]: non-zero = render; read by the MASKED trace and accumulate only
  float     *accum_sq;                // optional [pixel][3]: sum of v * v in sample order
  // optional job-tile lists of a render with sky tiles (rt_render.cu): [0] traced tiles, [1] sky tiles, then the traced
  // tile ids ascending from [2] and the sky tile ids from [2 + n_tiles - 1] down.  The primary trace and the accumulate
  // cover the traced tiles only (path ids are built on the list), rt_sky_kernel the sky tiles.  NULL = every tile traced.
  const unsigned *tiles;
  // many views in one call (rt_render.cu): the first path id of this view's primary trace; read by the BASED trace only
  unsigned   path_base;
};

// raytracer.c:582-594, one lane of hash12x8.  Ray generation is spelled with round-to-nearest intrinsics, which are
// never fused: the exact build compiles them to what it compiles the plain operators to, and the fast build
// (rt_render_fast.cu, FMA contraction on) generates the same rays as the exact one.
__device__ __forceinline__ float fract1(float v) { return __fsub_rn(v, floorf(v)); }
__device__ __forceinline__ float hash12(float px, float py) {
  float a = fract1(__fmul_rn(px, 0.1031f));
  float b = fract1(__fmul_rn(py, 0.1031f));
  float c = fract1(__fmul_rn(px, 0.1031f));
  float k = 33.33f;
  float d = __fadd_rn(__fadd_rn(__fmul_rn(a, __fadd_rn(b, k)), __fmul_rn(b, __fadd_rn(c, k))), __fmul_rn(c, __fadd_rn(a, k)));
  return fract1(__fmul_rn(__fadd_rn(__fadd_rn(a, b), __fmul_rn(d, 2.0f)), __fadd_rn(c, d)));
}

// raytracer.c:644-677: the direction of camera sample s of pixel (px, py); rand_a == rand_b, exact 1/sqrt instead of
// rsqrt_ps.  inv_w = 1 / width, inv_h = 1 / height, aspect = width / height.  The origin is the camera's (view column 3).
__device__ __forceinline__ void camera_dir(const SceneDev &sc, int px, int py, int s, float inv_w, float inv_h, float aspect,
                                           float &dx, float &dy, float &dz) {
  const float jit = hash12(__fadd_rn(__fmul_rn((float)px, 50.0f), (float)s), (float)py);
  const float ux = __fsub_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fadd_rn((float)px, jit), 0.5f), 2.0f), inv_w), 1.0f);
  const float uy = __fsub_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fadd_rn((float)py, jit), 0.5f), 2.0f), inv_h), 1.0f);
  const float cx = __fmul_rn(ux, aspect), cy = -uy, cz = -sc.focal_length;
  const float inv_len = 1.0f / __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz)));
  dx = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(sc.view[0][0], cx), __fmul_rn(sc.view[0][1], cy)), __fmul_rn(sc.view[0][2], cz)), inv_len);
  dy = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(sc.view[1][0], cx), __fmul_rn(sc.view[1][1], cy)), __fmul_rn(sc.view[1][2], cz)), inv_len);
  dz = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(sc.view[2][0], cx), __fmul_rn(sc.view[2][1], cy)), __fmul_rn(sc.view[2][2], cz)), inv_len);
}

// top-left pixel of job tile `tile` (8x4 pixels): row-major over the image, or — pixel-space split — the
// tile's place inside the k-th 32x32 chunk this rank owns (chunk id = k * split_world + split_rank)
__device__ __forceinline__ void tile_origin(const StageParams &P, unsigned tile, int &x0, int &y0) {
  if (P.split_world <= 1) {
    const unsigned row = rt_fastdiv(tile, P.div_tiles_x, (unsigned)P.tiles_x);
    x0 = (int)(tile - row * (unsigned)P.tiles_x) * 8;
    y0 = (int)row * 4;
  } else {
    const unsigned chunk = (tile >> 5) * (unsigned)P.split_world + (unsigned)P.split_rank, t = tile & 31u;
    const unsigned row = rt_fastdiv(chunk, P.div_chunks_x, (unsigned)P.chunks_x);
    x0 = (int)(chunk - row * (unsigned)P.chunks_x) * 32 + (int)(t & 3u) * 8;
    y0 = (int)row * 32 + (int)(t >> 2) * 4;                                 // beyond the last chunk row: y0 >= height
  }
}

// RT_PATH_LAYOUT 0: path id = (tile * S + s) * 32 + pixel-in-tile — a warp is one 8x4 pixel tile at one sample index.
// RT_PATH_LAYOUT 1: path id = (tile * 32 + pixel-in-tile) * S + s — a warp is 32 consecutive samples of ONE pixel:
// its primary rays differ by less than a pixel, so they walk the same nodes and test the same leaves.
#ifndef RT_PATH_LAYOUT
#define RT_PATH_LAYOUT 1
#endif
__device__ __forceinline__ void path_pixel(const StageParams &P, unsigned path, int &px, int &py, int &ls) {
#if RT_PATH_LAYOUT == 1
  const unsigned pix = rt_fastdiv(path, P.div_samples, (unsigned)P.n_samples);
  ls = (int)(path - pix * (unsigned)P.n_samples);
  const unsigned in_tile = pix & 31u, tile = P.tiles ? P.tiles[2 + (pix >> 5)] : pix >> 5;
#else
  unsigned in_tile = path & 31u, rest = path >> 5;
  unsigned tile = rest / (unsigned)P.n_samples;
  ls = (int)(rest - tile * (unsigned)P.n_samples);
  if (P.tiles) tile = P.tiles[2 + tile];
#endif
  int x0, y0;
  tile_origin(P, tile, x0, y0);
  px = x0 + (int)(in_tile & 7u);
  py = y0 + (int)(in_tile >> 3);
}

// ---------------------------------------------------------------------- trace
// Persistent warps walk the input queue's rays, scheduled as rt_trace.cuh describes: whenever RT_REFILL_MIN_* lanes have
// finished, those lanes append their results to the HIT / MISS queues and take the next rays.  PRIMARY: the ray is generated from the path id — 32 consecutive ids are 32 samples of one pixel
// (RT_PATH_LAYOUT 1), so a warp's rays are coherent.
// MIN_BLOCKS: resident blocks per SM the kernel is compiled for.  Coherent primary rays gain from a fourth block
// (64 registers; -2.8 % on their kernel).  Bounce rays: the long queues of the first bounces gain too (-2.7 % at
// bounce 1: more warps to cover the divergent loads), the short late queues lose 5-10 % to it (their time is the
// slowest ray's latency, which spills lengthen) — the host picks per bounce (rt_render.cu, RT_TRACE_WIDE_BOUNCES).
// MASKED (primary only): a path id whose pixel P.pixel_mask does not select takes no ray, as one outside the image.
// BASED (primary only): the path handed on is P.path_base + q, so the views of one call own disjoint ranges of path ids.
template <bool PRIMARY, int MIN_BLOCKS = (PRIMARY ? RT_TRACE_MIN_BLOCKS_PRIMARY : RT_TRACE_MIN_BLOCKS), bool MASKED = false,
          bool BASED = false>
__global__ void __launch_bounds__(RT_BLOCK, MIN_BLOCKS)
RT_KN(rt_trace_kernel)(const __grid_constant__ StageParams P) {
  extern __shared__ float4 level_store[];          // [depth - 1][2][RT_BLOCK] entry distances of pending levels (2 .. depth)
  const SceneDev &sc = P.scene;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned lt_mask = (1u << lane) - 1u;
  float4 *levels = level_store + threadIdx.x;
  unsigned *counts = P.q.counts + P.bounce * Q_STRIDE;
  const unsigned n_in = PRIMARY ? (P.tiles ? P.tiles[0] * 32u * (unsigned)P.n_samples : P.n_paths) : counts[Q_RAYS];
  unsigned c_rays = 0, c_nodes = 0, c_leaves = 0, c_accepts = 0, c_root_miss = 0;

  const float inv_w = 1.0f / (float)P.width, inv_h = 1.0f / (float)P.height;
  const float aspect = (float)P.width / (float)P.height;

  RayWalk w;
  w.flags = 0; w.leaf = -1; w.hit_slot = -1;
  bool     exhausted = false;
  unsigned q = 0, range_next = 0, range_end = 0;
  uint32_t seed0 = 0;                      // primary: the path's RNG seed, fixed when the ray is generated
  const unsigned total_warps = gridDim.x * (RT_BLOCK / 32);
  unsigned batch = ray_batch_first(n_in, total_warps);

  unsigned walking = 0;                    // lanes whose walk is not finished (WALK_LIVE), kept current across turns
  for (;;) {
    if (walking == 0 || (!exhausted && __popc(~walking) >= (PRIMARY ? RT_REFILL_MIN_PRIMARY : RT_REFILL_MIN_BOUNCE))) {
      // ---- emit: finished lanes hand their path to the next stage
      const bool fin = (w.flags & (WALK_RAY | WALK_LIVE)) == WALK_RAY;
      const bool is_hit = fin && w.hit_slot >= 0;
      const bool is_miss = fin && w.hit_slot < 0;
      if (__any_sync(RT_FULL, fin)) {
        unsigned path = BASED ? P.path_base + q : q;
        uint32_t rng = seed0;
        if (fin) {
          if (PRIMARY) {
            if (P.hit_ids) {                       // parity hook: primary-hit slot of the chunk's first sample
              int px, py, ls;
              path_pixel(P, q, px, py, ls);
              if (ls == 0) P.hit_ids[py * P.width + px] = w.hit_slot;
            }
          } else {
            const float4 b = P.q.ray_b[q];
            path = __float_as_uint(b.z);
            rng  = __float_as_uint(b.w);
          }
        }
#if RT_EMIT_ONE_ATOMIC
        // slots in the HIT and the MISS queue with ONE atomic: the two lengths are the halves of an aligned 64-bit word
        // (a queue is shorter than 2^31, the low half cannot carry into the high one)
        const unsigned hmask = __ballot_sync(RT_FULL, is_hit), mmask = __ballot_sync(RT_FULL, is_miss);
        unsigned long long both = 0;
        if (lane == 0)
          both = atomicAdd(reinterpret_cast<unsigned long long *>(&counts[Q_HITS]),
                           (unsigned long long)__popc(hmask) | ((unsigned long long)__popc(mmask) << 32));
        both = __shfl_sync(RT_FULL, both, 0);
        const unsigned hpos = (unsigned)both + (unsigned)__popc(hmask & lt_mask);
        const unsigned mpos = (unsigned)(both >> 32) + (unsigned)__popc(mmask & lt_mask);
#else
        const unsigned hpos = warp_append(&counts[Q_HITS], is_hit, lane);
        const unsigned mpos = warp_append(&counts[Q_MISSES], is_miss, lane);
#endif
        if (is_hit) {
          P.q.hit_a[hpos] = make_float4(w.ox, w.oy, w.oz, w.dx);
          P.q.hit_b[hpos] = make_float4(w.dy, w.dz, __uint_as_float(path), __uint_as_float(rng));
          P.q.hit_h[hpos] = make_float4(w.hit_t, w.hit_u, w.hit_v, __int_as_float(w.hit_slot));
        }
        if (is_miss) {
          P.q.miss_a[mpos] = make_float4(w.dx, w.dy, w.dz, __uint_as_float(path));
        }
        if (fin) w.flags = 0;
      }
      // ---- refill: lanes that are not walking take the next rays of the warp's reserved range;
      // a warp reserves `batch` consecutive rays per atomic (one round trip per batch, not per refill)
      if (!exhausted) {
        const unsigned idle = ~walking;
        if (range_next >= range_end) {
          const unsigned base = ray_fetch(&counts[Q_FETCH], batch, lane);
          exhausted = base >= n_in;
          range_next = base;
          range_end = exhausted ? base : min(base + batch, n_in);
          batch = ray_batch_next(batch, n_in - range_end, total_warps);
        }
        const unsigned take = min((unsigned)__popc(idle), range_end - range_next);
        const unsigned rank = (unsigned)__popc(idle & lt_mask);
        if ((idle >> lane & 1u) && rank < take) {
          q = range_next + rank;
          bool ok = true;
          float ox = 0, oy = 0, oz = 0, dx = 0, dy = 0, dz = -1;
          if (PRIMARY) {
            int px = 0, py = 0, ls = 0;
            path_pixel(P, q, px, py, ls);
            ok = px < P.width && py < P.height;
            if (MASKED && ok) ok = P.pixel_mask[py * P.width + px] != 0;
            if (ok) {
              const int s = P.sample0 + ls;
              camera_dir(sc, px, py, s, inv_w, inv_h, aspect, dx, dy, dz);
              ox = sc.view[0][3]; oy = sc.view[1][3]; oz = sc.view[2][3];       // raytracer.c:612
              seed0 = rt_path_seed((uint32_t)(py * P.width + px), (uint32_t)s, P.user_seed);
            }
          } else {
            const float4 a = P.q.ray_a[q], b = P.q.ray_b[q];
            ox = a.x; oy = a.y; oz = a.z; dx = a.w; dy = b.x; dz = b.y;
          }
          if (ok) {
            walk_begin(w, sc, ox, oy, oz, dx, dy, dz);
            c_rays++;
            if (walk_misses_root<PRIMARY>(w, sc)) { w.flags = WALK_RAY; c_nodes++; c_root_miss++; }      // the root visit, nothing entered
            // the root visit here, among the lanes that just took a ray (all at the same node), instead of in a voted turn
            else walk_node_step<PRIMARY, true>(w, sc, levels, c_nodes);
          }
        }
        range_next += take;
      }
      walking = __ballot_sync(RT_FULL, w.flags & WALK_LIVE);
      if (walking == 0) {
        // nobody walks: rays that finished at their root visit go out on the next turn; with none of those either
        // the queue is drained — or (chunk split) the 32 ids just taken were a job tile that lies outside the
        // image, or (MASKED) pixels the mask does not select, and the warp's reserved range goes on
        if (exhausted && __ballot_sync(RT_FULL, w.flags & WALK_RAY) == 0) break;
        continue;
      }
    }

    if (PRIMARY) {
      // coherent rays reach their leaves in nearly the same number of steps: plain while-while — every
      // lane walks until it holds a leaf (or is done), then the warp tests the triangles together
      // (measured 2.8 % faster than voting for them)
      while ((w.flags & (WALK_LIVE | WALK_LEAF)) == WALK_LIVE) walk_node_step<PRIMARY>(w, sc, levels, c_nodes);
      __syncwarp();
      if (w.flags & WALK_LEAF) walk_leaf<PRIMARY>(w, sc, c_leaves, c_accepts);
    } else {
      walk_turn_voted<PRIMARY>(w, sc, levels, walking, c_nodes, c_leaves, c_accepts);
    }
    walking = __ballot_sync(RT_FULL, w.flags & WALK_LIVE);
  }

  if (P.counters) {
    add_counter(P.counters, 0, c_rays);
    add_counter(P.counters, 1, c_nodes);
    add_counter(P.counters, 2, c_leaves);
    add_counter(P.counters, 3, c_accepts);
  }
  if (P.counters_ex) {
    add_counter(P.counters_ex, 0, c_root_miss);
    if (PRIMARY) add_counter(P.counters_ex, 1, c_rays);
  }
}

// ----------------------------------------------------------------------- miss
// raytracer.c:554: background(direction) * tint + emission ends the path.
// 32 registers (8 blocks per SM): the same time on the long bounce-0 queue, -7 % on bounce 1 (449 vs 484 us)
#ifndef RT_MISS_MIN_BLOCKS
#define RT_MISS_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(256, RT_MISS_MIN_BLOCKS)
RT_KN(rt_miss_kernel)(const __grid_constant__ StageParams P) {
  const unsigned n = P.q.counts[P.bounce * Q_STRIDE + Q_MISSES];
  unsigned done = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 a = P.q.miss_a[i];
    V3 env = environment(P.scene, mk3(a.x, a.y, a.z));
    V3 radiance;
    if (P.bounce == 0) {
      // primary rays carry tint 1 and emission 0 (raytracer.c:507-510): their records are not stored;
      // env * 1 + 0 is env bit for bit (a -0 channel would become +0, the environment is never negative)
      radiance = env;
    } else {
      const float4 t = P.q.tint[__float_as_uint(a.w)], e = P.q.emis[__float_as_uint(a.w)];
      radiance = add3(mul3(env, mk3(t.x, t.y, t.z)), mk3(e.x, e.y, e.z));
    }
    P.q.rad[__float_as_uint(a.w)] = make_float4(radiance.x, radiance.y, radiance.z, 0);
    done++;
  }
  if (P.counters) {
    add_counter(P.counters, 5, done);
    add_counter(P.counters, 7, done);
  }
}

// ------------------------------------------------------------------------ sky
// The camera samples of the sky tiles: job tiles no jittered camera ray of which can reach the root-union box
// (rt_render.cu), so every such ray is one the primary trace would end at walk_misses_root and the bounce-0 miss kernel
// would give the environment.  Here that is done without the path queues: one thread per pixel (a warp is one sky tile,
// so its lanes look up neighbouring directions together), looping over the call's samples [sample0, sample0 + n_samples)
// and summing each one as it comes — the sum (and v * v) in sample order exactly as accumulate_pixels forms it.  The
// counters gain what the trace and the miss kernel add for such rays.
// P.accumulate: the sum starts from P.accum (else +0); P.hit_ids gets -1 (no primary hit) for the call's first sample.
// 60 registers, 4 blocks per SM: 4.36 ms for the 286 M sky samples of a 256-spp helmet frame.  Capped at 48 / 40 registers
// (5 / 6 blocks) the environment lookup spills: the bounce-0 miss stage (miss + sky) takes 7.09 / 7.12 / 7.22 ms at 4 / 5 / 6
#ifndef RT_SKY_MIN_BLOCKS
#define RT_SKY_MIN_BLOCKS 4
#endif
__global__ void __launch_bounds__(256, RT_SKY_MIN_BLOCKS)
RT_KN(rt_sky_kernel)(const __grid_constant__ StageParams P) {
  const SceneDev &sc = P.scene;
  const float inv_w = 1.0f / (float)P.width, inv_h = 1.0f / (float)P.height;
  const float aspect = (float)P.width / (float)P.height;
  const unsigned n_pixels = P.tiles[1] * 32u;
  const unsigned *sky = P.tiles + 2 + P.n_tiles - 1;          // sky tile j at sky[-j]
  unsigned c_samples = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pixels; i += gridDim.x * blockDim.x) {
    int x0, y0;
    tile_origin(P, sky[-(int)(i >> 5)], x0, y0);
    const int px = x0 + (int)(i & 7u), py = y0 + (int)((i >> 3) & 3u);
    if (px >= P.width || py >= P.height) continue;
    const int pixel = py * P.width + px;
    if (P.pixel_mask && !P.pixel_mask[pixel]) {              // as the masked accumulate: zeroed or left alone
      if (!P.accumulate) {
        P.accum[3 * pixel + 0] = 0; P.accum[3 * pixel + 1] = 0; P.accum[3 * pixel + 2] = 0;
        if (P.accum_sq) { P.accum_sq[3 * pixel + 0] = 0; P.accum_sq[3 * pixel + 1] = 0; P.accum_sq[3 * pixel + 2] = 0; }
      }
      continue;
    }
    V3 sum = P.accumulate ? mk3(P.accum[3 * pixel], P.accum[3 * pixel + 1], P.accum[3 * pixel + 2]) : mk3(0, 0, 0);
    V3 sq = mk3(0, 0, 0);
    if (P.accum_sq && P.accumulate) sq = mk3(P.accum_sq[3 * pixel], P.accum_sq[3 * pixel + 1], P.accum_sq[3 * pixel + 2]);
    for (int s = 0; s < P.n_samples; s++) {
      float dx, dy, dz;
      camera_dir(sc, px, py, P.sample0 + s, inv_w, inv_h, aspect, dx, dy, dz);
      const V3 v = environment(sc, mk3(dx, dy, dz));          // bounce 0: tint 1, emission 0 (rt_miss_kernel)
      sum = add3(sum, v);
      if (P.accum_sq) sq = add3(sq, mul3(v, v));
      if (P.per_sample) {
        float *dst = P.per_sample + ((size_t)pixel * (size_t)P.per_sample_stride + (size_t)(P.per_sample_offset + s)) * 3;
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z;
      }
    }
    P.accum[3 * pixel + 0] = sum.x; P.accum[3 * pixel + 1] = sum.y; P.accum[3 * pixel + 2] = sum.z;
    if (P.accum_sq) { P.accum_sq[3 * pixel + 0] = sq.x; P.accum_sq[3 * pixel + 1] = sq.y; P.accum_sq[3 * pixel + 2] = sq.z; }
    if (P.hit_ids) P.hit_ids[pixel] = -1;
    c_samples += (unsigned)P.n_samples;
  }
  // per ray: the trace's ray, root visit and root-union miss (and primary ray), the miss kernel's miss and sample
  if (P.counters) {
    add_counter(P.counters, 0, c_samples);
    add_counter(P.counters, 1, c_samples);
    add_counter(P.counters, 5, c_samples);
    add_counter(P.counters, 7, c_samples);
  }
  if (P.counters_ex) {
    add_counter(P.counters_ex, 0, c_samples);
    add_counter(P.counters_ex, 1, c_samples);
  }
}

// ---------------------------------------------------------------------- shade
// raytracer.c:514-552 for one hit: attribute interpolation (:164-182), back-face
// pass-through, BSDF, emission/tint update, next origin.  Survivors go to the RAY
// queue of bounce + 1; paths that terminate or exhaust max_bounces (:557) write rad.
// raytracer.c:164-182: the shading input at a front-face hit of direction dir, from rows 3..5 of its record, its
// interpolated normal and its geometric normal
__device__ __forceinline__ ShadeIn shade_input(V3 dir, V3 normal, V3 ng, float4 r3, float4 r4, float4 r5,
                                               float w0, float w1, float w2) {
  ShadeIn in;
  in.dir = dir;
  in.normal = normalize3(normal);
  in.normal_geo = ng;
  in.tangent   = rec_tangent(r3);
  in.bitangent = rec_bitangent(r3, r4);
  in.u = rec_tex_u(r4, r5, w0, w1, w2);
  in.v = rec_tex_v(r4, r5, w0, w1, w2);
  return in;
}

// One surface interaction of cast_ray (raytracer.c:514-552) for the hit (t, u, v, slot) of the ray (o, d): returns
// whether the path goes on; o, d, tint, emis and rng are updated in place (emis is the path's radiance if it ends).
__device__ __forceinline__ bool shade_hit(const SceneDev &sc, V3 &o, V3 &d, V3 &tint, V3 &emis,
                                          uint32_t &rng, float hit_t, float hit_u, float hit_v, int slot,
                                          unsigned &c_shades, unsigned &c_pass) {
  const float4 *rec = sc.tri_rec + (size_t)slot * 7;
  float4 r0 = __ldg(rec + 0), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
  V3 ng = rec_normal_geo(r0);
  float w1 = hit_u, w2 = hit_v, w0 = 1 - w1 - w2;                       // raytracer.c:164-177
  V3 point  = hit_point(o, d, hit_t);
  V3 normal = rec_normal(r0, r1, r2, w0, w1, w2);
  if (hit_back_face(ng, normal, d)) {
    // raytracer.c:516-522: back face — step through, the bounce is consumed
    c_pass++;
    o = add3(point, scale3(d, RT_EPS));
    return true;
  }
  float4 r3 = __ldg(rec + 3), r4 = __ldg(rec + 4), r5 = __ldg(rec + 5), r6 = __ldg(rec + 6);
  ShadeIn in = shade_input(d, normal, ng, r3, r4, r5, w0, w1, w2);
  ShadeOut out;
  c_shades++;
  shade_pbr(sc, rec_material(r6), in, rng, out);
  emis = add3(emis, mul3(out.emission, tint));          // raytracer.c:537
  if (out.terminate) return false;
  d = out.dir;
  tint = mul3(tint, out.tint);
  float bias = (0.5f - (float)(dot3(ng, out.dir) < 0)) * 2.0f * RT_EPS;   // raytracer.c:551
  o = add3(point, scale3(ng, bias));
  return true;
}

// 64 registers (4 blocks per SM): the texel gathers are latency the extra warps cover — 2298 / 2073 / 2169 / 2610 us for
// the bounce-0 launch of a 64-spp helmet chunk at 3 / 4 / 5 / 6 blocks
#ifndef RT_SHADE_MIN_BLOCKS
#define RT_SHADE_MIN_BLOCKS 4
#endif
__global__ void __launch_bounds__(256, RT_SHADE_MIN_BLOCKS)
RT_KN(rt_shade_kernel)(const __grid_constant__ StageParams P) {
  const SceneDev &sc = P.scene;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned n = P.q.counts[P.bounce * Q_STRIDE + Q_HITS];
  unsigned *next_rays = &P.q.counts[(P.bounce + 1) * Q_STRIDE + Q_RAYS];
  const unsigned n_round = (n + 31u) & ~31u;          // whole warps stay in the loop for the collective append
  unsigned c_shades = 0, c_pass = 0, c_samples = 0;

  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
    const bool active = i < n;
    bool  cont = false;
    V3    o = mk3(0, 0, 0), d = mk3(0, 0, 0), tint = mk3(0, 0, 0), emis = mk3(0, 0, 0);
    unsigned path = 0;
    uint32_t rng = 0;
    if (active) {
      const float4 a = P.q.hit_a[i], b = P.q.hit_b[i], h = P.q.hit_h[i];
      o = mk3(a.x, a.y, a.z); d = mk3(a.w, b.x, b.y);
      path = __float_as_uint(b.z); rng = __float_as_uint(b.w);
      tint = mk3(1, 1, 1); emis = mk3(0, 0, 0);            // bounce 0 (raytracer.c:507-510): not stored
      if (P.bounce > 0) {
        const float4 c = P.q.tint[path], e = P.q.emis[path];
        tint = mk3(c.x, c.y, c.z); emis = mk3(e.x, e.y, e.z);
      }
      cont = shade_hit(sc, o, d, tint, emis, rng, h.x, h.y, h.z, __float_as_int(h.w), c_shades, c_pass);
      if (P.bounce + 1 >= P.max_bounces) cont = false;        // raytracer.c:557
      if (!cont) {
        P.q.rad[path] = make_float4(emis.x, emis.y, emis.z, 0);
        c_samples++;
      }
    }
    const unsigned pos = warp_append(next_rays, cont, lane);
    if (cont) {
      P.q.ray_a[pos] = make_float4(o.x, o.y, o.z, d.x);
      P.q.ray_b[pos] = make_float4(d.y, d.z, __uint_as_float(path), __uint_as_float(rng));
      P.q.tint[path] = make_float4(tint.x, tint.y, tint.z, 0);
      P.q.emis[path] = make_float4(emis.x, emis.y, emis.z, 0);
    }
  }
  if (P.counters) {
    add_counter(P.counters, 4, c_shades);
    add_counter(P.counters, 6, c_pass);
    add_counter(P.counters, 7, c_samples);
  }
}

