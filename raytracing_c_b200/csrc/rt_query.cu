// rt_query.cu — batched ray queries on a resident scene: closest hit and occlusion (include/rt_gpu.h).
//
// The walk is rt_trace.cuh's, unchanged: the reference's ray_scene_hit (raytracer.c:443-503) with hit.distance set to
// the ray's t_max before it starts.  The scheduling is the bounce trace kernel's by construction (rt_trace.cuh): the
// same reservation of ray ranges (ray_batch_first, ray_fetch, ray_batch_next), the refill at RT_REFILL_MIN_BOUNCE idle
// lanes with the root visit, and the voted turn (walk_turn_voted).  What is the queries' own is the input and output:
// rays are read and results stored at the ray's own index, so there are no queues and no append atomics.
//
// Occlusion (ANY): a lane is finished after the first leaf that accepts a triangle.  Up to that leaf its hit_t is still
// t_max, so its walk is the closest-hit walk's prefix: the same nodes in the same order, never more of them.
//
// Built with -fmad=false like rt_render.cu (the exact build): queries are never FMA-contracted.
#include <cuda_runtime.h>
#include <math_constants.h>

#include "rt_trace.cuh"
#include "rt_kernels.h"

// 64 registers: 4 blocks of 256 threads per SM, the build of the wide bounce trace (rt_trace_kernel<false, 4>)
#ifndef RT_QUERY_MIN_BLOCKS
#define RT_QUERY_MIN_BLOCKS 4
#endif

// raytracer.c:164-177 for the surface record: point, interpolated and geometric normal and tex_coords of the hit, read
// through the shading-record accessors (rt_device.cuh) as shade_hit reads them
__device__ __forceinline__ void store_surface(const SceneDev &sc, float *out, const RayWalk &w) {
  float s[11];
  if (w.hit_slot >= 0) {
    const float4 *rec = sc.tri_rec + (size_t)w.hit_slot * 7;
    const float4 r0 = __ldg(rec + 0), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
    const float4 r4 = __ldg(rec + 4), r5 = __ldg(rec + 5);
    const V3 ng = rec_normal_geo(r0);
    const float w1 = w.hit_u, w2 = w.hit_v, w0 = 1 - w1 - w2;
    const V3 point = hit_point(mk3(w.ox, w.oy, w.oz), mk3(w.dx, w.dy, w.dz), w.hit_t);
    const V3 normal = rec_normal(r0, r1, r2, w0, w1, w2);
    s[0] = point.x; s[1] = point.y; s[2] = point.z;
    s[3] = normal.x; s[4] = normal.y; s[5] = normal.z;
    s[6] = ng.x; s[7] = ng.y; s[8] = ng.z;
    s[9]  = rec_tex_u(r4, r5, w0, w1, w2);
    s[10] = rec_tex_v(r4, r5, w0, w1, w2);
  } else {
    #pragma unroll
    for (int k = 0; k < 11; k++) s[k] = 0.0f;
  }
  #pragma unroll
  for (int k = 0; k < 11; k++) out[k] = s[k];
}

template <bool ANY>
__global__ void __launch_bounds__(RT_BLOCK, RT_QUERY_MIN_BLOCKS)
rt_query_kernel(const __grid_constant__ QueryParams P) {
  extern __shared__ float4 level_store[];          // [depth - 1][2][RT_BLOCK]: the trace kernel's level store
  const SceneDev &sc = P.scene;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned lt_mask = (1u << lane) - 1u;
  float4 *levels = level_store + threadIdx.x;
  const unsigned n_in = P.n_rays;
  unsigned c_rays = 0, c_nodes = 0, c_leaves = 0, c_accepts = 0;

  RayWalk w;
  w.flags = 0; w.leaf = -1; w.hit_slot = -1;
  bool     exhausted = false;
  unsigned q = 0, range_next = 0, range_end = 0;
  const unsigned total_warps = gridDim.x * (RT_BLOCK / 32);
  unsigned batch = ray_batch_first(n_in, total_warps);

  unsigned walking = 0;
  for (;;) {
    if (walking == 0 || (!exhausted && __popc(~walking) >= RT_REFILL_MIN_BOUNCE)) {
      // ---- store: finished lanes write their result at their ray's index
      if ((w.flags & (WALK_RAY | WALK_LIVE)) == WALK_RAY) {
        if (ANY) {
          P.occluded[q] = w.hit_slot >= 0 ? 1 : 0;
        } else {
          const bool hit = w.hit_slot >= 0;
          P.hits[q] = make_float4(hit ? w.hit_t : CUDART_INF_F, w.hit_u, w.hit_v, __int_as_float(w.hit_slot));
          if (P.surface) store_surface(sc, P.surface + (size_t)q * 11, w);
        }
        w.flags = 0;
      }
      // ---- refill: idle lanes take the next rays of the warp's reserved range
      if (!exhausted) {
        const unsigned idle = ~walking;
        if (range_next >= range_end) {
          const unsigned base = ray_fetch(P.fetch, batch, lane);
          exhausted = base >= n_in;
          range_next = base;
          range_end = exhausted ? base : min(base + batch, n_in);
          batch = ray_batch_next(batch, n_in - range_end, total_warps);
        }
        const unsigned take = min((unsigned)__popc(idle), range_end - range_next);
        const unsigned rank = (unsigned)__popc(idle & lt_mask);
        if ((idle >> lane & 1u) && rank < take) {
          q = range_next + rank;
          const float *r = P.rays + (size_t)q * 6;
          walk_begin(w, sc, __ldg(r), __ldg(r + 1), __ldg(r + 2), __ldg(r + 3), __ldg(r + 4), __ldg(r + 5));
          // the reference's hit.distance before the walk: every box and triangle compare reads it
          w.hit_t = P.t_max ? __ldg(P.t_max + q) : CUDART_INF_F;
          c_rays++;
          // a regular ray that misses the root union at +inf misses it at every smaller t_max (and NaN acts as +inf
          // in the box test: both the reference's MINPS and fminf return the other operand)
          if (walk_misses_root<false>(w, sc)) { w.flags = WALK_RAY; c_nodes++; }
          else walk_node_step<false, true>(w, sc, levels, c_nodes);
        }
        range_next += take;
      }
      walking = __ballot_sync(RT_FULL, w.flags & WALK_LIVE);
      if (walking == 0) {
        if (exhausted && __ballot_sync(RT_FULL, w.flags & WALK_RAY) == 0) break;
        continue;
      }
    }

    walk_turn_voted<false>(w, sc, levels, walking, c_nodes, c_leaves, c_accepts);
    // the first accepted triangle answers the query (hit_slot changes only in walk_leaf, walk_begin resets it)
    if (ANY && w.hit_slot >= 0) w.flags &= ~WALK_LIVE;
    walking = __ballot_sync(RT_FULL, w.flags & WALK_LIVE);
  }

  if (P.counters) {
    add_counter(P.counters, 0, c_rays);
    add_counter(P.counters, 1, c_nodes);
    add_counter(P.counters, 2, c_leaves);
    add_counter(P.counters, 3, c_accepts);
  }
}

// dynamic shared memory opt-in and occupancy per device (cudaFuncSetAttribute is per device)
static int g_query_blocks_per_sm[RT_MAX_DEVICES][2];
static size_t g_query_level_bytes[RT_MAX_DEVICES];

int rt_launch_query(const QueryParams &p, bool any, int sm_count, cudaStream_t stream) {
  const size_t level_bytes = level_store_bytes(p.scene.depth);
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= RT_MAX_DEVICES) return (int)cudaErrorInvalidDevice;
  if (g_query_blocks_per_sm[dev][0] == 0 || level_bytes != g_query_level_bytes[dev]) {
    g_query_blocks_per_sm[dev][0] = level_store_blocks_per_sm((const void *)rt_query_kernel<false>, level_bytes);
    g_query_blocks_per_sm[dev][1] = level_store_blocks_per_sm((const void *)rt_query_kernel<true>, level_bytes);
    g_query_level_bytes[dev] = level_bytes;
  }
  const unsigned grid = (unsigned)(sm_count * g_query_blocks_per_sm[dev][any ? 1 : 0]);     // persistent: one wave
  if (any) rt_query_kernel<true><<<grid, RT_BLOCK, level_bytes, stream>>>(p);
  else     rt_query_kernel<false><<<grid, RT_BLOCK, level_bytes, stream>>>(p);
  return (int)cudaGetLastError();
}
