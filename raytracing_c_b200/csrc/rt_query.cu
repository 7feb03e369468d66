// rt_query.cu — batched ray queries on a resident scene: closest hit and occlusion (include/rt_gpu.h).
//
// The walk is rt_trace.cuh's, unchanged: the reference's ray_scene_hit (raytracer.c:443-503) with hit.distance set to
// the ray's t_max before it starts.  The scheduling is the bounce trace kernel's (rt_stages.cuh): a persistent grid,
// each warp reserves ranges of ray indices with one atomic per range, lanes refill when RT_REFILL_MIN_BOUNCE of them
// are idle, node and leaf turns go by majority vote.  What differs is the input and output: rays are read and results
// stored at the ray's own index, so there are no queues and no append atomics.
//
// Occlusion (ANY): a lane is finished after the first leaf that accepts a triangle.  Up to that leaf its hit_t is still
// t_max, so its walk is the closest-hit walk's prefix: the same nodes in the same order, never more of them.
//
// Built with -fmad=false like rt_render.cu (the exact build): queries are never FMA-contracted.
#include <cuda_runtime.h>
#include <math_constants.h>

#include "rt_trace.cuh"
#include "rt_kernels.h"

// The scheduling constants and the counter reduction of the bounce trace kernel (rt_stages.cuh, which cannot be
// included here: it defines the stage kernels, and a second translation unit would link them twice).
#define RT_Q_FULL 0xffffffffu
#define RT_Q_BATCH_MAX 256u            // RT_BATCH_MAX
#define RT_Q_MIN_BATCH 4u              // RT_MIN_BATCH
#define RT_Q_REFILL_MIN 20             // RT_REFILL_MIN_BOUNCE
// 64 registers: 4 blocks of 256 threads per SM, the build of the wide bounce trace (rt_trace_kernel<false, 4>)
#ifndef RT_QUERY_MIN_BLOCKS
#define RT_QUERY_MIN_BLOCKS 4
#endif

__device__ __forceinline__ void query_add_counter(unsigned long long *counters, int k, unsigned v) {
  v += __shfl_xor_sync(RT_Q_FULL, v, 16);
  v += __shfl_xor_sync(RT_Q_FULL, v, 8);
  v += __shfl_xor_sync(RT_Q_FULL, v, 4);
  v += __shfl_xor_sync(RT_Q_FULL, v, 2);
  v += __shfl_xor_sync(RT_Q_FULL, v, 1);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(&counters[k], (unsigned long long)v);
}

// raytracer.c:164-177 for the surface record: the expressions of shade_hit (rt_stages.cuh) and the tex_coords of
// raytracer.c:175-176 (shade_hit's in.u / in.v), gathered from the shading record of the slot
__device__ __forceinline__ void store_surface(const SceneDev &sc, float *out, const RayWalk &w) {
  float s[11];
  if (w.hit_slot >= 0) {
    const float4 *rec = sc.tri_rec + (size_t)w.hit_slot * 7;
    const float4 r0 = __ldg(rec + 0), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
    const float4 r4 = __ldg(rec + 4), r5 = __ldg(rec + 5);
    const V3 ng = mk3(r0.x, r0.y, r0.z);
    const V3 na = mk3(r0.w, r1.x, r1.y), nb = mk3(r1.z, r1.w, r2.x), nc = mk3(r2.y, r2.z, r2.w);
    const float w1 = w.hit_u, w2 = w.hit_v, w0 = 1 - w1 - w2;
    const V3 point = add3(mk3(w.ox, w.oy, w.oz), scale3(mk3(w.dx, w.dy, w.dz), w.hit_t));
    s[0] = point.x; s[1] = point.y; s[2] = point.z;
    s[3] = na.x * w0 + nb.x * w1 + nc.x * w2;
    s[4] = na.y * w0 + nb.y * w1 + nc.y * w2;
    s[5] = na.z * w0 + nb.z * w1 + nc.z * w2;
    s[6] = ng.x; s[7] = ng.y; s[8] = ng.z;
    s[9]  = r4.z * w0 + r5.x * w1 + r5.z * w2;
    s[10] = r4.w * w0 + r5.y * w1 + r5.w * w2;
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
  unsigned batch = (n_in / (total_warps * 4u)) & ~31u;
  if (batch > RT_Q_BATCH_MAX) batch = RT_Q_BATCH_MAX;
  if (batch < 32u) {
    batch = (n_in + total_warps - 1u) / total_warps;
    if (batch < RT_Q_MIN_BATCH) batch = RT_Q_MIN_BATCH;
    if (batch > 32u) batch = 32u;
  }

  unsigned walking = 0;
  for (;;) {
    if (walking == 0 || (!exhausted && __popc(~walking) >= RT_Q_REFILL_MIN)) {
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
      // ---- refill: idle lanes take the next rays of the warp's reserved range (guided self-scheduling)
      if (!exhausted) {
        const unsigned idle = ~walking;
        if (range_next >= range_end) {
          unsigned base = 0;
          if (lane == 0) base = atomicAdd(P.fetch, batch);
          base = __shfl_sync(RT_Q_FULL, base, 0);
          exhausted = base >= n_in;
          range_next = base;
          range_end = exhausted ? base : min(base + batch, n_in);
          if (batch > 32u) {
            const unsigned share = ((n_in - range_end) / (total_warps * 2u)) & ~31u;
            batch = share < 32u ? 32u : (share < batch ? share : batch);
          }
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
      walking = __ballot_sync(RT_Q_FULL, w.flags & WALK_LIVE);
      if (walking == 0) {
        if (exhausted && __ballot_sync(RT_Q_FULL, w.flags & WALK_RAY) == 0) break;
        continue;
      }
    }

    const unsigned want_leaf = __ballot_sync(RT_Q_FULL, w.flags & WALK_LEAF);
    if (2 * __popc(want_leaf) <= __popc(walking)) {
      if ((w.flags & (WALK_LIVE | WALK_LEAF)) == WALK_LIVE) walk_node_step<false>(w, sc, levels, c_nodes);
    } else if (w.flags & WALK_LEAF) {
      walk_leaf<false>(w, sc, c_leaves, c_accepts);
      if (ANY && w.hit_slot >= 0) w.flags &= ~WALK_LIVE;       // the first accepted triangle answers the query
    }
    walking = __ballot_sync(RT_Q_FULL, w.flags & WALK_LIVE);
  }

  if (P.counters) {
    query_add_counter(P.counters, 0, c_rays);
    query_add_counter(P.counters, 1, c_nodes);
    query_add_counter(P.counters, 2, c_leaves);
    query_add_counter(P.counters, 3, c_accepts);
  }
}

// dynamic shared memory opt-in and occupancy per device (cudaFuncSetAttribute is per device)
static int g_query_blocks_per_sm[RT_MAX_DEVICES][2];
static size_t g_query_level_bytes[RT_MAX_DEVICES];

int rt_launch_query(const QueryParams &p, bool any, int sm_count, cudaStream_t stream) {
  const size_t level_bytes = (size_t)(p.scene.depth > 1 ? p.scene.depth - 1 : 1) * 2 * RT_BLOCK * sizeof(float4);
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= RT_MAX_DEVICES) return (int)cudaErrorInvalidDevice;
  if (g_query_blocks_per_sm[dev][0] == 0 || level_bytes != g_query_level_bytes[dev]) {
    int n = 0;
    cudaFuncSetAttribute(rt_query_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_MAX_DEPTH * 2 * RT_BLOCK * 16);
    cudaFuncSetAttribute(rt_query_kernel<true>,  cudaFuncAttributeMaxDynamicSharedMemorySize, RT_MAX_DEPTH * 2 * RT_BLOCK * 16);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, rt_query_kernel<false>, RT_BLOCK, level_bytes) != cudaSuccess || n < 1) n = 1;
    g_query_blocks_per_sm[dev][0] = n;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, rt_query_kernel<true>, RT_BLOCK, level_bytes) != cudaSuccess || n < 1) n = 1;
    g_query_blocks_per_sm[dev][1] = n;
    g_query_level_bytes[dev] = level_bytes;
  }
  const unsigned grid = (unsigned)(sm_count * g_query_blocks_per_sm[dev][any ? 1 : 0]);     // persistent: one wave
  if (any) rt_query_kernel<true><<<grid, RT_BLOCK, level_bytes, stream>>>(p);
  else     rt_query_kernel<false><<<grid, RT_BLOCK, level_bytes, stream>>>(p);
  return (int)cudaGetLastError();
}
