// rt_trace.cuh — closest-hit BVH traversal, one thread per ray.
//
// Replaces reference raytracer.c:190-230 (ray_aabbs_hit_8), :84-188
// (ray_triangles_hit_8), :15-32 (min_f32x8) and :443-503 (ray_bvh_node_hit /
// ray_scene_hit).  The reference's AVX2 8-wide box and triangle tests become
// eight scalar tests per lane, so a warp tests 256 boxes per node step with no
// cross-lane traffic.  All arithmetic is IEEE f32 in the reference's operation
// order without FMA contraction (-fmad=false): visit order, every compare and the
// closest hit (ties included) are the reference's.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>

#include "rt_device.cuh"

#ifndef RT_BLOCK
#define RT_BLOCK 256
#endif
#define RT_FULL 0xffffffffu

// raytracer.c:190-230 for ONE child box, general form: the reference's nested MINPS/MAXPS with
// their "second operand when unordered" rule, as operand-order selects.  Needed only when a
// reciprocal direction component is infinite (0 * inf = NaN lanes, raytracer.c:212-225).
__device__ __forceinline__ float child_entry_any(float lox, float loy, float loz, float hix, float hiy, float hiz,
                                                 float ox, float oy, float oz, float ix, float iy, float iz, float t_max) {
  float ax = (lox - ox) * ix, ay = (loy - oy) * iy, az = (loz - oz) * iz;
  float bx = (hix - ox) * ix, by = (hiy - oy) * iy, bz = (hiz - oz) * iz;
  float nx = sel_min(ax, bx), ny = sel_min(ay, by), nz = sel_min(az, bz);
  float fx = sel_max(ax, bx), fy = sel_max(ay, by), fz = sel_max(az, bz);
  float enter = sel_max(RT_EPS, sel_max(nx, sel_max(ny, nz)));
  float leave = sel_min(t_max,  sel_min(fx, sel_min(fy, fz)));
  return (enter >= leave) ? CUDART_INF_F : enter;
}

// The same box for a REGULAR ray (all three reciprocals finite, so every product is finite and
// no NaN rule can fire).  IEEE subtraction and multiplication are monotonic and lo <= hi for every
// box scene_init writes (EPSILON-inflated, or all-zero padding), so (lo - o) * i <= (hi - o) * i
// when i > 0 and >= when i < 0: min(a, b) / max(a, b) of the reference are known from the sign
// of i alone.  The caller hands in the near and far plane per axis; the values — and therefore
// enter, leave and the compare — are the reference's (a zero's sign can differ, but enter >= EPS
// and leave is only compared).
// REL: the planes are already relative to the ray origin (camera-relative node copy, see
// rt_camera_relative_kernel) — the same f32 subtraction, done once per frame instead of per ray.
template <bool REL>
__device__ __forceinline__ float child_entry_regular(float nx, float ny, float nz, float fx, float fy, float fz,
                                                     float ox, float oy, float oz, float ix, float iy, float iz, float t_max) {
#if defined(RT_FAST) && RT_FAST
  // fast build: (plane - o) * i as one fused multiply-add, plane * i + (-o * i); the caller hands in -o * i for o
  // (12 instead of 18 instructions per box; not the reference's rounding)
  if (!REL) {
    float enter = fmaxf(fmaxf(fmaf(nx, ix, ox), fmaf(ny, iy, oy)), fmaxf(fmaf(nz, iz, oz), RT_EPS));
    float leave = fminf(fminf(fmaf(fx, ix, ox), fmaf(fy, iy, oy)), fminf(fmaf(fz, iz, oz), t_max));
    return (enter >= leave) ? CUDART_INF_F : enter;
  }
#endif
  if (!REL) { nx -= ox; ny -= oy; nz -= oz; fx -= ox; fy -= oy; fz -= oz; }
  float enter = fmaxf(fmaxf(nx * ix, ny * iy), fmaxf(nz * iz, RT_EPS));
  float leave = fminf(fminf(fx * ix, fy * iy), fminf(fz * iz, t_max));
  return (enter >= leave) ? CUDART_INF_F : enter;
}

// raytracer.c:190-230, ray_aabbs_hit_8: the eight children of one node, entry distance or +inf.
// A node is six 32-byte rows = twelve 16-byte vectors (min x/y/z at vectors 0/2/4, max x/y/z at 6/8/10; child j
// in column j): twelve 16-byte loads, warp-uniform for coherent rays.  on* is, per axis, the vector index of
// the row that holds the NEAR plane (the max row when the direction is negative on that axis) — fixed when
// the walk begins, so a node step pays one address add per row and no selects.
#define RT_ROW_X_SUM  6u     // near + far vector index of an axis: 0 + 6, 2 + 8, 4 + 10
#define RT_ROW_Y_SUM 10u
#define RT_ROW_Z_SUM 14u
// `upper` false: children 4..7 are known padding boxes (lo == hi on every axis).  Their near and far plane coincide,
// so enter = max(EPS, a, b, c) >= a >= min(t_max, a, b, c) = leave whatever the ray: the reference's test yields +inf
// for them, and so does skipping it.
template <bool REL>
__device__ __forceinline__ void node_entries_regular(const float4 *__restrict__ nb, unsigned onx, unsigned ony, unsigned onz,
                                                     float ox, float oy, float oz, float ix, float iy, float iz,
                                                     float t_max, float (&e)[8], bool upper = true) {
  const float4 *pnx = nb + onx, *pny = nb + ony, *pnz = nb + onz;
  const float4 *pfx = nb + (RT_ROW_X_SUM - onx), *pfy = nb + (RT_ROW_Y_SUM - ony), *pfz = nb + (RT_ROW_Z_SUM - onz);
  #pragma unroll
  for (int h = 0; h < 2; h++) {
    if (h == 1 && !upper) { e[4] = e[5] = e[6] = e[7] = CUDART_INF_F; break; }
    float4 nx = __ldg(pnx + h), ny = __ldg(pny + h), nz = __ldg(pnz + h);
    float4 fx = __ldg(pfx + h), fy = __ldg(pfy + h), fz = __ldg(pfz + h);
    e[4 * h + 0] = child_entry_regular<REL>(nx.x, ny.x, nz.x, fx.x, fy.x, fz.x, ox, oy, oz, ix, iy, iz, t_max);
    e[4 * h + 1] = child_entry_regular<REL>(nx.y, ny.y, nz.y, fx.y, fy.y, fz.y, ox, oy, oz, ix, iy, iz, t_max);
    e[4 * h + 2] = child_entry_regular<REL>(nx.z, ny.z, nz.z, fx.z, fy.z, fz.z, ox, oy, oz, ix, iy, iz, t_max);
    e[4 * h + 3] = child_entry_regular<REL>(nx.w, ny.w, nz.w, fx.w, fy.w, fz.w, ox, oy, oz, ix, iy, iz, t_max);
  }
}

// out of line and by value: the rare path must not cost the common one registers or code
struct Entries8 { float4 lo, hi; };
static __device__ __noinline__ Entries8 node_entries_any(const float4 *__restrict__ n4, float ox, float oy, float oz,
                                                  float ix, float iy, float iz, float t_max) {
  Entries8 r;
  {
    float4 lx = __ldg(n4 + 0), ly = __ldg(n4 + 2), lz = __ldg(n4 + 4), hx = __ldg(n4 + 6), hy = __ldg(n4 + 8), hz = __ldg(n4 + 10);
    r.lo.x = child_entry_any(lx.x, ly.x, lz.x, hx.x, hy.x, hz.x, ox, oy, oz, ix, iy, iz, t_max);
    r.lo.y = child_entry_any(lx.y, ly.y, lz.y, hx.y, hy.y, hz.y, ox, oy, oz, ix, iy, iz, t_max);
    r.lo.z = child_entry_any(lx.z, ly.z, lz.z, hx.z, hy.z, hz.z, ox, oy, oz, ix, iy, iz, t_max);
    r.lo.w = child_entry_any(lx.w, ly.w, lz.w, hx.w, hy.w, hz.w, ox, oy, oz, ix, iy, iz, t_max);
  }
  {
    float4 lx = __ldg(n4 + 1), ly = __ldg(n4 + 3), lz = __ldg(n4 + 5), hx = __ldg(n4 + 7), hy = __ldg(n4 + 9), hz = __ldg(n4 + 11);
    r.hi.x = child_entry_any(lx.x, ly.x, lz.x, hx.x, hy.x, hz.x, ox, oy, oz, ix, iy, iz, t_max);
    r.hi.y = child_entry_any(lx.y, ly.y, lz.y, hx.y, hy.y, hz.y, ox, oy, oz, ix, iy, iz, t_max);
    r.hi.z = child_entry_any(lx.z, ly.z, lz.z, hx.z, hy.z, hz.z, ox, oy, oz, ix, iy, iz, t_max);
    r.hi.w = child_entry_any(lx.w, ly.w, lz.w, hx.w, hy.w, hz.w, ox, oy, oz, ix, iy, iz, t_max);
  }
  return r;
}

// fminf ignores NaN operands: the minimum of the ordered entries (NaN only if all eight are NaN)
__device__ __forceinline__ float min8(const float (&e)[8]) {
  return fminf(fminf(fminf(e[0], e[1]), fminf(e[2], e[3])), fminf(fminf(e[4], e[5]), fminf(e[6], e[7])));
}

// per-thread slice of the level store: levels[(level - 1) * 2 + half][tid]
// (levels 2 .. depth: a node of level 1 hands out leaves and never parks its entries — its slot is not allocated)
#define RT_LEVELS(level, half) levels[(((level) - 2) * 2 + (half)) * RT_BLOCK]

// The level store of a block: [depth - 1][2][RT_BLOCK] float4 of dynamic shared memory (levels 2 .. depth only: 24 KB
// per block for the depth-4 trees of the shipped models; the driver's default carve-out is the smallest that holds the
// resident blocks — forcing a larger one costs up to 6 %, L1 beyond 96 KB gains nothing: measured)
static inline size_t level_store_bytes(int depth) { return (size_t)(depth > 1 ? depth - 1 : 1) * 2 * RT_BLOCK * sizeof(float4); }

// Opts a walking kernel in to the level store of the deepest tree and returns its resident blocks per SM at level_bytes
// on the current device (at least 1).  cudaFuncSetAttribute is per device: callers keep the result per device.
static inline int level_store_blocks_per_sm(const void *kernel, size_t level_bytes) {
  int n = 0;
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_MAX_DEPTH * 2 * RT_BLOCK * 16);
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, RT_BLOCK, level_bytes) == cudaSuccess && n >= 1 ? n : 1;
}

// raytracer.c:443-503: closest hit of one ray, one thread per ray, as a resumable walk.
// The reference recursion (8 entry distances per level on the C stack, up to 8 selection
// rounds per node) is a flat loop here: the tree is a complete 8-ary heap, parent = (n-1)>>3;
// the current node's entry distances live in registers, those of ancestors that still hold
// untried candidates in shared memory, and `pending` (bit = level) lets a pop jump straight
// to the nearest such ancestor.  Visit order and every compare are the reference's, so the
// closest hit — ties included — is the same triangle slot.
// Shape: two kinds of step, scheduled by the caller (rt_trace_kernel) by majority vote so the
// warp always runs the step most of its lanes are waiting for:
//   walk_node_step  box-test one node and pick its nearest untried child
//   walk_leaf       test the eight triangles of the leaf the lane holds
// The lane's state is one flag word (a warp votes on it every turn — one LOP3 per ballot):
#define WALK_RAY   1u     // the lane holds a ray (walking or finished, not yet emitted)
#define WALK_LIVE  2u     // ... and its walk is not finished
#define WALK_LEAF  4u     // ... and it holds a leaf to test (w.leaf) before the next node step
#define WALK_BOX   8u     // the node just entered still needs its box test
#define WALK_REG  16u     // all three reciprocal direction components are finite
struct RayWalk {
  float ox, oy, oz, dx, dy, dz, ix, iy, iz;
  float hit_t, hit_u, hit_v;
  int   hit_slot;
  int   node, level, leaf;
  unsigned pending, flags;
  unsigned onx, ony, onz;     // vector index of the near-plane row of each axis inside a node (node_entries_regular)
  float e[8];
};

__device__ __forceinline__ void walk_begin(RayWalk &w, const SceneDev &sc, float ox, float oy, float oz,
                                           float dx, float dy, float dz) {
  w.ox = ox; w.oy = oy; w.oz = oz; w.dx = dx; w.dy = dy; w.dz = dz;
  w.ix = 1.0f / dx; w.iy = 1.0f / dy; w.iz = 1.0f / dz;                // raytracer.c:198-202
  // a zero direction component makes 1/d infinite and 0 * inf NaN: only then the slab test
  // needs the exact MINPS/MAXPS operand-order rule (see child_entry_any)
  const bool regular = (fabsf(w.ix) < CUDART_INF_F) & (fabsf(w.iy) < CUDART_INF_F) & (fabsf(w.iz) < CUDART_INF_F);
  w.onx = w.ix < 0.0f ? 6u : 0u; w.ony = w.iy < 0.0f ? 8u : 2u; w.onz = w.iz < 0.0f ? 10u : 4u;
  w.node = 0; w.level = sc.depth;                                       // raytracer.c:501
  w.pending = 0; w.leaf = -1;
  w.flags = WALK_RAY | WALK_LIVE | WALK_BOX | (regular ? WALK_REG : 0u);
  w.hit_t = CUDART_INF_F; w.hit_u = 0; w.hit_v = 0; w.hit_slot = -1;
}

// A regular ray that misses the union of the root's child boxes misses every one of them: the union's
// near planes are <= and its far planes >= each child's, and the slab arithmetic is monotonic, so
// enter_child >= enter_union >= leave_union >= leave_child (same formulas, same rounding).  Such a
// ray's walk is the root visit alone — 18 instructions instead of eight box tests and a selection.
template <bool REL>
__device__ __forceinline__ bool walk_misses_root(const RayWalk &w, const SceneDev &sc) {
  if (!(w.flags & WALK_REG)) return false;
  const bool negx = w.ix < 0.0f, negy = w.iy < 0.0f, negz = w.iz < 0.0f;
  const float nx = negx ? sc.root_hi[0] : sc.root_lo[0], fx = negx ? sc.root_lo[0] : sc.root_hi[0];
  const float ny = negy ? sc.root_hi[1] : sc.root_lo[1], fy = negy ? sc.root_lo[1] : sc.root_hi[1];
  const float nz = negz ? sc.root_hi[2] : sc.root_lo[2], fz = negz ? sc.root_lo[2] : sc.root_hi[2];
  // (the root box itself is not stored relative: six subtractions per ray, once)
#if defined(RT_FAST) && RT_FAST
  return child_entry_regular<false>(nx, ny, nz, fx, fy, fz, -w.ox * w.ix, -w.oy * w.iy, -w.oz * w.iz, w.ix, w.iy, w.iz, CUDART_INF_F) == CUDART_INF_F;
#else
  return child_entry_regular<false>(nx, ny, nz, fx, fy, fz, w.ox, w.oy, w.oz, w.ix, w.iy, w.iz, CUDART_INF_F) == CUDART_INF_F;
#endif
}

// One node step: (box-test the node just entered,) pick the next child; ends with a leaf to test,
// a child to enter on the next step, or the walk finished.
// ROOT: the step is the walk's first (the caller guarantees w.node == 0 with its box test pending): the root's upper
// four children are skipped when the scene's are padding (a 15 000-triangle model fills four of the root's eight).
template <bool REL, bool ROOT = false>
__device__ __forceinline__ void walk_node_step(RayWalk &w, const SceneDev &sc, float4 *levels, unsigned &c_nodes) {
  float (&e)[8] = w.e;
  for (;;) {
    if (w.flags & WALK_BOX) {
      if (w.flags & WALK_REG) {
        const bool upper = !ROOT || !sc.root_upper_empty;
        const size_t first = ROOT ? 0 : (size_t)w.node * 12;
        if (REL) node_entries_regular<true >((const float4 *)sc.nodes_rel + first, w.onx, w.ony, w.onz, 0, 0, 0, w.ix, w.iy, w.iz, w.hit_t, e, upper);
#if defined(RT_FAST) && RT_FAST
        else     node_entries_regular<false>((const float4 *)sc.nodes + first, w.onx, w.ony, w.onz, -w.ox * w.ix, -w.oy * w.iy, -w.oz * w.iz, w.ix, w.iy, w.iz, w.hit_t, e, upper);
#else
        else     node_entries_regular<false>((const float4 *)sc.nodes + first, w.onx, w.ony, w.onz, w.ox, w.oy, w.oz, w.ix, w.iy, w.iz, w.hit_t, e, upper);
#endif
      } else {
        const Entries8 r = node_entries_any((const float4 *)(sc.nodes + (size_t)w.node * 48), w.ox, w.oy, w.oz, w.ix, w.iy, w.iz, w.hit_t);
        e[0] = r.lo.x; e[1] = r.lo.y; e[2] = r.lo.z; e[3] = r.lo.w; e[4] = r.hi.x; e[5] = r.hi.y; e[6] = r.hi.z; e[7] = r.hi.w;
      }
      w.flags &= ~WALK_BOX;
      c_nodes++;
    }
    // raytracer.c:459-472: nearest untried child strictly below the current hit, lowest index on ties
    const float best = min8(e);
    if (!(best < w.hit_t)) {
      if (w.pending == 0) { w.flags &= ~WALK_LIVE; break; }
      const int up = __ffs(w.pending) - 1;
      w.pending &= w.pending - 1;
      #pragma unroll 1
      for (; w.level < up; w.level++) w.node = (w.node - 1) >> 3;
      float4 a = RT_LEVELS(w.level, 0), b = RT_LEVELS(w.level, 1);
      e[0] = a.x; e[1] = a.y; e[2] = a.z; e[3] = a.w; e[4] = b.x; e[5] = b.y; e[6] = b.z; e[7] = b.w;
      continue;
    }
    int pick = 7;
    #pragma unroll
    for (int j = 6; j >= 0; j--) pick = (e[j] == best) ? j : pick;
    #pragma unroll
    for (int j = 0; j < 8; j++) e[j] = (j == pick) ? CUDART_INF_F : e[j];       // raytracer.c:481
    const int child = 8 * w.node + 1 + pick;
    if (w.level == 1) { w.leaf = child - sc.n_internal; w.flags |= WALK_LEAF; break; }
    if (min8(e) < w.hit_t) {                         // other candidates remain: remember this level
      RT_LEVELS(w.level, 0) = make_float4(e[0], e[1], e[2], e[3]);
      RT_LEVELS(w.level, 1) = make_float4(e[4], e[5], e[6], e[7]);
      w.pending |= 1u << w.level;
    }
    w.node = child;
    w.level -= 1;
    w.flags |= WALK_BOX;
    break;
  }
}

// raytracer.c:115-159 for ONE triangle of the leaf: three 16-byte records — p0 and the edges e1 = p1 - p0,
// e2 = p2 - p0 (the same f32 subtractions raytracer.c:116-122 does per ray, done once at upload).
// REL (camera-relative records): A.xyz is tv = o - p0 itself, C.yzw is qv = tv x e1 and `tq4` points at the
// fourth vector, which holds e2 . qv — none depends on the direction, so for rays that share the camera
// origin they are per-triangle constants (rt_camera_relative_kernel evaluates the same f32 expressions).
template <bool REL>
__device__ __forceinline__ void leaf_triangle(RayWalk &w, const float4 A, const float4 B, const float4 C,
                                              const float4 *tq4, int slot) {
  const float e1x = A.w, e1y = B.x, e1z = B.y, e2x = B.z, e2y = B.w, e2z = C.x;
  float pvx = w.dy * e2z - w.dz * e2y, pvy = w.dz * e2x - w.dx * e2z, pvz = w.dx * e2y - w.dy * e2x;
  float det = e1x * pvx + e1y * pvy + e1z * pvz;
  float inv_det = 1.0f / det;
  float tvx = REL ? A.x : w.ox - A.x, tvy = REL ? A.y : w.oy - A.y, tvz = REL ? A.z : w.oz - A.z;
  float u = inv_det * (tvx * pvx + tvy * pvy + tvz * pvz);
  // the reject mask is an OR (raytracer.c:137-152): a triangle that fails on u fails whatever v and t are
  if (!((u < -RT_EPS) | (u > 1 + RT_EPS))) {
    float qvx, qvy, qvz, tq;
    if (REL) { qvx = C.y; qvy = C.z; qvz = C.w; tq = __ldg(&tq4->x); }
    else {
      qvx = tvy * e1z - tvz * e1y; qvy = tvz * e1x - tvx * e1z; qvz = tvx * e1y - tvy * e1x;
      tq = e2x * qvx + e2y * qvy + e2z * qvz;
    }
    float v = inv_det * (w.dx * qvx + w.dy * qvy + w.dz * qvz);
    float t = inv_det * tq;
    bool miss = (v < -RT_EPS) | (u + v > 1 + RT_EPS) | (t < RT_EPS);
    // t <= 0 and NaN count as +inf (min_f32x8 with eps 0); NaN also fails the ordered compare
    if (!miss && t > 0.0f && t < w.hit_t) { w.hit_t = t; w.hit_u = u; w.hit_v = v; w.hit_slot = slot; }
  }
}

// raytracer.c:84-188: the eight triangles of the leaf the lane holds.  Strict <, ascending j: the lowest
// lane wins a tie inside the leaf and an earlier leaf wins across leaves (raytracer.c:15-32 with eps 0, :159).
template <bool REL>
__device__ __forceinline__ void walk_leaf(RayWalk &w, const SceneDev &sc, unsigned &c_leaves, unsigned &c_accepts) {
  const float t_before = w.hit_t;
  c_leaves++;
  // The loop is rolled (unrolled it is 9 KB of code).  For incoherent rays it is software-pipelined by
  // hand: the records of triangle j+1 are in flight while triangle j is tested, so a leaf pays one
  // load latency, not eight (measured -3 % on the bounce kernels; coherent primary rays hit L1 and
  // lose 3 % to the extra instructions, so they keep the plain loop).  Two triangles per trip: the two
  // record sets swap roles, so the pipeline needs no register moves (twelve per triangle in a 1-trip loop).
  if (!REL) {
    const float4 *tp = sc.tri_pos + (size_t)w.leaf * 24;
    float4 A0 = __ldg(tp), B0 = __ldg(tp + 1), C0 = __ldg(tp + 2);
    #pragma unroll 1
    for (int j = 0; j < 8; j += 2) {
      const float4 *odd = tp + 3 * (j + 1);
      const float4 A1 = __ldg(odd), B1 = __ldg(odd + 1), C1 = __ldg(odd + 2);
      leaf_triangle<false>(w, A0, B0, C0, nullptr, w.leaf * 8 + j);
      const float4 *even = tp + 3 * (j < 6 ? j + 2 : 7);
      A0 = __ldg(even); B0 = __ldg(even + 1); C0 = __ldg(even + 2);
      leaf_triangle<false>(w, A1, B1, C1, nullptr, w.leaf * 8 + j + 1);
    }
  } else {
    const float4 *tp = sc.tri_rel + (size_t)w.leaf * 32;
    #pragma unroll 1
    for (int j = 0; j < 8; j++) {
      const float4 A = __ldg(tp + 4 * j), B = __ldg(tp + 4 * j + 1), C = __ldg(tp + 4 * j + 2);
      leaf_triangle<true>(w, A, B, C, tp + 4 * j + 3, w.leaf * 8 + j);
    }
  }
  if (w.hit_t < t_before) c_accepts++;
  w.flags &= ~WALK_LEAF;
}

// incoherent rays: one step for the majority — node steps and leaf tests are different code, so the warp runs whichever
// more lanes wait for and the others keep their state for a later turn (`walking`: the lanes with WALK_LIVE)
template <bool REL>
__device__ __forceinline__ void walk_turn_voted(RayWalk &w, const SceneDev &sc, float4 *levels, unsigned walking,
                                                unsigned &c_nodes, unsigned &c_leaves, unsigned &c_accepts) {
  const unsigned want_leaf = __ballot_sync(RT_FULL, w.flags & WALK_LEAF);
  if (2 * __popc(want_leaf) <= __popc(walking)) {        // node steps wanted by at least as many lanes
    if ((w.flags & (WALK_LIVE | WALK_LEAF)) == WALK_LIVE) walk_node_step<REL>(w, sc, levels, c_nodes);
  } else {
    if (w.flags & WALK_LEAF) walk_leaf<REL>(w, sc, c_leaves, c_accepts);
  }
}

// ------------------------------------------------------------------ scheduling
// The warp-level scheduling of every walk over an input of rays: the trace kernel (rt_stages.cuh) and the ray queries
// (rt_query.cu) share its constants, the reservation of ray ranges and the voted turn.  Persistent warps pull rays from
// the input (the GPU form of the reference's atomic 32x32 chunk queue, raytracer.c:619-627) and keep their lanes full:
// whenever RT_REFILL_MIN_* lanes have finished, those lanes hand on their results and take the next rays of the warp's
// reserved range, while the others keep their walk state.

// rays a warp reserves per atomic on a long queue: 5823 / 5500 / 5372 / 5411 / 5831 us for the primary trace of a 64-spp helmet
// chunk at 64 / 128 / 256 / 512 / 1024 (consecutive ids are neighbouring pixels: short shares scatter a warp over the image
// and lose L1 reuse, long ones unbalance the last wave)
#ifndef RT_BATCH_MAX
#define RT_BATCH_MAX 256u
#endif
#ifndef RT_MIN_BATCH
#define RT_MIN_BATCH 4u
#endif
// Lanes that must have finished before the warp stops to emit results and take new rays.  The stop
// itself costs ~300 instructions at partial width, waiting costs idle lanes: measured optimum is "all
// 32" for primary rays (most finish in the same turn anyway; 9.17 / 8.60 / 8.20 / 8.08 ms per 64-spp
// chunk at 8 / 16 / 24 / 32) and 20 for bounce rays (7.36 / 7.15 / 7.13 / 7.27 / 8.90 ms at 12 / 16 / 20 / 24 / 32).
#ifndef RT_REFILL_MIN_PRIMARY
#define RT_REFILL_MIN_PRIMARY 32
#endif
#ifndef RT_REFILL_MIN_BOUNCE
#define RT_REFILL_MIN_BOUNCE 20
#endif

__device__ __forceinline__ void add_counter(unsigned long long *counters, int k, unsigned v) {
  v += __shfl_xor_sync(RT_FULL, v, 16);
  v += __shfl_xor_sync(RT_FULL, v, 8);
  v += __shfl_xor_sync(RT_FULL, v, 4);
  v += __shfl_xor_sync(RT_FULL, v, 2);
  v += __shfl_xor_sync(RT_FULL, v, 1);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(&counters[k], (unsigned long long)v);
}

// warp-aggregated append: returns this lane's slot in the queue whose length is *count
__device__ __forceinline__ unsigned warp_append(unsigned *count, bool want, unsigned lane) {
  const unsigned mask = __ballot_sync(RT_FULL, want);
  unsigned base = 0;
  if (lane == 0 && mask) base = atomicAdd(count, (unsigned)__popc(mask));
  base = __shfl_sync(RT_FULL, base, 0);
  return base + (unsigned)__popc(mask & ((1u << lane) - 1u));
}

// The reservation of a warp's ray ranges: the caller keeps the range and the batch in its own variables, and the helpers
// take and return plain values (helpers writing through references change the trace kernels' instruction schedule).

// rays reserved per atomic: large queues amortise the round trip, small ones (late bounces)
// spread over all warps of the grid
__device__ __forceinline__ unsigned ray_batch_first(unsigned n_in, unsigned total_warps) {
  unsigned batch = (n_in / (total_warps * 4u)) & ~31u;
  if (batch > RT_BATCH_MAX) batch = RT_BATCH_MAX;
  if (batch < 32u) {
    // a short queue: one share per warp, so the kernel lasts as long as a few rays, not as 32 in lock step
    batch = (n_in + total_warps - 1u) / total_warps;
    if (batch < RT_MIN_BATCH) batch = RT_MIN_BATCH;
    if (batch > 32u) batch = 32u;
  }
  return batch;
}

// the first index of the warp's next `batch` rays: one atomic on the input's fetch counter per range
__device__ __forceinline__ unsigned ray_fetch(unsigned *fetch, unsigned batch, unsigned lane) {
  unsigned base = 0;
  if (lane == 0) base = atomicAdd(fetch, batch);
  return __shfl_sync(RT_FULL, base, 0);
}

// guided self-scheduling: shares shrink as the queue drains (`left` rays after the range just reserved), so the kernel's
// last wave is short (a 256-ray share held by one warp while the others idle is ~8 steps of 32 rays)
__device__ __forceinline__ unsigned ray_batch_next(unsigned batch, unsigned left, unsigned total_warps) {
  if (batch > 32u) {
    const unsigned share = (left / (total_warps * 2u)) & ~31u;
    batch = share < 32u ? 32u : (share < batch ? share : batch);
  }
  return batch;
}
