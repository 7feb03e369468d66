/* query_oracle.c — TEST INFRASTRUCTURE.  The CPU reference of the ray queries (include/rt_gpu.h): for each ray, the
 * reference's ray_scene_hit (raytracer.c:443-503) with hit.distance = t_max before the walk; in `any` mode the walk
 * stops after the first leaf that accepts a triangle.
 *
 * The 8-wide slab and Möller–Trumbore kernels and the ordered walk are the oracle's (oracle/oracle_trace.c, which
 * restates raytracer.c:15-32,84-230,443-483), restated here with the initial distance and the early exit, which the
 * renderer's walk does not need.  tests/test_oracle_queries.py pins this file to oracle_trace_ray at t_max = +inf, to a
 * brute-force scan over every triangle and, where a reference checkout is available, to the reference's own
 * ray_scene_hit started at t_max.
 *
 * Build: gcc -O2 -mavx2 -mfma -ffp-contract=off -shared -fPIC -I include -I oracle (no contraction: every product and
 * sum rounds separately, as on the GPU with -fmad=false).
 */
#include <immintrin.h>
#include <math.h>
#include <pthread.h>
#include <stdbool.h>
#include <stdlib.h>
#include <string.h>

#include "raytracer.h"
#include "oracle_vec.h"

typedef struct { f32 t, u, v; i32 slot; } Query_Hit;

typedef struct {
  f32  distance, u, v;
  i32  slot;
  Vec3 point, normal, normal_geo;
  Vec2 tex_coords;
} Hit;

typedef struct { u64 rays, nodes, leaves, accepts; } Counters;

/* raytracer.c:15-32: horizontal min with lowest-lane argmin; lanes <= eps or NaN count as +inf */
static inline f32 lane_min(__m256 v, f32 eps, i32 *lane) {
  __m256 inf   = _mm256_set1_ps(INFINITY);
  __m256 keep  = _mm256_cmp_ps(v, _mm256_set1_ps(eps), _CMP_GT_OQ);
  __m256 clean = _mm256_blendv_ps(inf, v, keep);
  __m256 m = _mm256_min_ps(clean, _mm256_permute_ps(clean, 0xB1));
  m = _mm256_min_ps(m, _mm256_permute_ps(m, 0x4E));
  m = _mm256_min_ps(m, _mm256_permute2f128_ps(m, m, 0x01));
  int eq = _mm256_movemask_ps(_mm256_cmp_ps(clean, m, _CMP_EQ_OQ));
  *lane = __builtin_ctz((unsigned)eq);
  return _mm256_cvtss_f32(m);
}

#define SUB(a, b) _mm256_sub_ps(a, b)
#define MUL(a, b) _mm256_mul_ps(a, b)
#define ADD(a, b) _mm256_add_ps(a, b)

typedef struct { __m256 x, y, z; } V8;

static inline V8 v8_cross(V8 a, V8 b) {
  V8 r;
  r.x = SUB(MUL(a.y, b.z), MUL(a.z, b.y));
  r.y = SUB(MUL(a.z, b.x), MUL(a.x, b.z));
  r.z = SUB(MUL(a.x, b.y), MUL(a.y, b.x));
  return r;
}
static inline __m256 v8_dot(V8 a, V8 b) { return ADD(ADD(MUL(a.x, b.x), MUL(a.y, b.y)), MUL(a.z, b.z)); }

/* raytracer.c:84-188: the eight triangles of one leaf; takes the nearest when it is below hit->distance */
static bool leaf_test(Ray const *ray, Triangles const *tris, isize offset, Hit *hit) {
  V8 d  = { _mm256_set1_ps(ray->direction.x), _mm256_set1_ps(ray->direction.y), _mm256_set1_ps(ray->direction.z) };
  V8 o  = { _mm256_set1_ps(ray->position.x),  _mm256_set1_ps(ray->position.y),  _mm256_set1_ps(ray->position.z) };
  V8 p0 = { _mm256_load_ps(tris->x[0] + offset), _mm256_load_ps(tris->y[0] + offset), _mm256_load_ps(tris->z[0] + offset) };
  V8 p1 = { _mm256_load_ps(tris->x[1] + offset), _mm256_load_ps(tris->y[1] + offset), _mm256_load_ps(tris->z[1] + offset) };
  V8 p2 = { _mm256_load_ps(tris->x[2] + offset), _mm256_load_ps(tris->y[2] + offset), _mm256_load_ps(tris->z[2] + offset) };
  V8 e1 = { SUB(p1.x, p0.x), SUB(p1.y, p0.y), SUB(p1.z, p0.z) };
  V8 e2 = { SUB(p2.x, p0.x), SUB(p2.y, p0.y), SUB(p2.z, p0.z) };

  V8     pvec    = v8_cross(d, e2);
  __m256 det     = v8_dot(e1, pvec);
  __m256 inv_det = _mm256_div_ps(_mm256_set1_ps(1.0f), det);
  V8     tvec    = { SUB(o.x, p0.x), SUB(o.y, p0.y), SUB(o.z, p0.z) };
  V8     qvec    = v8_cross(tvec, e1);
  __m256 u = MUL(inv_det, v8_dot(tvec, pvec));
  __m256 v = MUL(inv_det, v8_dot(d, qvec));
  __m256 t = MUL(inv_det, v8_dot(e2, qvec));

  __m256 lo  = _mm256_set1_ps(-RT_EPSILON);
  __m256 hi  = _mm256_set1_ps(1 + RT_EPSILON);
  __m256 out = _mm256_or_ps(_mm256_cmp_ps(u, lo, _CMP_LT_OQ), _mm256_cmp_ps(u, hi, _CMP_GT_OQ));
  out = _mm256_or_ps(out, _mm256_or_ps(_mm256_cmp_ps(v, lo, _CMP_LT_OQ), _mm256_cmp_ps(ADD(u, v), hi, _CMP_GT_OQ)));
  out = _mm256_or_ps(out, _mm256_cmp_ps(t, _mm256_set1_ps(RT_EPSILON), _CMP_LT_OQ));
  __m256 dist = _mm256_blendv_ps(t, _mm256_set1_ps(INFINITY), out);

  i32 lane;
  f32 nearest = lane_min(dist, 0, &lane);
  if (!(nearest < hit->distance)) return false;

  f32 us[8] __attribute__((aligned(32))), vs[8] __attribute__((aligned(32)));
  _mm256_store_ps(us, u);
  _mm256_store_ps(vs, v);
  isize s  = lane + offset;
  f32   w1 = us[lane], w2 = vs[lane];
  f32   w0 = 1 - w1 - w2;
  Triangle_AOS const *rec = &tris->aos[s];
  /* raytracer.c:164-182 */
  hit->distance = nearest;
  hit->u = w1;
  hit->v = w2;
  hit->slot = (i32)s;
  hit->point  = v3_add(ray->position, v3_scale(ray->direction, nearest));
  hit->normal = v3(rec->normal_a.x * w0 + rec->normal_b.x * w1 + rec->normal_c.x * w2,
                   rec->normal_a.y * w0 + rec->normal_b.y * w1 + rec->normal_c.y * w2,
                   rec->normal_a.z * w0 + rec->normal_b.z * w1 + rec->normal_c.z * w2);
  hit->tex_coords.x = rec->tex_coords_a.x * w0 + rec->tex_coords_b.x * w1 + rec->tex_coords_c.x * w2;
  hit->tex_coords.y = rec->tex_coords_a.y * w0 + rec->tex_coords_b.y * w1 + rec->tex_coords_c.y * w2;
  hit->normal_geo = rec->normal;
  return true;
}

/* raytracer.c:190-230; _mm256_min_ps / max_ps return the SECOND operand when either is NaN */
static void child_box_test(Ray const *ray, f32 t_min, f32 t_max, BVH_Node const *node, f32 *out8) {
  __m256 ix = _mm256_set1_ps(1.0f / ray->direction.x);
  __m256 iy = _mm256_set1_ps(1.0f / ray->direction.y);
  __m256 iz = _mm256_set1_ps(1.0f / ray->direction.z);
  __m256 ox = _mm256_set1_ps(ray->position.x);
  __m256 oy = _mm256_set1_ps(ray->position.y);
  __m256 oz = _mm256_set1_ps(ray->position.z);
  __m256 ax = MUL(SUB(_mm256_load_ps(node->mins[0]), ox), ix);
  __m256 ay = MUL(SUB(_mm256_load_ps(node->mins[1]), oy), iy);
  __m256 az = MUL(SUB(_mm256_load_ps(node->mins[2]), oz), iz);
  __m256 bx = MUL(SUB(_mm256_load_ps(node->maxs[0]), ox), ix);
  __m256 by = MUL(SUB(_mm256_load_ps(node->maxs[1]), oy), iy);
  __m256 bz = MUL(SUB(_mm256_load_ps(node->maxs[2]), oz), iz);
  __m256 nx = _mm256_min_ps(ax, bx), ny = _mm256_min_ps(ay, by), nz = _mm256_min_ps(az, bz);
  __m256 fx = _mm256_max_ps(ax, bx), fy = _mm256_max_ps(ay, by), fz = _mm256_max_ps(az, bz);
  __m256 enter = _mm256_max_ps(_mm256_set1_ps(t_min), _mm256_max_ps(nx, _mm256_max_ps(ny, nz)));
  __m256 leave = _mm256_min_ps(_mm256_set1_ps(t_max), _mm256_min_ps(fx, _mm256_min_ps(fy, fz)));
  __m256 miss = _mm256_cmp_ps(enter, leave, _CMP_GE_OQ);
  _mm256_store_ps(out8, _mm256_blendv_ps(enter, _mm256_set1_ps(INFINITY), miss));
}

/* raytracer.c:443-483; any: stop the whole walk after the first leaf that accepts a triangle (returns true) */
static bool visit_node(Ray const *ray, Scene const *scene, isize index, Hit *hit, isize depth, bool any, Counters *c) {
  f32 entry[8] __attribute__((aligned(32)));
  child_box_test(ray, RT_EPSILON, hit->distance, &scene->bvh.nodes.data[index], entry);
  c->nodes++;
  for (int round = 0; round < RT_SIMD_WIDTH; round++) {
    f32 best = hit->distance;
    int pick = -1;
    for (int j = 0; j < RT_SIMD_WIDTH; j++) {
      if (entry[j] < best) { best = entry[j]; pick = j; }
    }
    if (pick < 0 || best >= hit->distance) return false;
    isize child = RT_SIMD_WIDTH * index + 1 + pick;
    if (depth == 1) {
      c->leaves++;
      bool took = leaf_test(ray, &scene->triangles, (child - scene->bvh.last_row_offset) * RT_SIMD_WIDTH, hit);
      if (took) c->accepts++;
      if (took && any) return true;
    } else if (visit_node(ray, scene, child, hit, depth - 1, any, c)) {
      return true;
    }
    entry[pick] = INFINITY;
  }
  return false;
}

typedef struct {
  Scene const *scene;
  Ray const   *rays;
  f32 const   *t_max;
  isize        begin, end;
  bool         any;
  Query_Hit   *hits;
  f32         *surface;
  u8          *occluded;
  Counters     counters;
  pthread_t    thread;
} Worker;

static void *worker(void *arg) {
  Worker *w = arg;
  for (isize i = w->begin; i < w->end; i++) {
    Hit hit;
    memset(&hit, 0, sizeof hit);
    hit.distance = w->t_max ? w->t_max[i] : INFINITY;      /* the query: the reference's walk started at t_max */
    hit.slot = -1;
    w->counters.rays++;
    visit_node(&w->rays[i], w->scene, 0, &hit, w->scene->bvh.depth, w->any, &w->counters);
    bool found = hit.slot >= 0;
    if (w->hits) {
      Query_Hit h = { INFINITY, 0, 0, -1 };
      if (found) { h.t = hit.distance; h.u = hit.u; h.v = hit.v; h.slot = hit.slot; }
      w->hits[i] = h;
    }
    if (w->surface) {
      f32 *o = w->surface + 11 * i;
      memset(o, 0, 11 * sizeof(f32));
      if (found) {
        o[0] = hit.point.x;      o[1] = hit.point.y;      o[2] = hit.point.z;
        o[3] = hit.normal.x;     o[4] = hit.normal.y;     o[5] = hit.normal.z;
        o[6] = hit.normal_geo.x; o[7] = hit.normal_geo.y; o[8] = hit.normal_geo.z;
        o[9] = hit.tex_coords.x; o[10] = hit.tex_coords.y;
      }
    }
    if (w->occluded) w->occluded[i] = found ? 1 : 0;
  }
  return NULL;
}

/* n rays split over n_threads; every output optional; counters = rays, nodes, leaves, accepts */
void query_oracle_rays(Scene const *scene, Ray const *rays, f32 const *t_max, isize n, i32 any, Query_Hit *hits,
                       f32 *surface, u8 *occluded, u64 counters[4], i32 n_threads) {
  if (n_threads < 1) n_threads = 1;
  Worker *ws = calloc((size_t)n_threads, sizeof *ws);
  for (i32 k = 0; k < n_threads; k++) {
    Worker *w = &ws[k];
    w->scene = scene; w->rays = rays; w->t_max = t_max; w->any = any != 0;
    w->hits = hits; w->surface = surface; w->occluded = occluded;
    w->begin = n * k / n_threads;
    w->end = n * (k + 1) / n_threads;
  }
  for (i32 k = 1; k < n_threads; k++) pthread_create(&ws[k].thread, NULL, worker, &ws[k]);
  worker(&ws[0]);
  for (i32 k = 1; k < n_threads; k++) pthread_join(ws[k].thread, NULL);
  if (counters) {
    memset(counters, 0, 4 * sizeof(u64));
    for (i32 k = 0; k < n_threads; k++) {
      counters[0] += ws[k].counters.rays;    counters[1] += ws[k].counters.nodes;
      counters[2] += ws[k].counters.leaves;  counters[3] += ws[k].counters.accepts;
    }
  }
  free(ws);
}
