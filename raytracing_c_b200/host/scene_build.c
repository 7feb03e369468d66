/* scene_build.c — host-side scene_init: implicit complete 8-ary BVH over padded
 * triangle slots, plus SoA/AoS triangle packing.  This is the buffer the GPU
 * library uploads once (include/scene.h describes the layout).
 *
 * Behavioural contract = reference scene.c:78-242,311-426 (count-balanced
 * split at multiples of 8^depth, best-of-3-axes by summed surface area with
 * ties to the later axis, children numbered in completion order), with the two
 * fixes DESIGN.md lists (leaf early-out only at leaf level; depth >= 1).
 *
 * Implementation is NOT the reference's: the reference re-sorts whole slices of
 * 112-byte Triangle records in place 3-4 times per split with a comparison
 * sort.  Here triangles are never moved: a permutation of u32 ids is sorted,
 * per-triangle keys and boxes are computed once, and each of the reference's
 * successive stable sorts (axis 0, then 1, then 2, then the winner) is a stable
 * LSD radix sort of the ids on the 32-bit order-preserving image of the f32 key
 * (3 passes of 11 bits: O(n), ~0.1 ms for the helmet's 15 452 triangles where a
 * comparison sort under the composite key took ~1.5 ms) — stability carries the
 * earlier orders exactly as the reference's stable sort does.  Sibling subtrees
 * are built by a small pthread pool.  tests/test_scene_build.py checks the
 * result byte-for-byte against the oracle's literal restatement.
 */
#define _GNU_SOURCE
#include <assert.h>
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "scene.h"
#include "rt_host.h"

#ifndef RT_BUILD_THREADS
#define RT_BUILD_THREADS 12   /* reference scene.c:425 */
#endif

typedef struct {
  f32 key[3];          /* p0[a] + p1[a] + p2[a] */
  f32 lo[3], hi[3];    /* triangle box inflated by EPSILON */
} Tri_Info;

typedef struct {
  Scene          *scene;
  Triangle const *tris;
  Tri_Info       *info;
  i32            *slot_of;   /* optional: slot_of[source index] = slot (rt_scene_init_slots) */
} Builder;

typedef struct { u32 id; } Item;

/* f32 -> u32 whose unsigned order is the float order; -0 and +0 map to the same value (the reference's `<`
 * comparator calls them equal, which makes them a tie that the earlier order decides) */
static inline u32 orderable(f32 k) {
  k += 0.0f;
  u32 u;
  memcpy(&u, &k, 4);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

/* stable sort of `it` (n ids) by key[axis]; `tmp` has room for n items and 2 * n u32 */
static void radix_sort_axis(Tri_Info const *info, Item *it, isize n, int axis, Item *tmp, u32 *keys, u32 *keys_tmp) {
  if (n < 2) return;
  for (isize i = 0; i < n; i++) keys[i] = orderable(info[it[i].id].key[axis]);
  if (n <= 96) {
    /* the lower levels sort a few dozen ids thousands of times: a histogram pass would cost more than the sort */
    for (isize i = 1; i < n; i++) {
      Item v = it[i];
      u32 k = keys[i];
      isize j = i;
      for (; j > 0 && keys[j - 1] > k; j--) { it[j] = it[j - 1]; keys[j] = keys[j - 1]; }
      it[j] = v; keys[j] = k;
    }
    return;
  }
  Item *src = it, *dst = tmp;
  u32 *ksrc = keys, *kdst = keys_tmp;
  for (int pass = 0; pass < 3; pass++) {
    int shift = pass * 11;
    u32 mask = pass == 2 ? 0x3ffu : 0x7ffu;
    u32 count[2048];
    memset(count, 0, sizeof count);
    for (isize i = 0; i < n; i++) count[(ksrc[i] >> shift) & mask]++;
    if (count[(ksrc[0] >> shift) & mask] == (u32)n) continue;          /* every key has the same digit: nothing moves */
    u32 sum = 0;
    for (u32 d = 0; d <= mask; d++) { u32 c = count[d]; count[d] = sum; sum += c; }
    for (isize i = 0; i < n; i++) {
      u32 pos = count[(ksrc[i] >> shift) & mask]++;
      dst[pos] = src[i];
      kdst[pos] = ksrc[i];
    }
    Item *t = src; src = dst; dst = t;
    u32 *kt = ksrc; ksrc = kdst; kdst = kt;
  }
  if (src != it) memcpy(it, src, sizeof(Item) * (size_t)n);
}

static inline f32 minf(f32 a, f32 b) { return a < b ? a : b; }
static inline f32 maxf(f32 a, f32 b) { return a > b ? a : b; }

static void range_box(Tri_Info const *info, Item const *it, isize n, f32 lo[3], f32 hi[3]) {
  for (int a = 0; a < 3; a++) { lo[a] = 0; hi[a] = 0; }
  for (isize i = 0; i < n; i++) {
    Tri_Info const *t = &info[it[i].id];
    for (int a = 0; a < 3; a++) {
      if (i == 0) { lo[a] = t->lo[a]; hi[a] = t->hi[a]; }
      lo[a] = minf(lo[a], t->lo[a]);
      hi[a] = maxf(hi[a], t->hi[a]);
    }
  }
}

static f32 box_area(f32 const lo[3], f32 const hi[3]) {
  f32 x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
  return 2.0f * (x * y + y * z + z * x);
}

static isize split_point(isize n, isize per_child) {
  isize taken = 0, rest = n;
  while (taken < n / 2 && rest > per_child) { taken += per_child; rest -= per_child; }
  return taken;
}

static void pack_leaf(Builder *b, Item const *it, isize n, isize first_slot) {
  Triangles *dst = &b->scene->triangles;
  assert(first_slot >= 0 && first_slot + n <= dst->len);
  for (isize i = 0; i < n; i++) {
    Triangle const *t = &b->tris[it[i].id];
    isize s = first_slot + i;
    if (b->slot_of) b->slot_of[it[i].id] = (i32)s;
    Vec3 const *p = t->positions;
    for (int v = 0; v < 3; v++) { dst->x[v][s] = p[v].x; dst->y[v][s] = p[v].y; dst->z[v][s] = p[v].z; }

    f32 e1[3], e2[3];
    for (int a = 0; a < 3; a++) { e1[a] = p[1].data[a] - p[0].data[a]; e2[a] = p[2].data[a] - p[0].data[a]; }
    f32 du1 = t->tex_coords[1].x - t->tex_coords[0].x, dv1 = t->tex_coords[1].y - t->tex_coords[0].y;
    f32 du2 = t->tex_coords[2].x - t->tex_coords[0].x, dv2 = t->tex_coords[2].y - t->tex_coords[0].y;
    f32 det = du1 * dv2 - du2 * dv1;
    if (fabsf(det) < 0.0001f) det = det < 0 ? -0.0001f : 0.0001f;
    f32 inv = 1.0f / det;

    f32 tg[3], bt[3], nm[3];
    for (int a = 0; a < 3; a++) {
      tg[a] = (e1[a] * dv2 - e2[a] * dv1) * inv;
      bt[a] = (e2[a] * du1 - e1[a] * du2) * inv;
    }
    nm[0] = e1[1] * e2[2] - e1[2] * e2[1];
    nm[1] = e1[2] * e2[0] - e1[0] * e2[2];
    nm[2] = e1[0] * e2[1] - e1[1] * e2[0];
    f32 s_tg = 1.0f / sqrtf(tg[0] * tg[0] + tg[1] * tg[1] + tg[2] * tg[2]);
    f32 s_bt = 1.0f / sqrtf(bt[0] * bt[0] + bt[1] * bt[1] + bt[2] * bt[2]);
    f32 s_nm = 1.0f / sqrtf(nm[0] * nm[0] + nm[1] * nm[1] + nm[2] * nm[2]);

    Triangle_AOS *r = &dst->aos[s];
    memset(r, 0, sizeof *r);
    for (int a = 0; a < 3; a++) {
      r->tangent.data[a]   = tg[a] * s_tg;
      r->bitangent.data[a] = bt[a] * s_bt;
      r->normal.data[a]    = nm[a] * s_nm;
    }
    r->normal_a = t->normals[0]; r->normal_b = t->normals[1]; r->normal_c = t->normals[2];
    r->tex_coords_a = t->tex_coords[0]; r->tex_coords_b = t->tex_coords[1]; r->tex_coords_c = t->tex_coords[2];
    r->shader = t->shader;
  }
}

/* ---- subtree task pool: children of the top levels are independent ---- */
typedef struct { Item *it; isize n, depth, index; } Task;
typedef struct {
  Builder        *b;
  Task           *tasks;
  isize           n_tasks, next;
  pthread_mutex_t lock;
} Pool;

static void build_subtree(Builder *b, Item *it, isize n, isize depth, isize index, Pool *defer);

static void *pool_worker(void *arg) {
  Pool *p = arg;
  for (;;) {
    pthread_mutex_lock(&p->lock);
    isize k = p->next < p->n_tasks ? p->next++ : -1;
    pthread_mutex_unlock(&p->lock);
    if (k < 0) return NULL;
    Task t = p->tasks[k];
    build_subtree(p->b, t.it, t.n, t.depth, t.index, NULL);
  }
}

static void build_subtree(Builder *b, Item *it, isize n, isize depth, isize index, Pool *defer) {
  Scene *scene = b->scene;
  if (depth == 0) {
    pack_leaf(b, it, n, (index - scene->bvh.last_row_offset) * RT_SIMD_WIDTH);
    return;
  }
  isize per_child = bvh_n_leaf_nodes(depth);
  assert(per_child * RT_SIMD_WIDTH >= n);

  struct { Item *it; isize n; } todo[RT_SIMD_WIDTH], done[RT_SIMD_WIDTH];
  isize n_todo = 0, n_done = 0;
  Item *tmp = malloc(sizeof(Item) * (size_t)(n ? n : 1));
  u32 *keys = malloc(sizeof(u32) * 2 * (size_t)(n ? n : 1));
  todo[n_todo].it = it; todo[n_todo].n = n; n_todo++;

  while (n_todo) {
    n_todo--;
    Item *s = todo[n_todo].it;
    isize sn = todo[n_todo].n;
    isize split = split_point(sn, per_child);

    /* reference scene.c:346-360: stable sort by axis 0, 1, 2 in turn, the split's cost after each; then once more
     * by the winner unless it is the last one */
    f32 best_area = INFINITY;
    int best_axis = 0;
    for (int axis = 0; axis < 3; axis++) {
      radix_sort_axis(b->info, s, sn, axis, tmp, keys, keys + n);
      f32 llo[3], lhi[3], rlo[3], rhi[3];
      range_box(b->info, s, split, llo, lhi);
      range_box(b->info, s + split, sn - split, rlo, rhi);
      f32 area = box_area(llo, lhi) + box_area(rlo, rhi);
      if (area <= best_area) { best_area = area; best_axis = axis; }
    }
    if (best_axis != 2) radix_sort_axis(b->info, s, sn, best_axis, tmp, keys, keys + n);

    isize ln = split, rn = sn - split;
    if (ln > per_child)   { todo[n_todo].it = s; todo[n_todo].n = ln; n_todo++; }
    else if (ln)          { done[n_done].it = s; done[n_done].n = ln; n_done++; }
    if (rn > per_child)   { todo[n_todo].it = s + split; todo[n_todo].n = rn; n_todo++; }
    else if (rn)          { done[n_done].it = s + split; done[n_done].n = rn; n_done++; }
    assert(n_todo <= RT_SIMD_WIDTH && n_done <= RT_SIMD_WIDTH);
  }
  free(tmp);
  free(keys);
  BVH_Node node;
  memset(&node, 0, sizeof node);
  for (isize i = 0; i < n_done; i++) {
    f32 lo[3], hi[3];
    range_box(b->info, done[i].it, done[i].n, lo, hi);
    for (int a = 0; a < 3; a++) { node.mins[a][i] = lo[a]; node.maxs[a][i] = hi[a]; }
    isize child = index * RT_SIMD_WIDTH + 1 + i;
    if (defer) {
      Task t = { done[i].it, done[i].n, depth - 1, child };
      defer->tasks[defer->n_tasks++] = t;
    } else {
      build_subtree(b, done[i].it, done[i].n, depth - 1, child, NULL);
    }
  }
  scene->bvh.nodes.data[index] = node;
}

static isize depth_for(isize n_triangles) {
  isize groups = (n_triangles + RT_SIMD_WIDTH - 1) / RT_SIMD_WIDTH, cap = 1, d = 0;
  while (cap < groups) { cap *= RT_SIMD_WIDTH; d++; }
  return d < 1 ? 1 : d;
}

void rt_scene_init_slots(Scene *scene, Triangle_Slice src, i32 *slot_of) {
  isize depth = depth_for(src.len);
  isize n_internal = bvh_n_internal_nodes(depth);
  scene->bvh.depth = depth;
  scene->bvh.last_row_offset = n_internal;
  scene->bvh.nodes.len = n_internal;
  scene->bvh.nodes.data = rt_host_buffer_alloc((size_t)n_internal * sizeof(BVH_Node));
  memset(scene->bvh.nodes.data, 0, (size_t)n_internal * sizeof(BVH_Node));

  isize slots = bvh_n_leaf_nodes(depth) * RT_SIMD_WIDTH;
  size_t bytes = (TRIANGLES_ALLOCATION_SIZE(slots) + 63) & ~(size_t)63;
  f32 *block = rt_host_buffer_alloc(bytes);
  memset(block, 0, bytes);
  scene->triangles.len = (i32)slots;
  for (int v = 0; v < 3; v++) {
    scene->triangles.x[v] = block + slots * (0 + v);
    scene->triangles.y[v] = block + slots * (3 + v);
    scene->triangles.z[v] = block + slots * (6 + v);
  }
  scene->triangles.aos = (Triangle_AOS *)(block + slots * 9);

  isize n = src.len;
  Builder b = { scene, src.data, malloc(sizeof(Tri_Info) * (size_t)(n ? n : 1)), slot_of };
  Item *items = malloc(sizeof(Item) * (size_t)(n ? n : 1));
  for (isize i = 0; i < n; i++) {
    Vec3 const *p = src.data[i].positions;
    for (int a = 0; a < 3; a++) {
      b.info[i].key[a] = p[0].data[a] + p[1].data[a] + p[2].data[a];
      b.info[i].lo[a]  = minf(p[0].data[a], minf(p[1].data[a], p[2].data[a])) - RT_EPSILON;
      b.info[i].hi[a]  = maxf(p[0].data[a], maxf(p[1].data[a], p[2].data[a])) + RT_EPSILON;
    }
    items[i].id = (u32)i;
  }

  /* Root on this thread, its (up to 8) child subtrees on the pool. */
  Task tasks[RT_SIMD_WIDTH];
  Pool pool;
  pool.b = &b; pool.tasks = tasks; pool.n_tasks = 0; pool.next = 0;
  pthread_mutex_init(&pool.lock, NULL);
  build_subtree(&b, items, n, depth, 0, &pool);
  int n_threads = RT_BUILD_THREADS < pool.n_tasks ? RT_BUILD_THREADS : (int)pool.n_tasks;
  pthread_t th[RT_BUILD_THREADS];
  for (int i = 1; i < n_threads; i++) pthread_create(&th[i], NULL, pool_worker, &pool);
  pool_worker(&pool);
  for (int i = 1; i < n_threads; i++) pthread_join(th[i], NULL);
  pthread_mutex_destroy(&pool.lock);

  free(items);
  free(b.info);
}

void scene_init(Scene *scene, Triangle_Slice src) { rt_scene_init_slots(scene, src, NULL); }

void scene_destroy(Scene *scene) {
  rt_host_buffer_free(scene->bvh.nodes.data);
  rt_host_buffer_free(scene->triangles.x[0]);
  memset(&scene->bvh, 0, sizeof scene->bvh);
  memset(&scene->triangles, 0, sizeof scene->triangles);
}
