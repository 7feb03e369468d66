/* refit_oracle.c — CPU restatement of the refit (rt_gpu_scene_refit*, include/rt_gpu.h) for the tests.
 *
 * Written from scene_build.c's rules, not from the device code: every node child's box is the range over the
 * occupied slots below it (scene_init's range_box over its subtree, taken directly over the slot range, where the
 * device reduces level by level), and every occupied slot's record is pack_leaf's, recomputed from the new positions
 * and the slot's own UVs.  A slot is occupied when its Triangle_AOS has a shader (what the upload records).
 *
 *   refit_oracle(scene, positions, normals): positions f32[9][n_slots] (x0 x1 x2 y0 y1 y2 z0 z1 z2), normals optional
 *   f32[n_slots][9] (normal_a, normal_b, normal_c).  The Scene's buffers are rewritten in place; padding slots get zero
 *   positions (and zero normals when normals are given), as the host form of the refit leaves them.
 */
#include <math.h>
#include <string.h>

#include "scene.h"

static inline f32 minf(f32 a, f32 b) { return a < b ? a : b; }
static inline f32 maxf(f32 a, f32 b) { return a > b ? a : b; }

static int occupied(Scene const *scene, isize s) {
  Shader const *sh = &scene->triangles.aos[s].shader;
  return sh->proc || sh->data;
}

static void pack_slot(Scene *scene, isize s) {
  Triangles *t = &scene->triangles;
  Triangle_AOS *r = &t->aos[s];
  f32 p[3][3];
  for (int v = 0; v < 3; v++) { p[v][0] = t->x[v][s]; p[v][1] = t->y[v][s]; p[v][2] = t->z[v][s]; }
  f32 e1[3], e2[3];
  for (int a = 0; a < 3; a++) { e1[a] = p[1][a] - p[0][a]; e2[a] = p[2][a] - p[0][a]; }
  f32 du1 = r->tex_coords_b.x - r->tex_coords_a.x, dv1 = r->tex_coords_b.y - r->tex_coords_a.y;
  f32 du2 = r->tex_coords_c.x - r->tex_coords_a.x, dv2 = r->tex_coords_c.y - r->tex_coords_a.y;
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
  for (int a = 0; a < 3; a++) {
    r->tangent.data[a]   = tg[a] * s_tg;
    r->bitangent.data[a] = bt[a] * s_bt;
    r->normal.data[a]    = nm[a] * s_nm;
  }
}

/* range_box over the occupied slots [first, first + n): 0 when there is none */
static void slot_range_box(Scene const *scene, isize first, isize n, f32 lo[3], f32 hi[3]) {
  Triangles const *t = &scene->triangles;
  int any = 0;
  for (int a = 0; a < 3; a++) { lo[a] = 0; hi[a] = 0; }
  for (isize s = first; s < first + n; s++) {
    if (!occupied(scene, s)) continue;
    for (int a = 0; a < 3; a++) {
      f32 *const *c = a == 0 ? t->x : a == 1 ? t->y : t->z;
      f32 tlo = minf(c[0][s], minf(c[1][s], c[2][s])) - RT_EPSILON;
      f32 thi = maxf(c[0][s], maxf(c[1][s], c[2][s])) + RT_EPSILON;
      if (!any) { lo[a] = tlo; hi[a] = thi; }
      lo[a] = minf(lo[a], tlo);
      hi[a] = maxf(hi[a], thi);
    }
    any = 1;
  }
}

void refit_oracle(Scene *scene, f32 const *positions, f32 const *normals) {
  Triangles *t = &scene->triangles;
  isize n = t->len, depth = scene->bvh.depth;
  for (isize s = 0; s < n; s++) {
    int occ = occupied(scene, s);
    for (int v = 0; v < 3; v++) {
      t->x[v][s] = occ ? positions[(0 + v) * n + s] : 0.0f;
      t->y[v][s] = occ ? positions[(3 + v) * n + s] : 0.0f;
      t->z[v][s] = occ ? positions[(6 + v) * n + s] : 0.0f;
    }
    if (normals) {
      Vec3 *dst[3] = { &t->aos[s].normal_a, &t->aos[s].normal_b, &t->aos[s].normal_c };
      for (int v = 0; v < 3; v++)
        for (int a = 0; a < 3; a++) dst[v]->data[a] = occ ? normals[s * 9 + v * 3 + a] : 0.0f;
    }
    if (occ) pack_slot(scene, s);
  }
  /* node i of level L (first index sum_{k<L} 8^k): child j is node 8i+1+j of level L+1, whose subtree covers
   * 8^(depth-L-1) leaves of 8 slots each */
  isize first = 0, count = 1;
  for (isize level = 0; level < depth; level++) {
    isize leaves_per_child = bvh_n_leaf_nodes(depth - level - 1);
    for (isize r = 0; r < count; r++) {
      BVH_Node node;
      memset(&node, 0, sizeof node);
      for (int j = 0; j < RT_SIMD_WIDTH; j++) {
        isize child_row = r * RT_SIMD_WIDTH + j;        /* the child's index within level + 1 */
        f32 lo[3], hi[3];
        slot_range_box(scene, child_row * leaves_per_child * RT_SIMD_WIDTH, leaves_per_child * RT_SIMD_WIDTH, lo, hi);
        for (int a = 0; a < 3; a++) { node.mins[a][j] = lo[a]; node.maxs[a][j] = hi[a]; }
      }
      scene->bvh.nodes.data[first + r] = node;
    }
    first += count;
    count *= RT_SIMD_WIDTH;
  }
}
