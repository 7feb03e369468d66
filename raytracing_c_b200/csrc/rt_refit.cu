// rt_refit.cu — refit of a resident scene from new vertex positions (rt_gpu_scene_refit*, orchestrated in rt_scene.cu).
//
// The topology stays what scene_init decided: which triangle sits in which slot and which child is which.  What
// depends on positions is recomputed with host/scene_build.c's f32 expressions (IEEE, no contraction: the library is
// built with -fmad=false, and every division and square root is the _rn intrinsic):
//   * per occupied slot: tri_soa (the nine vertex arrays), tri_pos (p0, e1, e2) and the geometric normal, tangent and
//     bitangent of tri_rec (pack_leaf, with its |det| < 0.0001f clamp); the vertex normals when given.  UVs and the
//     material index are kept;
//   * per node child: min / max over the subtree's triangles of minf(p0, minf(p1, p2)) - RT_EPS and maxf(...) + RT_EPS,
//     scene_init's inflated triangle boxes.  With finite inputs min and max are exact in any order and an exact zero
//     difference rounds to +0, so the bottom-up reduction equals range_box bit for bit.  A child whose subtree holds no
//     triangle keeps the all-zero box (lo == hi) scene_init writes.
// Occupancy is the upload's: `masks` holds, for node k < n_internal, bit j = child 8k+1+j has a triangle in its subtree,
// and for leaf l (index n_internal + l), bit j = slot 8l+j is a triangle.  Padding slots are never read or written.
// Every kernel returns at once when the validation flag is set, so a refused refit writes nothing.
#include <cuda_runtime.h>

#include "rt_kernels.h"

namespace {

__device__ __forceinline__ bool finite(float v) { return isfinite(v); }

__global__ void rt_refit_validate_kernel(const float *__restrict__ pos, int n_slots, const unsigned char *__restrict__ masks,
                                         int n_internal, int *flag) {
  const size_t N = (size_t)n_slots;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_slots; s += gridDim.x * blockDim.x) {
    if (!((masks[n_internal + (s >> 3)] >> (s & 7)) & 1)) continue;
    bool ok = true;
    #pragma unroll
    for (int k = 0; k < 9; k++) ok &= finite(pos[k * N + s]);
    if (!ok) atomicOr(flag, 1);
  }
}

// one thread per slot; the eight slots of a leaf are eight consecutive lanes, reduced with shuffles into the leaf's
// row of its parent node.  n_slots is a multiple of 64 and the stride a multiple of 32, so warps stay whole.
__global__ void rt_refit_slots_kernel(const float *__restrict__ pos, const float *__restrict__ normals, int normal_stride,
                                      int n_slots, const unsigned char *__restrict__ masks, int n_internal,
                                      const int *__restrict__ flag, float *__restrict__ nodes, float4 *__restrict__ tri_pos,
                                      float4 *__restrict__ tri_rec, float *__restrict__ tri_soa) {
  if (*flag) return;
  const size_t N = (size_t)n_slots;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_slots; s += gridDim.x * blockDim.x) {
    const int leaf = s >> 3, lane8 = s & 7;
    const bool occupied = (masks[n_internal + leaf] >> lane8) & 1;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (occupied) {
      float p[3][3];       // p[vertex][axis]
      #pragma unroll
      for (int a = 0; a < 3; a++)
        #pragma unroll
        for (int v = 0; v < 3; v++) {
          p[v][a] = pos[(3 * a + v) * N + s];
          tri_soa[(3 * a + v) * N + s] = p[v][a];
        }
      #pragma unroll
      for (int a = 0; a < 3; a++) {
        const float mn = sel_min(p[0][a], sel_min(p[1][a], p[2][a])), mx = sel_max(p[0][a], sel_max(p[1][a], p[2][a]));
        lo[a] = __fsub_rn(mn, RT_EPS);
        hi[a] = __fadd_rn(mx, RT_EPS);
      }
      float e1[3], e2[3];
      #pragma unroll
      for (int a = 0; a < 3; a++) { e1[a] = __fsub_rn(p[1][a], p[0][a]); e2[a] = __fsub_rn(p[2][a], p[0][a]); }
      tri_pos[3 * (size_t)s + 0] = make_float4(p[0][0], p[0][1], p[0][2], e1[0]);
      tri_pos[3 * (size_t)s + 1] = make_float4(e1[1], e1[2], e2[0], e2[1]);
      tri_pos[3 * (size_t)s + 2] = make_float4(e2[2], 0.0f, 0.0f, 0.0f);

      // pack_leaf (scene_build.c) on the slot's own UVs: rows 4.zw, 5.xy, 5.zw of the record
      float4 *rec = tri_rec + 7 * (size_t)s;
      float4 r0 = rec[0], r1 = rec[1], r2 = rec[2];
      const float4 r4 = rec[4], r5 = rec[5];
      const float du1 = __fsub_rn(r5.x, r4.z), dv1 = __fsub_rn(r5.y, r4.w);
      const float du2 = __fsub_rn(r5.z, r4.z), dv2 = __fsub_rn(r5.w, r4.w);
      float det = __fsub_rn(__fmul_rn(du1, dv2), __fmul_rn(du2, dv1));
      if (fabsf(det) < 0.0001f) det = det < 0 ? -0.0001f : 0.0001f;
      const float inv = __fdiv_rn(1.0f, det);
      float tg[3], bt[3], nm[3];
      #pragma unroll
      for (int a = 0; a < 3; a++) {
        tg[a] = __fmul_rn(__fsub_rn(__fmul_rn(e1[a], dv2), __fmul_rn(e2[a], dv1)), inv);
        bt[a] = __fmul_rn(__fsub_rn(__fmul_rn(e2[a], du1), __fmul_rn(e1[a], du2)), inv);
      }
      nm[0] = __fsub_rn(__fmul_rn(e1[1], e2[2]), __fmul_rn(e1[2], e2[1]));
      nm[1] = __fsub_rn(__fmul_rn(e1[2], e2[0]), __fmul_rn(e1[0], e2[2]));
      nm[2] = __fsub_rn(__fmul_rn(e1[0], e2[1]), __fmul_rn(e1[1], e2[0]));
      auto inv_len = [](const float *v) {
        return __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(v[0], v[0]), __fmul_rn(v[1], v[1])), __fmul_rn(v[2], v[2]))));
      };
      const float s_tg = inv_len(tg), s_bt = inv_len(bt), s_nm = inv_len(nm);
      r0.x = __fmul_rn(nm[0], s_nm); r0.y = __fmul_rn(nm[1], s_nm); r0.z = __fmul_rn(nm[2], s_nm);
      if (normals) {      // normal_a (r0.w, r1.xy), normal_b (r1.zw, r2.x), normal_c (r2.yzw)
        const float *n = normals + (size_t)normal_stride * (size_t)s;
        r0.w = n[0]; r1 = make_float4(n[1], n[2], n[3], n[4]); r2 = make_float4(n[5], n[6], n[7], n[8]);
        rec[1] = r1; rec[2] = r2;
      }
      rec[0] = r0;
      rec[3] = make_float4(__fmul_rn(tg[0], s_tg), __fmul_rn(tg[1], s_tg), __fmul_rn(tg[2], s_tg), __fmul_rn(bt[0], s_bt));
      rec[4] = make_float4(__fmul_rn(bt[1], s_bt), __fmul_rn(bt[2], s_bt), r4.z, r4.w);
    }
    #pragma unroll
    for (int off = 1; off < 8; off <<= 1)
      #pragma unroll
      for (int a = 0; a < 3; a++) {
        lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], off));
        hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], off));
      }
    if (lane8 == 0) {
      const int k = n_internal + leaf, parent = (k - 1) >> 3, j = (k - 1) & 7;
      const bool any = masks[k] != 0;
      float *node = nodes + 48 * (size_t)parent;
      #pragma unroll
      for (int a = 0; a < 3; a++) { node[a * 8 + j] = any ? lo[a] : 0.0f; node[(3 + a) * 8 + j] = any ? hi[a] : 0.0f; }
    }
  }
}

// nodes [first, first + count) of one internal level: the union of each node's present children goes into the node's
// row of its parent
__global__ void rt_refit_level_kernel(float *__restrict__ nodes, int first, int count, const unsigned char *__restrict__ masks,
                                      const int *__restrict__ flag) {
  if (*flag) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const int k = first + i, parent = (k - 1) >> 3, j = (k - 1) & 7;
    const unsigned m = masks[k];
    const float *node = nodes + 48 * (size_t)k;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int c = 0; c < 8; c++) {
      if (!((m >> c) & 1)) continue;
      #pragma unroll
      for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], node[a * 8 + c]); hi[a] = fmaxf(hi[a], node[(3 + a) * 8 + c]); }
    }
    float *row = nodes + 48 * (size_t)parent;
    #pragma unroll
    for (int a = 0; a < 3; a++) { row[a * 8 + j] = m ? lo[a] : 0.0f; row[(3 + a) * 8 + j] = m ? hi[a] : 0.0f; }
  }
}

unsigned grid_for(size_t n) {
  unsigned grid = (unsigned)((n + 255) / 256);
  if (grid > 148u * 8u) grid = 148u * 8u;
  return grid < 1 ? 1 : grid;
}

}  // namespace

int rt_launch_refit(const RefitParams &p, cudaStream_t stream) {
  if (p.depth < 1 || p.depth > RT_MAX_DEPTH || p.n_slots % 64) return (int)cudaErrorInvalidValue;
  rt_refit_validate_kernel<<<grid_for((size_t)p.n_slots), 256, 0, stream>>>(p.positions, p.n_slots, p.masks, p.n_internal, p.flag);
  rt_refit_slots_kernel<<<grid_for((size_t)p.n_slots), 256, 0, stream>>>(p.positions, p.normals, p.normal_stride, p.n_slots,
                                                                         p.masks, p.n_internal, p.flag, p.nodes, p.tri_pos,
                                                                         p.tri_rec, p.tri_soa);
  // levels depth-1 .. 1 (the root's own box is the host's root union): level L starts at sum_{k<L} 8^k
  for (int level = p.depth - 1; level >= 1; level--) {
    int first = 0, count = 1;
    for (int k = 0; k < level; k++) { first += count; count *= 8; }
    rt_refit_level_kernel<<<grid_for((size_t)count), 256, 0, stream>>>(p.nodes, first, count, p.masks, p.flag);
  }
  return (int)cudaGetLastError();
}
