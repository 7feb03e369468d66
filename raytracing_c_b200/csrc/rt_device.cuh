// rt_device.cuh — device-side data layout and small vector helpers.
//
// HBM layout (uploaded once per Scene, see rt_cabi.cu):
//   nodes     f32[n_nodes][6][8]   exactly the host BVH_Node bytes (192 B): row r of
//                                  node n is one 32-byte sector, lane j of an octet
//                                  is child j's bound; a thread reads a node as twelve
//                                  16-byte vectors (warp-uniform for coherent rays).
//   tri_pos   float4[n_slots][3]   the host's nine strided SoA arrays regrouped per
//                                  triangle slot (one thread tests a whole leaf, so a
//                                  triangle is three 16-byte loads): (p0.xyz, e1.x)
//                                  (e1.yz, e2.xy) (e2.z, 0, 0, 0) with the edges
//                                  e1 = p1-p0 and e2 = p2-p0; leaf l = slots 8l..8l+7.
//   tri_rec   float4[n_slots][7]   shading record (112 B): geometric normal, three
//                                  vertex normals, tangent, bitangent, three UVs,
//                                  material index (Triangle_AOS with the Shader
//                                  function pointer replaced by a table index).
//                                  Read through the rec_* accessors below.
//   materials, textures            PBR_Shader_Data with Image* -> texture slot;
//                                  texels repacked RGB8 -> RGBA8 (one 32-bit load per tap).
// Everything is read-only during a render and small enough (<= ~75 MB with the
// helmet's four 2048^2 textures) to live in the 126 MB L2.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "rt_math.h"
#include "rt_seed.h"

#define RT_EPS 0.0001f
#define RT_MAX_DEPTH 8

struct V3 { float x, y, z; };

struct TextureDev {
  const uchar4 *texels;
  int width, height;
  // the environment only: the same texels as three floats (texel / 255.999f, the sampler's own IEEE division, done
  // once at upload) — one 16-byte load per tap instead of a 4-byte load, three byte extractions and three table reads
  const float4 *texels_f32;
};

struct MaterialDev {
  float base[3], emission[3];
  float roughness, metalness, normal_strength, sheen, sheen_tint, aniso;
  int   tex_albedo, tex_normal, tex_mr, tex_emission;   // -1 = none
};

struct SceneDev {
  const float       *nodes;
  const float4      *tri_pos;
  const float4      *tri_rec;
  const float       *tri_soa;        // the host's nine vertex arrays x0 x1 x2 y0 y1 y2 z0 z1 z2, n_slots each (lightmap_bake)
  float             *nodes_rel;      // nodes minus the camera origin, refreshed per render (primary rays)
  float4            *tri_rel;        // float4[n_slots][4]: (o-p0, e1.x)(e1.yz, e2.xy)(e2.z, (o-p0) x e1)(e2 . that, -, -, -)
  const MaterialDev *materials;
  const TextureDev  *textures;
  int                env_texture;
  int                depth, n_internal, n_slots;
  float              root_lo[3], root_hi[3];   // union of the root's non-empty child boxes (rt_trace.cuh)
  float              srgb_of_zero;             // decode_srgb(0): the sRGB decode of a black texel (rt_shade.cuh)
  int                root_upper_empty;         // the root's children 4..7 are padding boxes (lo == hi): never entered
  float              view[3][4];      // rows 0..2 of the camera-to-world matrix
  float              focal_length;
};

#define RT_MAX_DEVICES 64    // CUDA device ordinals the library keeps per-device kernel attributes for
#define RT_MAX_PARTS 16      // accumulators one reduce+resolve launch can combine

struct ReduceParts { const float *part[RT_MAX_PARTS]; int n; };

// the fields of a Camera the renderer reads: rows 0..2 of the camera-to-world matrix and the focal length
struct ViewCamera { float view[3][4]; float focal_length; };

struct RenderParams {
  SceneDev  scene;
  int       width, height;
  int       fast;                        // bounce stages from rt_render_fast.cu (RT_GPU_Options.fast_math)
  int       split_rank, split_world;     // pixel-space split over 32x32 chunks (rt_render.cu), world <= 1 = whole image
  cudaEvent_t shading_ready;             // optional: textures/environment complete (the primary trace does not wait for it)
  int       sample_begin, sample_end, max_bounces;
  uint32_t  user_seed;
  int       accumulate;
  float    *accum;
  float    *per_sample;
  int      *hit_ids;
  unsigned long long *counters;
  unsigned long long *counters_ex;
  const unsigned char *pixel_mask;       // optional W*H: only pixels with a non-zero byte are rendered (masked passes)
  float    *accum_sq;                    // optional W*H*3: per-channel sum of squared radiance in sample order
  // many views of the scene in one call (rt_gpu_render_views_device): with cameras, view v renders from cameras[v] with
  // the seed user_seeds[v] (NULL: user_seed) into accum + v * view_stride.  NULL cameras = one view, the scene's camera.
  int       n_views;
  const ViewCamera *cameras;             // host array [n_views]
  const uint32_t   *user_seeds;          // optional host array [n_views]
  size_t    view_stride;                 // floats between the views' accumulators
};

__device__ __forceinline__ V3 mk3(float x, float y, float z) { V3 v; v.x = x; v.y = y; v.z = z; return v; }
__device__ __forceinline__ V3 add3(V3 a, V3 b)   { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 sub3(V3 a, V3 b)   { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 mul3(V3 a, V3 b)   { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ V3 scale3(V3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
// left-to-right sum, products rounded separately (built with -fmad=false)
__device__ __forceinline__ float dot3(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross3(V3 a, V3 b) {
  return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ V3 normalize3(V3 a) {
  float inv = 1.0f / __fsqrt_rn(dot3(a, a));
  return scale3(a, inv);
}
__device__ __forceinline__ float lerp1(float a, float b, float t) { return a * (1 - t) + b * t; }
__device__ __forceinline__ V3 lerp3(V3 a, V3 b, float t) { return mk3(lerp1(a.x, b.x, t), lerp1(a.y, b.y, t), lerp1(a.z, b.z, t)); }
__device__ __forceinline__ float sel_min(float a, float b) { return a < b ? a : b; }   // MINPS: b when unordered
__device__ __forceinline__ float sel_max(float a, float b) { return a > b ? a : b; }   // MAXPS: b when unordered
__device__ __forceinline__ float clamp1(float x, float lo, float hi) { return x < lo ? lo : (x > hi ? hi : x); }

// ---- the shading record of a hit (tri_rec above, rows r0..r6 as float4): raytracer.c:164-182 in the f32 expressions
// every reader uses.  Barycentric weights of hit (u, v): w1 = u, w2 = v, w0 = 1 - w1 - w2 (raytracer.c:164-166).
__device__ __forceinline__ V3 rec_normal_geo(float4 r0) { return mk3(r0.x, r0.y, r0.z); }
// the vertex normals (r0.w, r1.xy) (r1.zw, r2.x) (r2.yzw), interpolated (raytracer.c:167-172; not normalised)
__device__ __forceinline__ V3 rec_normal(float4 r0, float4 r1, float4 r2, float w0, float w1, float w2) {
  return mk3(r0.w * w0 + r1.z * w1 + r2.y * w2,
             r1.x * w0 + r1.w * w1 + r2.z * w2,
             r1.y * w0 + r2.x * w1 + r2.w * w2);
}
// the three UVs (r4.zw) (r5.xy) (r5.zw), interpolated (raytracer.c:175-176)
__device__ __forceinline__ float rec_tex_u(float4 r4, float4 r5, float w0, float w1, float w2) { return r4.z * w0 + r5.x * w1 + r5.z * w2; }
__device__ __forceinline__ float rec_tex_v(float4 r4, float4 r5, float w0, float w1, float w2) { return r4.w * w0 + r5.y * w1 + r5.w * w2; }
__device__ __forceinline__ V3 rec_tangent(float4 r3) { return mk3(r3.x, r3.y, r3.z); }
__device__ __forceinline__ V3 rec_bitangent(float4 r3, float4 r4) { return mk3(r3.w, r4.x, r4.y); }
__device__ __forceinline__ int rec_material(float4 r6) { return __float_as_int(r6.x); }
// the hit point o + d * t (raytracer.c:173)
__device__ __forceinline__ V3 hit_point(V3 o, V3 d, float t) { return add3(o, scale3(d, t)); }
// raytracer.c:516: the ray leaves through the back of the geometric or of the interpolated normal
__device__ __forceinline__ bool hit_back_face(V3 ng, V3 normal, V3 d) { return dot3(ng, d) > 0 || dot3(normal, d) > 0; }
