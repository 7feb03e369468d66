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
