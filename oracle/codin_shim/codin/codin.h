/* codin.h — TEST INFRASTRUCTURE.  A stand-in for the reference author's "Codin"
 * standard library, which every reference file includes (common.h:3-4,
 * raytracer.c:3-7, scene.c:1-6, driver.c:1-8) but which is not vendored.
 *
 * Purpose: let the UNMODIFIED reference sources compile, from where they lie
 * in a reference checkout (RT_REFERENCE_DIR), into oracle/_ref/libref.so (recipe: oracle/Makefile,
 * target `ref`), so the oracle's restatement can be checked against the
 * reference's own code.  Only what those sources use is provided; every other
 * codin/X.h in this directory just includes this file.
 *
 * Everything here is inferred from usage (SURVEY.md Appendix A).  Choices that
 * affect arithmetic are the UNPINNED ones DESIGN.md lists — the same choices
 * the oracle makes: vec3_dot sums left to right, vec3_normalize scales by
 * 1/sqrt(len2), lerp is a*(1-t)+b*t, reflect is I-2(I.N)N, from_basis puts its
 * arguments in columns, sort_slice_by is stable, allocations are zeroed, PI is
 * a double, and the transcendental functions are rt_math.h's.
 */
#ifndef CODIN_SHIM_H
#define CODIN_SHIM_H

#include <assert.h>
#include <math.h>
#include <pthread.h>
#include <sched.h>
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "rt_math.h"

/* ------------------------------------------------------------------ basics */
typedef float     f32;
typedef double    f64;
typedef int8_t    i8;
typedef int16_t   i16;
typedef int32_t   i32;
typedef int64_t   i64;
typedef uint8_t   u8;
typedef uint16_t  u16;
typedef uint32_t  u32;
typedef uint64_t  u64;
typedef ptrdiff_t isize;
typedef size_t    usize;
typedef uintptr_t uintptr;
typedef void     *rawptr;
typedef u8        byte;

#define internal     static
#define thread_local _Thread_local
#define nil          NULL
#define loop         for (;;)
#define for_range(i, a, b) for (isize i = (a); i < (b); i++)
#define size_of(x)   ((isize)sizeof(x))
#define count_of(a)  ((isize)(sizeof(a) / sizeof((a)[0])))
#define type_of(x)   __typeof__(x)
#define CASE         break; case
#define DEFAULT      break; default

#define F32_INFINITY ((f32)INFINITY)
#define U32_MAX      0xffffffffu
#define PI           3.14159265358979323846

#undef min
#undef max
#define min(a, b)         ((a) < (b) ? (a) : (b))
#define max(a, b)         ((a) > (b) ? (a) : (b))
#define clamp(x, lo, hi)  ((x) < (lo) ? (lo) : ((x) > (hi) ? (hi) : (x)))

/* ------------------------------------------------------------------ slices */
#define Slice(T) struct { T *data; isize len; }
typedef Slice(byte) Byte_Slice;
typedef Slice(char) String;
typedef Slice(String) String_Slice;

#define IDX(arr, i) (arr).data[(i)]
#define LIT(s) ((String){ .data = (char *)(s), .len = (isize)sizeof(s) - 1 })

#define slice_array(T, arr)   ((T){ .data = (arr), .len = count_of(arr) })
#define slice_end(s, n)       ((__typeof__(s)){ .data = (s).data, .len = (isize)(n) })
#define slice_start(s, n)     ((__typeof__(s)){ .data = (s).data + (isize)(n), .len = (s).len - (isize)(n) })
#define slice_to_bytes(s)     ((Byte_Slice){ .data = (byte *)(s).data, .len = (s).len * size_of((s).data[0]) })
#define slice_iter_v(slice, v, i, ...)                                           \
  do {                                                                          \
    __auto_type _it_s = (slice);                                                \
    for (isize i = 0; i < _it_s.len; i++) {                                     \
      __typeof__(*_it_s.data) v = _it_s.data[i];                                \
      (void)v;                                                                  \
      __VA_ARGS__                                                               \
    }                                                                           \
  } while (0)

/* --------------------------------------------------------------- allocators */
typedef struct { int kind; } Allocator;
typedef struct { int unused; } Logger;
typedef struct { Allocator allocator, temp_allocator; Logger logger; } Codin_Context;
extern thread_local Codin_Context context;

typedef struct { rawptr value; int err; } Alloc_Result;
internal inline Alloc_Result mem_alloc_aligned(isize size, isize align, Allocator a) {
  (void)a;
  usize al = (usize)(align < 16 ? 16 : align);
  usize n = ((usize)(size > 0 ? size : 1) + al - 1) / al * al;
  Alloc_Result r = { aligned_alloc(al, n), 0 };
  if (!r.value) r.err = 1; else memset(r.value, 0, n);        /* UNPINNED: zero-filled */
  return r;
}
internal inline void mem_free(rawptr p, isize size, Allocator a) { (void)size; (void)a; free(p); }
#define mem_copy(dst, src, n) memcpy((dst), (src), (usize)(n))

#define unwrap_err(e) ({ __auto_type _ur = (e); assert(!_ur.err); _ur.value; })
#define or_do_err(e, errname, ...) ({ __auto_type _or = (e); if (_or.err) { __auto_type errname = _or.err; (void)errname; __VA_ARGS__ } _or.value; })

#define slice_init(sp, n, alloc)                                                             \
  do {                                                                                       \
    (sp)->len  = (isize)(n);                                                                 \
    (sp)->data = unwrap_err(mem_alloc_aligned((isize)(n) * size_of((sp)->data[0]), 64, alloc)); \
  } while (0)
#define slice_make_aligned(T, n, align, alloc) ({ T _sm; _sm.len = (isize)(n); _sm.data = unwrap_err(mem_alloc_aligned((isize)(n) * size_of(_sm.data[0]), (align), alloc)); _sm; })

#define Vector(T) struct { T *data; isize len, cap; Allocator allocator; }
#define vector_init(vp, n, capacity, alloc)                                                  \
  do {                                                                                       \
    (vp)->len = (n); (vp)->cap = (capacity) > (n) ? (capacity) : (n);                        \
    if ((vp)->cap < 8) (vp)->cap = 8;                                                        \
    (vp)->allocator = (alloc);                                                               \
    (vp)->data = calloc((usize)(vp)->cap, sizeof((vp)->data[0]));                            \
  } while (0)
#define vector_append(vp, value)                                                             \
  {                                                                                          \
    if ((vp)->len == (vp)->cap) {                                                            \
      (vp)->cap *= 2;                                                                        \
      (vp)->data = realloc((vp)->data, (usize)(vp)->cap * sizeof((vp)->data[0]));            \
    }                                                                                        \
    (vp)->data[(vp)->len++] = (value);                                                       \
  }

#define Hash_Map(K, V) struct { K *keys; V *values; isize len, cap; bool (*equal)(K, K); }
#define hash_map_init(mp, capacity, eq, hash, alloc)                                         \
  do {                                                                                       \
    (mp)->len = 0; (mp)->cap = (capacity); (mp)->equal = (eq);                               \
    (mp)->keys = calloc((usize)(mp)->cap, sizeof((mp)->keys[0]));                            \
    (mp)->values = calloc((usize)(mp)->cap, sizeof((mp)->values[0]));                        \
  } while (0)
#define hash_map_get(m, key) ({ __typeof__((m).values) _hg = nil; for (isize _hi = 0; _hi < (m).len; _hi++) if ((m).equal((m).keys[_hi], (key))) { _hg = &(m).values[_hi]; break; } _hg; })
#define hash_map_insert(mp, key, value)                                                      \
  do {                                                                                       \
    if ((mp)->len == (mp)->cap) {                                                            \
      (mp)->cap *= 2;                                                                        \
      (mp)->keys = realloc((mp)->keys, (usize)(mp)->cap * sizeof((mp)->keys[0]));            \
      (mp)->values = realloc((mp)->values, (usize)(mp)->cap * sizeof((mp)->values[0]));      \
    }                                                                                        \
    (mp)->keys[(mp)->len] = (key); (mp)->values[(mp)->len] = (value); (mp)->len++;           \
  } while (0)

typedef struct { int unused; } Growing_Arena_Allocator;
internal inline Allocator growing_arena_allocator_init(Growing_Arena_Allocator *a, isize size, Allocator backing) { (void)a; (void)size; return backing; }

/* ----------------------------------------------------------------- strings */
internal inline bool string_equal(String a, String b) { return a.len == b.len && (a.len == 0 || !memcmp(a.data, b.data, (usize)a.len)); }
internal inline u64  string_hash(String s) { u64 h = 1469598103934665603ull; for (isize i = 0; i < s.len; i++) h = (h ^ (u8)s.data[i]) * 1099511628211ull; return h; }
internal inline bool string_has_suffix(String s, String suffix) { return s.len >= suffix.len && !memcmp(s.data + s.len - suffix.len, suffix.data, (usize)suffix.len); }
internal inline String bytes_to_string(Byte_Slice b) { String s = { (char *)b.data, b.len }; return s; }
internal inline isize parse_int(String *s) { isize v = 0, i = 0, sign = 1; if (s->len && s->data[0] == '-') { sign = -1; i = 1; } for (; i < s->len && s->data[i] >= '0' && s->data[i] <= '9'; i++) v = v * 10 + (s->data[i] - '0'); return v * sign; }
extern String_Slice os_args;

/* the reference only prints through these; the shim drops the output */
internal inline void codin_fmt_sink(char const *fmt, ...) { (void)fmt; }
#define fmt_printflnc   codin_fmt_sink
#define fmt_printfc     codin_fmt_sink
#define fmt_printlnc    codin_fmt_sink
#define fmt_eprintflnc  codin_fmt_sink
#define fmt_eprintlnc   codin_fmt_sink

#define X_ENUM_ITEM(x) x,
#define X_ENUM(Name, LIST) typedef enum { LIST(X_ENUM_ITEM) Name##__count } Name;
#define enum_iter(Name, v) for (Name v = (Name)0; v < Name##__count; v = (Name)(v + 1))

/* ------------------------------------------------------------------- linalg */
typedef union { struct { f32 x, y; }; struct { f32 u, v; }; f32 data[2]; } Vec2;
typedef union { struct { f32 x, y, z; }; struct { f32 r, g, b; }; f32 data[3]; } Vec3;
typedef union { struct { f32 x, y, z, w; }; struct { f32 r, g, b, a; }; struct { Vec3 xyz; f32 _w; }; struct { Vec3 rgb; f32 _a; }; f32 data[4]; } Vec4;
typedef Vec3 Color3;
typedef Vec4 Color4;
typedef struct { f32 rows[3][3]; } Matrix_3x3;
typedef struct { f32 rows[4][4]; } Matrix_4x4;

#define vec2(...) ((Vec2){ __VA_ARGS__ })
#define vec3(...) ((Vec3){ __VA_ARGS__ })
#define vec4(...) ((Vec4){ __VA_ARGS__ })

#define sqrt_f32(x)      RT_SQRT_F32((f32)(x))
#define pow_f32(x, y)    rt_powf((f32)(x), (f32)(y))
#define sin_f32(x)       rt_sinf((f32)(x))
#define cos_f32(x)       rt_cosf((f32)(x))
#define tan_f32(x)       tanf((f32)(x))            /* host-only: camera focal length */
#define atan2_f32(y, x)  rt_atan2f((f32)(y), (f32)(x))
/* asin's argument is clamped like the oracle's (driver.c:100 feeds NaN into an integer cast otherwise) */
#define asin_f32(x)      rt_asinf(clamp((f32)(x), -1.0f, 1.0f))
internal inline f32 abs_f32(f32 x) { return x < 0 ? -x : x; }

internal inline Vec3 vec3_broadcast(f32 s)          { return vec3(s, s, s); }
internal inline Vec3 vec3_add(Vec3 a, Vec3 b)       { return vec3(a.x + b.x, a.y + b.y, a.z + b.z); }
internal inline Vec3 vec3_sub(Vec3 a, Vec3 b)       { return vec3(a.x - b.x, a.y - b.y, a.z - b.z); }
internal inline Vec3 vec3_mul(Vec3 a, Vec3 b)       { return vec3(a.x * b.x, a.y * b.y, a.z * b.z); }
internal inline Vec3 vec3_scale(Vec3 a, f32 s)      { return vec3(a.x * s, a.y * s, a.z * s); }
internal inline f32  vec3_dot(Vec3 a, Vec3 b)       { return a.x * b.x + a.y * b.y + a.z * b.z; }
internal inline f32  vec3_length2(Vec3 a)           { return vec3_dot(a, a); }
internal inline Vec3 vec3_cross(Vec3 a, Vec3 b)     { return vec3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
internal inline Vec3 vec3_normalize(Vec3 a)         { f32 inv = 1.0f / sqrt_f32(vec3_dot(a, a)); return vec3_scale(a, inv); }
internal inline Vec3 vec3_lerp(Vec3 a, Vec3 b, f32 t) { return vec3(a.x * (1 - t) + b.x * t, a.y * (1 - t) + b.y * t, a.z * (1 - t) + b.z * t); }
internal inline Vec3 vec3_reflect(Vec3 i, Vec3 n)   { return vec3_sub(i, vec3_scale(n, 2.0f * vec3_dot(i, n))); }
internal inline Vec2 vec2_sub(Vec2 a, Vec2 b)       { return vec2(a.x - b.x, a.y - b.y); }
internal inline Vec2 vec2_mul(Vec2 a, Vec2 b)       { return vec2(a.x * b.x, a.y * b.y); }
internal inline Vec2 vec2_fract(Vec2 a)             { return vec2(a.x - floorf(a.x), a.y - floorf(a.y)); }

internal inline Vec4 matrix_4x4_mul_vec4(Matrix_4x4 m, Vec4 v) {
  Vec4 r;
  for (int i = 0; i < 4; i++) r.data[i] = m.rows[i][0] * v.x + m.rows[i][1] * v.y + m.rows[i][2] * v.z + m.rows[i][3] * v.w;
  return r;
}
internal inline Matrix_4x4 matrix_4x4_translation_rotation_scale(Vec3 t, Vec4 q, Vec3 s) {
  f32 x = q.x, y = q.y, z = q.z, w = q.w;
  Matrix_4x4 m = {{
    { (1 - 2 * (y * y + z * z)) * s.x, (2 * (x * y - z * w)) * s.y,     (2 * (x * z + y * w)) * s.z,     t.x },
    { (2 * (x * y + z * w)) * s.x,     (1 - 2 * (x * x + z * z)) * s.y, (2 * (y * z - x * w)) * s.z,     t.y },
    { (2 * (x * z - y * w)) * s.x,     (2 * (y * z + x * w)) * s.y,     (1 - 2 * (x * x + y * y)) * s.z, t.z },
    { 0, 0, 0, 1 } }};
  return m;
}
internal inline Matrix_3x3 matrix_3x3_from_basis(Vec3 a, Vec3 b, Vec3 c) {
  Matrix_3x3 m = {{ { a.x, b.x, c.x }, { a.y, b.y, c.y }, { a.z, b.z, c.z } }};
  return m;
}
internal inline Matrix_3x3 matrix_3x3_transpose(Matrix_3x3 m) {
  Matrix_3x3 r;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) r.rows[i][j] = m.rows[j][i];
  return r;
}
internal inline Vec3 matrix_3x3_mul_vec3(Matrix_3x3 m, Vec3 v) {
  return vec3(m.rows[0][0] * v.x + m.rows[0][1] * v.y + m.rows[0][2] * v.z,
              m.rows[1][0] * v.x + m.rows[1][1] * v.y + m.rows[1][2] * v.z,
              m.rows[2][0] * v.x + m.rows[2][1] * v.y + m.rows[2][2] * v.z);
}

/* -------------------------------------------------------------------- image */
typedef enum { PT_u8 = 0 } Pixel_Type;
/* same field order as include/rt_base.h so one ctypes definition serves both */
typedef struct {
  Byte_Slice pixels;
  isize      width, height, stride;
  i32        components;
  i32        pixel_type;
} Image;

/* --------------------------------------------------------------------- time */
typedef i64 Timestamp;
typedef i64 Duration;
#define Nanosecond  ((i64)1)
#define Millisecond ((i64)1000000)
#define Second      ((i64)1000000000)
internal inline Timestamp time_now(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (i64)ts.tv_sec * Second + ts.tv_nsec; }
internal inline Duration  time_since(Timestamp t) { return time_now() - t; }
internal inline void      time_sleep(Duration d) { usleep((useconds_t)(d / 1000)); }

/* ------------------------------------------------------------------ threads */
typedef void (*Thread_Proc)(rawptr);
#define THREAD_STACK_DEFAULT 0
#define THREAD_TLS_DEFAULT   0
#define processor_yield() sched_yield()
void thread_create(Thread_Proc proc, rawptr arg, isize stack, isize tls);

/* ------------------------------------------------------------------- io, os */
typedef int Fd;
typedef struct { Fd fd; } Writer;
typedef struct { Fd value; int err; } Fd_Result;
typedef struct { Byte_Slice value; int err; } Bytes_Result;
enum { FP_Read_Write = 1, FP_Create = 2, FP_Truncate = 4 };
Fd_Result    file_open(String path, int flags);
Writer       writer_from_handle(Fd fd);
Bytes_Result read_entire_file_path(String path, Allocator a);
void         write_bytes(Writer const *w, Byte_Slice bytes);
#define write_any(w, ptr) write_bytes((w), (Byte_Slice){ .data = (byte *)(ptr), .len = size_of(*(ptr)) })
#define process_exit(code) exit(code)
bool png_save_writer(Writer const *w, Image const *image);
bool qoi_save_writer(Writer const *w, Image const *image);
bool ppm_save_writer(Writer const *w, Image const *image);
bool stb_image_load_bytes(Byte_Slice bytes, Image *image, Allocator a);

/* --------------------------------------------------------------------- sort */
/* UNPINNED: stable.  Merge-sorts an index permutation with the caller's
 * `less` expression (which indexes the unmodified slice through i and j), then
 * applies the permutation. */
#define sort_slice_by(slice, i, j, less)                                                     \
  do {                                                                                       \
    isize _n = (slice).len;                                                                  \
    if (_n < 2) break;                                                                       \
    isize *_a = malloc(sizeof(isize) * (usize)_n), *_b = malloc(sizeof(isize) * (usize)_n);  \
    for (isize _k = 0; _k < _n; _k++) _a[_k] = _k;                                           \
    for (isize _w = 1; _w < _n; _w *= 2) {                                                   \
      for (isize _lo = 0; _lo < _n; _lo += 2 * _w) {                                         \
        isize _mid = _lo + _w < _n ? _lo + _w : _n, _hi = _lo + 2 * _w < _n ? _lo + 2 * _w : _n; \
        isize _p = _lo, _q = _mid, _o = _lo;                                                 \
        while (_p < _mid && _q < _hi) {                                                      \
          isize i = _a[_q], j = _a[_p];                                                      \
          if (less) _b[_o++] = _a[_q++]; else _b[_o++] = _a[_p++];                           \
        }                                                                                    \
        while (_p < _mid) _b[_o++] = _a[_p++];                                               \
        while (_q < _hi)  _b[_o++] = _a[_q++];                                               \
      }                                                                                      \
      isize *_t = _a; _a = _b; _b = _t;                                                      \
    }                                                                                        \
    __typeof__((slice).data) _tmp = malloc(sizeof((slice).data[0]) * (usize)_n);             \
    for (isize _k = 0; _k < _n; _k++) _tmp[_k] = (slice).data[_a[_k]];                       \
    memcpy((slice).data, _tmp, sizeof((slice).data[0]) * (usize)_n);                         \
    free(_tmp); free(_a); free(_b);                                                          \
  } while (0)

/* ------------------------------------------------------------- obj and gltf */
typedef struct { String path; } Obj_Texture;
typedef struct {
  Vec3 diffuse, emissive;
  Obj_Texture texture_diffuse, texture_emissive;
  bool is_pbr;
  struct { f32 roughness, metallic, sheen, anisotropic; Obj_Texture texture_roughness, texture_metallic, texture_normal, texture_sheen; } pbr;
  struct { Obj_Texture texture_specular_color, texture_specular, texture_ambient, texture_alpha, texture_bump; } simple;
} Obj_Material;
typedef struct { Vec3 position, normal; Vec2 tex_coords; } Obj_Vertex;
typedef struct { Obj_Vertex vertices[3]; isize material; } Obj_Triangle;
typedef struct { Slice(Obj_Material) materials; Slice(Obj_Triangle) triangles; } Obj_File;
bool obj_load(String text, Obj_File *obj, bool flag, Allocator a);

typedef struct { isize index; } Gltf_Texture_Info;
typedef struct { isize camera; Matrix_4x4 matrix; } Gltf_Node;
typedef struct { bool is_orthographic; struct { f32 y_fov; } perspective; } Gltf_Camera;
typedef struct {
  Color4 base_color; f32 roughness, metallic; Color3 sheen_color; Vec3 emissive;
  Gltf_Texture_Info texture_normal, texture_emissive, texture_base_color, texture_metallic_roughness;
  f32 texture_normal_scale;
} Gltf_Material;
typedef struct { Byte_Slice data; String mime_type, uri; } Gltf_Image;
typedef struct { isize source, sampler; } Gltf_Texture;
typedef struct { int unused; } Gltf_Sampler;
typedef struct {
  Slice(Gltf_Node) nodes; Slice(Gltf_Camera) cameras; Slice(Gltf_Material) materials;
  Slice(Gltf_Image) images; Slice(Gltf_Texture) textures; Slice(Gltf_Sampler) samplers;
} Gltf_File;
typedef struct { Obj_Vertex vertices[3]; isize material; } Gltf_Triangle;
typedef Vector(Gltf_Triangle) Gltf_Triangle_Vector;
bool gltf_parse(Byte_Slice data, String path, Gltf_File *gltf, Allocator a);
bool gltf_load_buffers(String path, Gltf_File *gltf, Allocator a);
void gltf_to_triangles(Gltf_File *gltf, Gltf_Triangle_Vector *out);

#endif
