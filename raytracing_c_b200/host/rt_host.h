/* rt_host.h — host-side (CPU, plain C) services around the GPU path: model
 * ingestion, image decode/encode, default camera, procedural environment.
 * These mirror what the reference's driver.c does through Codin
 * (driver.c:106-116, 510-728, 747-767, 839-873); none of it is on the GPU.
 */
#ifndef RT_HOST_H
#define RT_HOST_H

#include "scene.h"
#include "rt_pbr.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
  Triangle_Slice   triangles;     /* shader.data points into `materials` */
  PBR_Shader_Data *materials;
  isize            n_materials;
  Image           *images;        /* decoded textures, referenced by materials */
  isize            n_images;
} RT_Model;

/* driver.c:685-728.  `proc` is stamped into every triangle's Shader (the
 * reference stamps disney_shader_proc, driver.c:574-577,670-673).  `camera` is
 * overwritten only when the file carries a perspective camera (glTF). */
bool rt_load_model_file(char const *path, Shader_Proc proc, RT_Model *model, Camera *camera);
void rt_model_free(RT_Model *model);

/* driver.c:765-767: translation (0,0,3), identity rotation, fov 70 degrees. */
void rt_camera_default(Camera *camera);
/* Look-at helper for the camera overrides BASELINE configs 2 and 5 need. */
void rt_camera_look_at(Camera *camera, Vec3 eye, Vec3 target, Vec3 up, f32 fov_radians);

/* stb_image_load_bytes stand-in (driver.c:107,621): baseline JPEG and PNG. */
bool rt_image_decode(u8 const *bytes, size_t len, Image *out);
/* With deferral on, baseline JPEGs are not decoded on the host: rt_image_decode / rt_load_texture / the glTF loader
 * return Images that carry the compressed bytes (pixel_type PT_RT_JPEG_BYTES, rt_base.h) for the GPU library to
 * decode during the scene upload.  Such images cannot be sampled on the CPU. */
void rt_host_defer_jpeg_decode(bool on);
/* driver.c:106-116 */
bool rt_load_texture(char const *path, Image *out);
void rt_image_free(Image *image);
Image rt_image_alloc(isize width, isize height, i32 components);

/* background.png is not in the reference tree (.MISSING_LARGE_BLOBS:1); this
 * is the deterministic stand-in (integer arithmetic only). */
void rt_generate_background(Image *out, isize width, isize height);

/* driver.c:839-873: encoder chosen by suffix (.png stored-deflate, .qoi, .ppm). */
bool rt_save_image(char const *path, Image const *image);
bool rt_save_png(char const *path, Image const *image);
bool rt_save_qoi(char const *path, Image const *image);
bool rt_save_ppm(char const *path, Image const *image);

/* Where texels, BVH nodes, the triangle block and images come from (default: aligned_alloc).  A GPU host installs
 * rt_gpu_host_alloc / rt_gpu_host_free so these buffers are pinned and the scene upload DMA-reads them in place. */
void  rt_host_set_buffer_allocator(void *(*alloc)(size_t), void (*release)(void *));
void *rt_host_buffer_alloc(size_t bytes);
void  rt_host_buffer_free(void *p);

/* The scene cache (reference scene.c:13-76, scene_save_writer / scene_load_bytes): the reference's container, with
 * material indices where the reference writes raw Shader pointers (host/scene_cache.c).  A loaded scene owns its
 * buffers like one from scene_init (scene_destroy releases them); `materials` / `proc` re-bind the shaders. */
bool scene_save_file(char const *path, Scene const *scene, PBR_Shader_Data const *materials, isize n_materials);
bool scene_load_file(char const *path, Scene *scene, PBR_Shader_Data *materials, isize n_materials, Shader_Proc proc);

/* scene_init that also reports where each source triangle went: slot_of_triangle[i] = the slot of src[i] (NULL
 * allowed; scene_init is this call with NULL).  A host that keeps its vertices in source order (skinning output, a
 * simulation) scatters them through this map into the slot order rt_gpu_scene_refit* takes. */
void rt_scene_init_slots(Scene *scene, Triangle_Slice src, i32 *slot_of_triangle);

char const *rt_host_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
