/* ref_query_glue.c — TEST INFRASTRUCTURE.  oracle/ref_glue_rt.c (the reference's raytracer.c, unmodified, with its
 * doors) plus one more door: ray_scene_hit started with hit.distance = t_max, the reference's own form of a ray query.
 * Compiled only where a reference checkout is available, with the flags of oracle/Makefile's `ref` target, in place of
 * ref_glue_rt.c (tests/query_ffi.py). */
#include "ref_glue_rt.c"

/* raytracer.c:497 with an initial distance */
void ref_query_ray(Scene const *scene, Ray ray, f32 t_max, Ref_Hit *out) {
  Hit hit = { .distance = t_max, };
  ray_scene_hit(&ray, scene, &hit);
  out->distance = hit.distance; out->normal = hit.normal; out->normal_geo = hit.normal_geo; out->point = hit.point;
  out->tangent = hit.tangent; out->bitangent = hit.bitangent; out->tex_coords = hit.tex_coords; out->shader_data = hit.shader.data;
}
