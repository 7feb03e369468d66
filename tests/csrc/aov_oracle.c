/* aov_oracle.c — TEST INFRASTRUCTURE.  The CPU reference of rt_gpu_render_aov (include/rt_gpu.h): for every pixel and
 * every sample of [sample_begin, sample_end), the renderer's camera ray (oracle_render's lines, oracle_trace.c:335-374,
 * one lane at a time with the exact 1/sqrt), walked through back faces as trace_path does (raytracer.c:516-522) for at
 * most max_bounces walks; at the first front face the material is fetched as the oracle's shader fetches it.  Per pixel
 * the records are summed in sample order, from zero.
 *
 * Like cast_rays_oracle.c, this file includes the oracle's sources UNMODIFIED: oracle_trace.c for its closest_hit, Hit
 * record and work counters, oracle_shade.c for the texture fetch, sRGB decode and normal mapping its shader uses.
 * aov_surface below is the first half of oracle_disney_shader_proc (oracle_shade.c:210-231, reference
 * driver.c:129-153,350-367) line for line, stopped before the BSDF draws its random numbers;
 * tests/test_oracle_aov.py pins it to the oracle renderer.
 *
 * Build: gcc -O2 -std=gnu11 -mavx2 -mfma -ffp-contract=off -shared -fPIC -I include -I oracle ...
 * (the oracle's own flags: no contraction, every product and sum rounds separately).
 */
#include "oracle_trace.c"
#include "oracle_shade.c"

/* oracle_shade.c:210-231: shading normal, base colour, roughness and metalness after their textures and rescale, emission */
static void aov_surface(PBR_Shader_Data const *mat, Shader_Input const *in, Vec3 *n_out, Color3 *base_out,
                        f32 *roughness_out, f32 *metalness_out, Color3 *glow_out) {
  Vec3 n = perturb_normal(mat->texture_normal, mat->normal_map_strength, in);

  Color3 base = mat->base_color;
  if (mat->texture_albedo)
    base = v3_mul(base, decode_srgb(oracle_sample_texture_bilinear(mat->texture_albedo, in->tex_coords)));

  f32 roughness = mat->roughness, metalness = mat->metalness;
  if (mat->texture_metal_roughness) {
    Vec3 mr = oracle_sample_texture_bilinear(mat->texture_metal_roughness, in->tex_coords);
    roughness *= mr.y;
    metalness *= mr.z;
  }
  roughness = f32_clamp(roughness, 0.001f, 1);
  if (metalness > 0.9f) metalness = 0.9f;
  metalness /= 0.9f;

  Color3 glow = mat->emission;
  if (mat->texture_emission)
    glow = v3_mul(glow, decode_srgb(oracle_sample_texture_bilinear(mat->texture_emission, in->tex_coords)));
  *n_out = n;
  *base_out = base;
  *roughness_out = roughness;
  *metalness_out = metalness;
  *glow_out = glow;
}

enum { AOV_FLOATS = 16 };            /* RT_GPU_AOV: albedo, coverage, normal, depth, position, roughness, emission, metalness */

typedef struct {
  Scene const *scene;
  isize        width, height, sample_begin, sample_end, max_bounces;
  f32         *aov;                  /* [height][width][AOV_FLOATS] */
  atomic_long  next_row;
} Aov_Job;

typedef struct {
  Aov_Job  *job;
  Counters  counters;
  pthread_t thread;
} Aov_Worker;

/* the first-surface record of one camera ray added to sum[AOV_FLOATS]; false if the sample has no surface */
static bool aov_sample(Aov_Job const *job, Ray ray, Vec3 eye, f32 *sum) {
  for (isize walk = 0; walk < job->max_bounces; walk++) {
    Hit hit;
    memset(&hit, 0, sizeof hit);
    hit.distance = INFINITY;
    hit.slot = -1;
    closest_hit(&ray, job->scene, &hit);
    if (hit.distance == INFINITY) {
      tl_counters->c[ORACLE_CTR_MISSES]++;
      return false;
    }
    if (v3_dot(hit.normal_geo, ray.direction) > 0 || v3_dot(hit.normal, ray.direction) > 0) {
      tl_counters->c[ORACLE_CTR_PASSTHROUGH]++;
      ray.position = v3_add(hit.point, v3_scale(ray.direction, RT_EPSILON));
      continue;
    }
    Shader_Input in;
    memset(&in, 0, sizeof in);
    in.direction  = ray.direction;
    in.normal     = v3_normalize(hit.normal);
    in.normal_geo = hit.normal_geo;
    in.tangent    = hit.tangent;
    in.bitangent  = hit.bitangent;
    in.position   = hit.point;
    in.tex_coords = hit.tex_coords;
    tl_counters->c[ORACLE_CTR_SHADES]++;
    Vec3 n;
    Color3 base, glow;
    f32 roughness, metalness;
    aov_surface((PBR_Shader_Data const *)hit.shader.data, &in, &n, &base, &roughness, &metalness, &glow);
    f32 dx = hit.point.x - eye.x, dy = hit.point.y - eye.y, dz = hit.point.z - eye.z;
    f32 depth = sqrtf(dx * dx + dy * dy + dz * dz);
    f32 const rec[AOV_FLOATS] = { base.x, base.y, base.z, 1.0f, n.x, n.y, n.z, depth,
                                  hit.point.x, hit.point.y, hit.point.z, roughness, glow.x, glow.y, glow.z, metalness };
    for (int k = 0; k < AOV_FLOATS; k++) sum[k] += rec[k];
    return true;
  }
  return false;
}

static void *aov_worker(void *arg) {
  Aov_Worker *w = arg;
  Aov_Job *job = w->job;
  tl_counters = &w->counters;
  Camera const *cam = &job->scene->camera;
  f32 const (*m)[4] = cam->view_matrix.rows;
  Vec3 eye = v3(m[0][3], m[1][3], m[2][3]);
  isize width = job->width, height = job->height;
  f32 inv_width = 1.0f / (f32)width, inv_height = 1.0f / (f32)height, aspect = (f32)width / (f32)height;
  for (;;) {
    isize y = atomic_fetch_add(&job->next_row, 1);
    if (y >= height) break;
    for (isize x = 0; x < width; x++) {
      f32 *sum = job->aov + (y * width + x) * AOV_FLOATS;
      memset(sum, 0, AOV_FLOATS * sizeof *sum);
      for (isize s = job->sample_begin; s < job->sample_end; s++) {
        /* oracle_trace.c:340-365 for one lane */
        f32 jit = oracle_hash12((f32)x * 50.0f + (f32)s, (f32)y);
        f32 ux = ((f32)x + jit - 0.5f) * 2.0f * inv_width - 1.0f;
        f32 uy = ((f32)y + jit - 0.5f) * 2.0f * inv_height - 1.0f;
        f32 cx = ux * aspect, cy = -uy, cz = -cam->focal_length;
        f32 inv_len = 1.0f / sqrtf(cx * cx + cy * cy + cz * cz);
        Ray r;
        r.position  = eye;
        r.direction = v3((m[0][0] * cx + m[0][1] * cy + m[0][2] * cz) * inv_len,
                         (m[1][0] * cx + m[1][1] * cy + m[1][2] * cz) * inv_len,
                         (m[2][0] * cx + m[2][1] * cy + m[2][2] * cz) * inv_len);
        aov_sample(job, r, eye, sum);
        w->counters.c[ORACLE_CTR_SAMPLES]++;
      }
    }
  }
  tl_counters = NULL;
  return NULL;
}

/* aov: width*height*16 f32 in RT_GPU_AOV order; counters (optional, ORACLE_CTR_*, summed over threads).  A call with
 * max_bounces = 0 or an empty range gives zero records and counts nothing, as the GPU call. */
void oracle_render_aov(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                       isize max_bounces, f32 *aov, u64 counters[8], i32 n_threads) {
  if (n_threads < 1) n_threads = 1;
  Aov_Job job = { scene, width, height, sample_begin, sample_end, max_bounces, aov, 0 };
  if (sample_end <= sample_begin || max_bounces < 1) {
    memset(aov, 0, (size_t)(width * height * AOV_FLOATS) * sizeof *aov);
    if (counters) memset(counters, 0, 8 * sizeof *counters);
    return;
  }
  Aov_Worker *workers = calloc((size_t)n_threads, sizeof *workers);
  for (i32 i = 0; i < n_threads; i++) workers[i].job = &job;
  for (i32 i = 1; i < n_threads; i++) pthread_create(&workers[i].thread, NULL, aov_worker, &workers[i]);
  aov_worker(&workers[0]);
  for (i32 i = 1; i < n_threads; i++) pthread_join(workers[i].thread, NULL);
  if (counters) {
    memset(counters, 0, 8 * sizeof *counters);
    for (i32 i = 0; i < n_threads; i++)
      for (int k = 0; k < 8; k++) counters[k] += workers[i].counters.c[k];
  }
  free(workers);
}
