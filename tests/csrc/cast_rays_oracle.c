/* cast_rays_oracle.c — TEST INFRASTRUCTURE.  The CPU reference of rt_gpu_cast_rays (include/rt_gpu.h): cast_ray
 * (raytracer.c:505-558) for a batch of caller rays, path (i, s) traced with the shader generator seeded to
 * rt_path_seed(key_i, sample_begin + s, user_seed) just before it; sums[i] is the f32 sum over the samples in sample
 * order, from zero.
 *
 * The oracle's path loop (trace_path) and its work counters are file-local to oracle/oracle_trace.c, so this file
 * includes that source UNMODIFIED (as oracle/ref_glue_rt.c includes the reference's raytracer.c) and drives its
 * trace_path with the counters set, on threads.  The shading and environment callbacks stay liboracle.so's: the library
 * is linked against it, so oracle_shader_random_state() is the generator those callbacks draw from.
 * tests/test_oracle_cast_rays.py pins this file to liboracle.so's oracle_cast_ray and oracle_render.
 *
 * Build: gcc -O2 -std=gnu11 -mavx2 -mfma -ffp-contract=off -shared -fPIC -I include -I oracle ... -L oracle -loracle
 * (the oracle's own flags: no contraction, every product and sum rounds separately).
 */
#include "oracle_trace.c"

typedef struct {
  Scene const *scene;
  Ray const   *rays;
  u32 const   *keys;
  isize        n, sample_begin, samples, max_bounces;
  u32          user_seed;
  f32         *sums, *per_sample;
  atomic_long  next;
} Cast_Job;

typedef struct {
  Cast_Job *job;
  Counters  counters;
  pthread_t thread;
} Cast_Worker;

/* rays are dealt through one atomic counter; every path's arithmetic is its own, so the dealing changes nothing */
static void *cast_worker(void *arg) {
  Cast_Worker *w = arg;
  Cast_Job *job = w->job;
  tl_counters = &w->counters;
  u32 *rng = oracle_shader_random_state();
  for (;;) {
    isize i = atomic_fetch_add(&job->next, 1);
    if (i >= job->n) break;
    u32 key = job->keys ? job->keys[i] : (u32)i;
    Color3 sum = v3(0, 0, 0);
    for (isize s = 0; s < job->samples; s++) {
      *rng = rt_path_seed(key, (u32)(job->sample_begin + s), job->user_seed);
      Color3 radiance = trace_path(job->scene, job->rays[i], job->max_bounces, NULL);
      sum = v3_add(sum, radiance);
      w->counters.c[ORACLE_CTR_SAMPLES]++;
      if (job->per_sample) {
        f32 *dst = job->per_sample + ((size_t)i * (size_t)job->samples + (size_t)s) * 3;
        dst[0] = radiance.x; dst[1] = radiance.y; dst[2] = radiance.z;
      }
    }
    if (job->sums) {
      job->sums[3 * i + 0] = sum.x;
      job->sums[3 * i + 1] = sum.y;
      job->sums[3 * i + 2] = sum.z;
    }
  }
  tl_counters = NULL;
  return NULL;
}

/* sums (optional, n*3), per_sample (optional, n*samples*3), counters (optional, ORACLE_CTR_*, summed over threads) */
void oracle_cast_rays(Scene const *scene, Ray const *rays, u32 const *keys, isize n, isize sample_begin, isize samples,
                      isize max_bounces, u32 user_seed, f32 *sums, f32 *per_sample, u64 counters[8], i32 n_threads) {
  if (n_threads < 1) n_threads = 1;
  Cast_Job job = { scene, rays, keys, n, sample_begin, samples, max_bounces, user_seed, sums, per_sample, 0 };
  Cast_Worker *workers = calloc((size_t)n_threads, sizeof *workers);
  for (i32 i = 0; i < n_threads; i++) workers[i].job = &job;
  for (i32 i = 1; i < n_threads; i++) pthread_create(&workers[i].thread, NULL, cast_worker, &workers[i]);
  cast_worker(&workers[0]);
  for (i32 i = 1; i < n_threads; i++) pthread_join(workers[i].thread, NULL);
  if (counters) {
    memset(counters, 0, 8 * sizeof *counters);
    for (i32 i = 0; i < n_threads; i++)
      for (int k = 0; k < 8; k++) counters[k] += workers[i].counters.c[k];
  }
  free(workers);
}
