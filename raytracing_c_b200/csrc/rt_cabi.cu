// rt_cabi.cu — the C ABI of libraytracer_gpu.so.
//
// Exports the reference's own entry points (raytracer.h:51-56, denoiser.h:4) plus the additive rt_gpu_* calls
// declared in include/rt_gpu.h.  Host-side work here:
//   * the reference's threading protocol around render_thread_proc (driver.c:793-818): the thread that claims
//     chunk 0 owns the launch;
//   * one frame over 1..N devices of this process: split (rt_multi.cu), per-device wavefront render
//     (rt_render.cu), fused reduce + resolve on the first device, D2H of the u8 image;
//   * per-call status: the reference's entry points return void, rt_gpu_last_status() says whether the last one failed.
// Scene residency is rt_scene.cu.  There is no CPU fallback: every compute call fails if CUDA does.
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sched.h>
#include <thread>

#include "rt_state.h"
#include "rt_gpu_internal.h"

namespace rt {

State g;
std::mutex g_mutex;

namespace {
std::mutex g_error_mutex;
char g_error_shared[512] = "";
thread_local char g_error_copy[512] = "";
std::atomic<int> g_status{0};
}

int fail(const char *fmt, ...) {
  char text[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(text, sizeof text, fmt, ap);
  va_end(ap);
  std::lock_guard<std::mutex> lock(g_error_mutex);
  memcpy(g_error_shared, text, sizeof text);
  return 1;
}

void clear_error() {
  std::lock_guard<std::mutex> lock(g_error_mutex);
  g_error_shared[0] = 0;
}

int launch_failed(const char *what, int launch_error) {
  if (launch_error) return fail("%s kernel launch failed: %s", what, cudaGetErrorString((cudaError_t)launch_error));
  return 0;
}

}  // namespace rt

using namespace rt;

namespace {

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

int init_devices_locked(int n, const int *ids) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail("no CUDA device available (%s); libraytracer_gpu has no CPU fallback", cudaGetErrorString(e));
  if (n < 1 || n > RT_MAX_PARTS) return fail("init: between 1 and %d devices, got %d", RT_MAX_PARTS, n);
  std::vector<int> want;
  for (int k = 0; k < n; k++) {
    const int id = ids ? ids[k] : k;
    if (id < 0 || id >= count || id >= RT_MAX_DEVICES) return fail("device %d out of range (%d visible)", id, count);
    for (int prev : want) if (prev == id) return fail("device %d listed twice", id);
    want.push_back(id);
  }
  if (g.ready) {
    bool same = g.devs.size() == want.size();
    for (size_t k = 0; same && k < want.size(); k++) same = g.devs[k].id == want[k];
    if (same) return 0;
    nccl_shutdown();
    ipc_close_all();
    for (Device &d : g.devs) release_device(d);
    g.devs.clear();
    g.ready = false;
    g.peers_enabled = false;
  }
  g.devs.resize(want.size());
  if (want.size() > 1) {
    // a CUDA context takes ~0.9 s to create; the contexts of different devices can be created side by side
    std::vector<std::thread> makers;
    for (int id : want) makers.emplace_back([id] { if (cudaSetDevice(id) == cudaSuccess) cudaFree(nullptr); });
    for (std::thread &t : makers) t.join();
    cudaGetLastError();
  }
  for (size_t k = 0; k < want.size(); k++) {
    Device &d = g.devs[k];
    CUDA_TRY(cudaSetDevice(want[k]));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, want[k]));
    if (prop.major < 10) return fail("device %d is sm_%d%d; this library is built for sm_100a only", want[k], prop.major, prop.minor);
    d.id = want[k];
    d.sm_count = prop.multiProcessorCount;
    d.l2_persist_max = prop.persistingL2CacheMaxSize > 0 ? (size_t)prop.persistingL2CacheMaxSize : 0;
    d.l2_window_max = prop.accessPolicyMaxWindowSize > 0 ? (size_t)prop.accessPolicyMaxWindowSize : 0;
    CUDA_TRY(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&d.copy, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&d.ev0));
    CUDA_TRY(cudaEventCreate(&d.ev1));
    CUDA_TRY(cudaEventCreateWithFlags(&d.busy, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&d.done, cudaEventDisableTiming));
  }
  CUDA_TRY(cudaSetDevice(want[0]));
  g.ready = true;
  return 0;
}

int ensure_init() {
  if (g.ready) return 0;
  const int zero = 0;
  return init_devices_locked(1, &zero);
}

// bytes of path-queue workspace a call asks for: the preferred size and the least it accepts (want 0: none)
struct WorkspaceRequest { size_t want = 0, floor = 0; };

// the camera path's request (render, AOV) for n_samples samples of every pixel: one chunk of them, or one sample
WorkspaceRequest camera_workspace(isize width, isize height, isize n_samples, isize max_bounces, int split_world) {
  return {rt_render_workspace_bytes((int)width, (int)height, (int)n_samples, (int)max_bounces, split_world),
          rt_render_workspace_bytes((int)width, (int)height, 1, (int)max_bounces, split_world)};
}

// Path-queue workspace of one device.  The preferred size (up to 26.6 GB) is a throughput choice, not a requirement:
// on a device that cannot spare it the request is halved down to the floor (one sample of every pixel per chunk for
// a render), and the size that was refused is remembered so later calls do not walk the same ladder again.
int ensure_workspace(Device &d, const WorkspaceRequest &r, cudaStream_t stream) {
  const size_t want = r.want, floor_bytes = r.floor;
  if (d.workspace_bytes >= want) return 0;
  if (d.workspace_denied && want >= d.workspace_denied && d.workspace_bytes >= floor_bytes) return 0;
  CUDA_TRY(cudaStreamSynchronize(stream));      // an earlier launch may still read the old queues
  CUDA_TRY(cudaStreamSynchronize(d.stream));
  size_t ask = want + want / 50;      // 2 % headroom: a slightly larger request later (another split, another slice) fits
  for (;;) {
    if (d.d_workspace) { cudaFree(d.d_workspace); d.d_workspace = nullptr; d.workspace_bytes = 0; }
    if (cudaMalloc(&d.d_workspace, ask) == cudaSuccess) { d.workspace_bytes = ask; break; }
    cudaGetLastError();                          // clear the allocation failure
    d.d_workspace = nullptr;
    d.workspace_denied = ask;
    if (ask <= floor_bytes) return fail("render: cannot allocate %zu bytes of path queues", ask);
    ask = ask / 2 > floor_bytes ? ask / 2 : floor_bytes;
  }
  return 0;
}

// Every user of a device's path-queue workspace (render, lightmap bake, cast_rays, AOV) is serialised on the device
// whatever stream it comes from: it waits for the event the previous user recorded (busy) and records busy after its
// last kernel.  Renders and AOV calls also rewrite the scene's camera-relative copies, which the same event covers.
// A user waits for the scene's geometry, and for its texels unless its launch defers that wait (the renderer's
// shading_ready).
int workspace_begin(Device &d, const DeviceScene &ds, const WorkspaceRequest &r, bool wait_texels, cudaStream_t stream) {
  if (ensure_workspace(d, r, stream)) return 1;
  if (d.busy_valid) CUDA_TRY(cudaStreamWaitEvent(stream, d.busy, 0));
  CUDA_TRY(cudaStreamWaitEvent(stream, ds.geom_ready, 0));
  if (wait_texels) CUDA_TRY(cudaStreamWaitEvent(stream, ds.tex_ready, 0));
  set_l2_window(d, ds, stream);
  return 0;
}

int workspace_end(Device &d, const char *what, int launch_error, cudaStream_t stream) {
  if (launch_failed(what, launch_error)) return 1;
  CUDA_TRY(cudaEventRecord(d.busy, stream));
  d.busy_valid = true;
  return 0;
}

// the result of a launcher that enqueues one kernel: an error fails the call, a success counts the launch
int launched(const char *what, int launch_error) {
  if (launch_failed(what, launch_error)) return 1;
  g.last_launches++;
  return 0;
}

// The reference's entry points return void: whether `call` failed is left for rt_gpu_last_status, and a failure is
// also reported on stderr.
template <class Call>
void report_status(const char *entry, Call call) {
  clear_error();
  g_status.store(0);
  if (call()) {
    g_status.store(1);
    fprintf(stderr, "%s: %s\n", entry, rt_gpu_last_error());
  }
}

// An image's round trip through the pinned buffer: d.d_image and the pinned buffer sized for it, the caller's image
// up into d.d_image, and an image on the device back, all on d.stream.
int image_buffers(Device &d, size_t bytes) {
  if (grow(reinterpret_cast<void **>(&d.d_image), &d.image_bytes, bytes)) return 1;
  return grow_pinned(d, bytes);
}

int image_to_device(Device &d, const void *pixels, size_t bytes) {
  memcpy(d.h_pinned, pixels, bytes);
  CUDA_TRY(cudaMemcpyAsync(d.d_image, d.h_pinned, bytes, cudaMemcpyHostToDevice, d.stream));
  return 0;
}

// into the pinned buffer, synchronised: the renderer times its own copy out, the denoiser keeps padded rows' bytes
int image_to_pinned(Device &d, const unsigned char *d_pixels, size_t bytes) {
  CUDA_TRY(cudaMemcpyAsync(d.h_pinned, d_pixels, bytes, cudaMemcpyDeviceToHost, d.stream));
  CUDA_TRY(cudaStreamSynchronize(d.stream));
  return 0;
}

int image_from_device(Device &d, const unsigned char *d_pixels, size_t bytes, void *pixels) {
  if (image_to_pinned(d, d_pixels, bytes)) return 1;
  memcpy(pixels, d.h_pinned, bytes);
  return 0;
}

struct Share {            // what one device (or process) renders of a frame
  isize s_begin, s_end;
  int   split_rank, split_world;
};

// the views of a many-view call (rt_gpu_render_views_device): cameras and optional seeds, host arrays of n
struct Views { int n; const ViewCamera *cameras; const u32 *seeds; };

// One render of `share` on device d, enqueued on `stream`: a workspace user.  d_mask / d_accum_sq (optional) make it a
// masked pass (rt_gpu_render_masked_device); `views` (optional) renders each of them into its slice of d_accum
// (rt_gpu_render_views_device).
int render_on_device(Device &d, const Scene *scene, isize width, isize height, const Share &share, isize max_bounces,
                     u32 seed, int accumulate, float *d_accum, float *d_per_sample, int *d_hit_ids,
                     unsigned long long *d_counters, cudaStream_t stream, const u8 *d_mask = nullptr,
                     float *d_accum_sq = nullptr, const Views *views = nullptr) {
  if (width < 1 || height < 1) return fail("render: empty image");
  CUDA_TRY(cudaSetDevice(d.id));
  auto it = d.scenes.find(scene);
  if (it == d.scenes.end()) return fail("render: scene is not resident on device %d", d.id);
  const DeviceScene &ds = it->second;
  const isize n_samples = share.s_end - share.s_begin;
  WorkspaceRequest r;
  if (n_samples > 0 && views)
    r = {rt_render_views_workspace_bytes((int)width, (int)height, views->n, (int)n_samples, (int)max_bounces, false),
         rt_render_views_workspace_bytes((int)width, (int)height, views->n, 1, (int)max_bounces, true)};
  else if (n_samples > 0)
    r = camera_workspace(width, height, n_samples, max_bounces, share.split_world);
  if (workspace_begin(d, ds, r, false, stream)) return 1;
  RenderParams p{};
  p.scene = ds.dev;
  p.shading_ready = ds.tex_ready;
  p.fast = g.options.fast_math != 0;
  p.width = (int)width; p.height = (int)height;
  p.split_rank = share.split_rank; p.split_world = share.split_world;
  p.sample_begin = (int)share.s_begin; p.sample_end = (int)share.s_end; p.max_bounces = (int)max_bounces;
  p.user_seed = seed;
  p.accumulate = accumulate;
  p.accum = d_accum; p.per_sample = d_per_sample; p.hit_ids = d_hit_ids;
  p.counters = d_counters;
  p.counters_ex = (d_counters && d_counters == d.d_counters) ? d_counters + 8 : nullptr;   // the library's own buffer has 16 slots
  p.pixel_mask = d_mask; p.accum_sq = d_accum_sq;
  if (views) {
    p.n_views = views->n; p.cameras = views->cameras; p.user_seeds = views->seeds;
    p.view_stride = (size_t)width * (size_t)height * 3;
  }
  return workspace_end(d, "render", rt_launch_render(p, d.sm_count, d.d_workspace, d.workspace_bytes, stream, &g.last_launches),
                       stream);
}

int ensure_frame_buffers(Device &d, size_t n_pixels, bool hit_ids) {
  CUDA_TRY(cudaSetDevice(d.id));
  size_t have = d.accum_floats * sizeof(float);
  if (grow(reinterpret_cast<void **>(&d.d_accum), &have, n_pixels * 3 * sizeof(float))) return 1;
  d.accum_floats = have / sizeof(float);
  if (hit_ids) {
    have = d.hit_pixels * sizeof(int);
    if (grow(reinterpret_cast<void **>(&d.d_hit_ids), &have, n_pixels * sizeof(int))) return 1;
    d.hit_pixels = have / sizeof(int);
  }
  if (!d.d_counters) CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d.d_counters), 16 * sizeof(unsigned long long)));
  return 0;
}

}  // namespace

// ======================================================================= ABI
extern "C" {

int rt_gpu_init(int device) {
  std::lock_guard<std::mutex> lock(g_mutex);
  return init_devices_locked(1, &device);
}

int rt_gpu_init_devices(int n_devices, int const *devices) {
  std::lock_guard<std::mutex> lock(g_mutex);
  return init_devices_locked(n_devices, devices);
}

int rt_gpu_device_count(void) { return g.ready ? (int)g.devs.size() : 0; }

int rt_gpu_visible_devices(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
  return count;
}

void rt_gpu_shutdown(void) {
  std::lock_guard<std::mutex> lock(g_mutex);
  nccl_shutdown();
  ipc_close_all();
  jpeg_shutdown();
  for (Device &d : g.devs) release_device(d);
  std::vector<Shader_Proc> pbr = g.pbr_procs;
  std::vector<Background_Proc> bg = g.bg_procs;
  g = State{};
  g.pbr_procs = pbr;
  g.bg_procs = bg;
}

char const *rt_gpu_last_error(void) {
  std::lock_guard<std::mutex> lock(g_error_mutex);
  memcpy(g_error_copy, g_error_shared, sizeof g_error_copy);
  return g_error_copy;
}

int rt_gpu_last_status(void) { return g_status.load(); }

int rt_gpu_sm_count(void) {
  std::lock_guard<std::mutex> lock(g_mutex);
  return ensure_init() ? 0 : g.devs[0].sm_count;
}

f64 rt_gpu_measure_fp32_issue(void) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 0;
  cudaSetDevice(g.devs[0].id);
  return rt_measure_fp32_issue(g.devs[0].sm_count, g.devs[0].stream, nullptr);
}

isize rt_gpu_scene_device_bytes(Scene const *scene) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g.devs.empty()) return 0;
  auto it = g.devs[0].scenes.find(scene);
  return it == g.devs[0].scenes.end() ? 0 : (isize)it->second.bytes;
}

isize rt_gpu_scene_upload_bytes(Scene const *scene) {
  std::lock_guard<std::mutex> lock(g_mutex);
  isize total = 0;
  for (Device &d : g.devs) {
    auto it = d.scenes.find(scene);
    if (it != d.scenes.end()) total += (isize)it->second.h2d_bytes;
  }
  return total;
}

void rt_gpu_register_pbr_shader(Shader_Proc proc) {
  std::lock_guard<std::mutex> lock(g_mutex);
  for (Shader_Proc p : g.pbr_procs) if (p == proc) return;
  g.pbr_procs.push_back(proc);
}

void rt_gpu_register_background(Background_Proc proc) {
  std::lock_guard<std::mutex> lock(g_mutex);
  for (Background_Proc p : g.bg_procs) if (p == proc) return;
  g.bg_procs.push_back(proc);
}

void rt_gpu_pbr_shader_proc(rawptr, Shader_Input const *, Shader_Output *) {
  fprintf(stderr, "rt_gpu_pbr_shader_proc called on the CPU: this build has no CPU shading path\n");
  abort();
}

Color3 rt_gpu_background_proc(rawptr, Vec3) {
  fprintf(stderr, "rt_gpu_background_proc called on the CPU: this build has no CPU shading path\n");
  abort();
}

int rt_gpu_scene_upload(Scene const *scene) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  if (g.devs.size() > 1 && enable_peers()) return 1;
  return scene_upload_all(scene);
}

void rt_gpu_scene_release(Scene const *scene) {
  std::lock_guard<std::mutex> lock(g_mutex);
  scene_release_all(scene);
}

void *rt_gpu_host_alloc(size_t bytes) {
  void *p = nullptr;
  // portable: pinned for every device this process drives, not only the current one
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    fail("rt_gpu_host_alloc(%zu): %s", bytes, cudaGetErrorString(cudaGetLastError()));
    return nullptr;
  }
  return p;
}

void rt_gpu_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

// Allocates what a frame of this size will need (accumulators, image, path-queue workspace on every device) ahead of
// the first render, so the allocations (tens of ms for a 69 GB workspace) can overlap the host's model load.
int rt_gpu_prepare_frame(isize width, isize height, isize samples, isize max_bounces) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  if (width < 1 || height < 1 || samples < 1 || max_bounces < 1) return fail("prepare_frame: empty frame");
  const size_t n_dev = g.devs.size();
  if (n_dev > 1 && enable_peers()) return 1;
  const i32 mode = n_dev > 1 ? rt_gpu_shard_mode((i32)samples, (i32)n_dev, g.options.split_mode) : RT_GPU_SPLIT_SAMPLES;
  const int world = n_dev > 1 && mode == RT_GPU_SPLIT_CHUNKS ? (int)n_dev : 1;
  isize share = samples;
  if (n_dev > 1 && mode == RT_GPU_SPLIT_SAMPLES) share = (samples + (isize)n_dev - 1) / (isize)n_dev;
  isize slice = g.options.slice_samples > 0 ? g.options.slice_samples : rt_render_chunk_samples((int)width, (int)height, world);
  if (slice > share) slice = share;
  for (Device &d : g.devs) {
    if (ensure_frame_buffers(d, (size_t)width * (size_t)height, g.options.keep_hit_ids != 0)) return 1;
    if (ensure_workspace(d, camera_workspace(width, height, slice, max_bounces, world), d.stream)) return 1;
  }
  if (n_dev > 1 && g.options.reduce_mode == RT_GPU_REDUCE_NCCL && nccl_prepare()) return 1;
  CUDA_TRY(cudaSetDevice(g.devs[0].id));
  return 0;
}

void rt_gpu_set_options(RT_GPU_Options const *options) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.options = *options;
  if (g.options.slice_samples < 0) g.options.slice_samples = 0;
  // the communicator costs seconds to create: when the NCCL film is asked for, do it here, not inside the first frame
  if (g.ready && g.devs.size() > 1 && g.options.reduce_mode == RT_GPU_REDUCE_NCCL) nccl_prepare();
}

void rt_gpu_get_options(RT_GPU_Options *options) {
  std::lock_guard<std::mutex> lock(g_mutex);
  *options = g.options;
}

// ------------------------------------------------------------ device-pointer level
int rt_gpu_render_accum_device(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                               isize max_bounces, u32 user_seed, i32 accumulate, f32 *d_accum, f32 *d_per_sample,
                               i32 *d_hit_ids, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  if (scene_on_devices(scene)) return 1;
  const Share share{sample_begin, sample_end, g.options.pixel_rank, g.options.pixel_world};
  return render_on_device(g.devs[0], scene, width, height, share, max_bounces, user_seed, accumulate, d_accum, d_per_sample,
                          d_hit_ids, reinterpret_cast<unsigned long long *>(d_counters), static_cast<cudaStream_t>(stream));
}

int rt_gpu_render_shard_device(Scene const *scene, isize width, isize height, isize samples, isize max_bounces,
                               u32 user_seed, i32 rank, i32 world, i32 split_mode, i32 *mode_used,
                               f32 *d_accum, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  if (world < 1 || rank < 0 || rank >= world) return fail("render_shard: rank %d of %d", rank, world);
  if (scene_on_devices(scene)) return 1;
  const i32 mode = rt_gpu_shard_mode((i32)samples, world, split_mode);
  if (mode_used) *mode_used = mode;
  Share share{0, samples, 0, 1};
  if (mode == RT_GPU_SPLIT_SAMPLES) {
    i32 a = 0, b = 0;
    rt_gpu_shard_samples(rank, world, (i32)samples, &a, &b);
    share.s_begin = a; share.s_end = b;
  } else {
    share.split_rank = rank; share.split_world = world;
  }
  return render_on_device(g.devs[0], scene, width, height, share, max_bounces, user_seed, 0, d_accum, nullptr, nullptr,
                          reinterpret_cast<unsigned long long *>(d_counters), static_cast<cudaStream_t>(stream));
}

int rt_gpu_accum_buffer(isize width, isize height, f32 **d_accum_out) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  if (width < 1 || height < 1) return fail("accum_buffer: empty image");
  if (ensure_frame_buffers(g.devs[0], (size_t)width * (size_t)height, false)) return 1;
  *d_accum_out = g.devs[0].d_accum;
  return 0;
}

int rt_gpu_reduce_resolve_device(f32 const *const *d_parts, i32 n_parts, f32 *d_sum_out, isize width, isize height,
                                 isize samples, u8 *d_pixels, isize stride, i32 components, void *stream) {
  if (n_parts < 1 || n_parts > RT_MAX_PARTS) return fail("reduce_resolve: between 1 and %d parts", RT_MAX_PARTS);
  if (samples < 1 || (d_pixels && components < 3)) return fail("reduce_resolve: samples >= 1 and components >= 3 required");
  ReduceParts parts{};
  parts.n = n_parts;
  for (int k = 0; k < n_parts; k++) parts.part[k] = d_parts[k];
  return launched("reduce+resolve", rt_launch_reduce_resolve(parts, d_sum_out, (int)width, (int)height, (int)samples, d_pixels,
                                                             (int)stride, components, static_cast<cudaStream_t>(stream)));
}

int rt_gpu_resolve_counts_device(f32 const *d_accum, i32 const *d_samples, isize width, isize height, u8 *d_pixels,
                                 isize stride, i32 components, void *stream) {
  if (!d_samples || components < 3) return fail("resolve_counts: d_samples and components >= 3 required");
  return launched("resolve", rt_launch_resolve_counts(d_accum, d_samples, (int)width, (int)height, d_pixels, (int)stride,
                                                      components, static_cast<cudaStream_t>(stream)));
}

int rt_gpu_resolve_device(f32 const *d_accum, isize width, isize height, isize samples, u8 *d_pixels, isize stride,
                          i32 components, void *stream) {
  if (samples < 1 || components < 3) return fail("resolve: samples >= 1 and components >= 3 required");
  return launched("resolve", rt_launch_resolve(d_accum, (int)width, (int)height, (int)samples, d_pixels, (int)stride, components,
                                               static_cast<cudaStream_t>(stream)));
}

int rt_gpu_denoise_device(u8 const *d_src, u8 *d_dst, isize width, isize height, isize src_stride, isize dst_stride,
                          i32 components, void *stream) {
  if (d_src == d_dst) return fail("denoise: src and dst must differ (reference denoiser.c:130)");
  return launched("denoise", rt_launch_denoise(d_src, d_dst, (int)width, (int)height, (int)src_stride, (int)dst_stride,
                                               components, static_cast<cudaStream_t>(stream)));
}

// ------------------------------------------------------------------ ray queries
}  // extern "C"

namespace {

// ---- the checks the validations are made of, in each validation's order; every message starts with the call's name
int check_rays(const char *what, isize n_rays) {
  if (n_rays < 0 || n_rays > INT32_MAX) return fail("%s: n_rays = %lld, must be in [0, INT32_MAX]", what, (long long)n_rays);
  return 0;
}

int check_bounces(const char *what, isize max_bounces) {
  if (max_bounces < 0 || max_bounces > INT32_MAX) return fail("%s: max_bounces = %lld, must be >= 0", what, (long long)max_bounces);
  return 0;
}

int check_given(const char *what, const void *p, const char *name) {
  if (!p) return fail("%s: null %s", what, name);
  return 0;
}

// the tail of the cast_rays, AOV and refit validations: afterwards the scene is resident (and current) on every device
int scene_resident(const char *what, const Scene *scene) {
  if (check_given(what, scene, "scene")) return 1;
  if (ensure_init()) return 1;
  if (g.devs[0].scenes.find(scene) == g.devs[0].scenes.end())
    return fail("%s: scene is not resident (rt_gpu_scene_upload it first)", what);
  return scene_on_devices(scene);
}

// A part of a host-memory call's staging: `bytes` on the device (0: none, NULL), filled from the host's `in` before the
// device step and copied to the host's `out` after it (either may be NULL).
struct HostPart { size_t bytes; const void *in; void *out; };

// The host-memory form of a call (queries, cast_rays, AOV), after its validation: the parts are staged in the first
// device's staging block, each 16-byte aligned; the inputs go up on d.stream, `step` enqueues the device form there
// with the parts' device pointers, the outputs come back in part order and the call synchronises.  The calls share the
// block: each runs on d.stream under g_mutex and synchronises before it returns, and grow() frees the old block
// through cudaFree, which waits for the device.
template <int N, class Step>
int host_call(const HostPart (&parts)[N], Step step) {
  Device &d = g.devs[0];
  CUDA_TRY(cudaSetDevice(d.id));
  size_t offset[N], total = 0;
  for (int i = 0; i < N; i++) { offset[i] = total; total += (parts[i].bytes + 15) & ~(size_t)15; }
  if (grow(&d.d_stage, &d.stage_bytes, total)) return 1;
  void *dev[N];
  for (int i = 0; i < N; i++) dev[i] = parts[i].bytes ? static_cast<char *>(d.d_stage) + offset[i] : nullptr;
  for (int i = 0; i < N; i++)
    if (parts[i].bytes && parts[i].in)
      CUDA_TRY(cudaMemcpyAsync(dev[i], parts[i].in, parts[i].bytes, cudaMemcpyHostToDevice, d.stream));
  if (step(dev, d.stream)) return 1;
  for (int i = 0; i < N; i++)
    if (parts[i].bytes && parts[i].out)
      CUDA_TRY(cudaMemcpyAsync(parts[i].out, dev[i], parts[i].bytes, cudaMemcpyDeviceToHost, d.stream));
  CUDA_TRY(cudaStreamSynchronize(d.stream));
  return 0;
}

// Everything that is refused before a query; afterwards the scene is resident (and current) on every device: unlike
// the other calls, a query uploads a scene that is not.
int query_validate(const char *what, const Scene *scene, const void *rays, isize n_rays, const void *out, const void *hits) {
  if (check_rays(what, n_rays)) return 1;
  if (n_rays == 0) return 0;
  if (check_given(what, scene, "scene")) return 1;
  if (check_given(what, rays, "rays")) return 1;
  if (check_given(what, out, "output")) return 1;
  if (reinterpret_cast<uintptr_t>(hits) & 15) return fail("%s: hits must be 16-byte aligned", what);
  if (ensure_init()) return 1;
  return scene_on_devices(scene);
}

// One query launch on the first device, ordered on `stream`.  It reads the scene's geometry only, so it waits for
// geom_ready and not for the texels; it touches neither the render workspace nor the camera-relative copies, so it
// does not wait for renders.  Queries of one device share its work counter: each waits for the previous one.
int query_on_device(const Scene *scene, const Ray *rays, const f32 *t_max, isize n_rays, bool any, RT_GPU_Hit *hits,
                    RT_GPU_Surface *surface, u8 *occluded, u64 *counters, cudaStream_t stream) {
  Device &d = g.devs[0];
  DeviceScene *ds = first_device_scene(scene);
  if (!ds) return 1;
  if (!d.d_query_fetch) CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d.d_query_fetch), sizeof(unsigned)));
  if (!d.query_busy) CUDA_TRY(cudaEventCreateWithFlags(&d.query_busy, cudaEventDisableTiming));
  CUDA_TRY(cudaStreamWaitEvent(stream, ds->geom_ready, 0));
  if (d.query_busy_valid) CUDA_TRY(cudaStreamWaitEvent(stream, d.query_busy, 0));
  CUDA_TRY(cudaMemsetAsync(d.d_query_fetch, 0, sizeof(unsigned), stream));
  QueryParams p{};
  p.scene = ds->dev;
  p.rays = reinterpret_cast<const float *>(rays);
  p.t_max = t_max;
  p.n_rays = (unsigned)n_rays;
  p.hits = reinterpret_cast<float4 *>(hits);
  p.surface = reinterpret_cast<float *>(surface);
  p.occluded = occluded;
  p.fetch = d.d_query_fetch;
  p.counters = reinterpret_cast<unsigned long long *>(counters);
  if (launched("query", rt_launch_query(p, any, d.sm_count, stream))) return 1;
  CUDA_TRY(cudaEventRecord(d.query_busy, stream));
  d.query_busy_valid = true;
  return 0;
}

int query_device_call(const char *what, const Scene *scene, const Ray *d_rays, const f32 *d_t_max, isize n_rays, bool any,
                      RT_GPU_Hit *d_hits, RT_GPU_Surface *d_surface, u8 *d_occluded, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (query_validate(what, scene, d_rays, n_rays, any ? static_cast<const void *>(d_occluded) : d_hits, d_hits)) return 1;
  if (n_rays == 0) return 0;
  return query_on_device(scene, d_rays, d_t_max, n_rays, any, d_hits, d_surface, d_occluded, d_counters,
                         static_cast<cudaStream_t>(stream));
}

// Host memory: rays (and t_max) up, query, results back.
int query_host_call(const char *what, const Scene *scene, const Ray *rays, const f32 *t_max, isize n_rays, bool any,
                    RT_GPU_Hit *hits, RT_GPU_Surface *surface, u8 *occluded) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  // host arrays need no alignment: the device copy of hits is a staging part
  if (query_validate(what, scene, rays, n_rays, any ? static_cast<const void *>(occluded) : hits, nullptr)) return 1;
  if (n_rays == 0) return 0;
  const size_t n = (size_t)n_rays;
  return host_call({HostPart{any ? 0 : n * sizeof(RT_GPU_Hit), nullptr, hits},
                    {surface && !any ? n * sizeof(RT_GPU_Surface) : 0, nullptr, surface},
                    {n * sizeof(Ray), rays, nullptr},
                    {t_max ? n * sizeof(f32) : 0, t_max, nullptr},
                    {any ? n : 0, nullptr, occluded}},
                   [&](void **part, cudaStream_t stream) {
                     return query_on_device(scene, static_cast<Ray *>(part[2]), static_cast<f32 *>(part[3]), n_rays, any,
                                            static_cast<RT_GPU_Hit *>(part[0]), static_cast<RT_GPU_Surface *>(part[1]),
                                            static_cast<u8 *>(part[4]), nullptr, stream);
                   });
}

}  // namespace

extern "C" {

int rt_gpu_closest_hit_device(Scene const *scene, Ray const *d_rays, f32 const *d_t_max, isize n_rays, RT_GPU_Hit *d_hits,
                              RT_GPU_Surface *d_surface, u64 *d_counters, void *stream) {
  return query_device_call("closest_hit", scene, d_rays, d_t_max, n_rays, false, d_hits, d_surface, nullptr, d_counters, stream);
}

int rt_gpu_occluded_device(Scene const *scene, Ray const *d_rays, f32 const *d_t_max, isize n_rays, u8 *d_occluded,
                           u64 *d_counters, void *stream) {
  return query_device_call("occluded", scene, d_rays, d_t_max, n_rays, true, nullptr, nullptr, d_occluded, d_counters, stream);
}

int rt_gpu_closest_hit(Scene const *scene, Ray const *rays, f32 const *t_max, isize n_rays, RT_GPU_Hit *hits,
                       RT_GPU_Surface *surface) {
  return query_host_call("closest_hit", scene, rays, t_max, n_rays, false, hits, surface, nullptr);
}

int rt_gpu_occluded(Scene const *scene, Ray const *rays, f32 const *t_max, isize n_rays, u8 *occluded) {
  return query_host_call("occluded", scene, rays, t_max, n_rays, true, nullptr, nullptr, occluded);
}

// ------------------------------------------------------------- radiance for caller rays
}  // extern "C"

namespace {

// Everything that is refused before a launch; afterwards the scene is resident (and current) on the first device.
int cast_rays_validate(const char *what, const Scene *scene, const void *rays, isize n_rays, isize sample_begin,
                       isize samples, isize max_bounces, const void *radiance) {
  if (check_rays(what, n_rays)) return 1;
  if (samples < 0 || sample_begin < 0 || sample_begin > INT32_MAX - samples)
    return fail("%s: samples [%lld, %lld + %lld) must lie in [0, INT32_MAX]", what, (long long)sample_begin,
                (long long)sample_begin, (long long)samples);
  if (check_bounces(what, max_bounces)) return 1;
  if (n_rays == 0) return 0;
  if (check_given(what, rays, "rays")) return 1;
  if (check_given(what, radiance, "radiance")) return 1;
  return scene_resident(what, scene);
}

// One cast_rays call on the first device, ordered on `stream`: a workspace user that shades, so it waits for the
// scene's texels as well as its geometry.
int cast_rays_on_device(const Scene *scene, const Ray *rays, const u32 *keys, isize n_rays, isize sample_begin, isize samples,
                        isize max_bounces, u32 user_seed, int accumulate, float *radiance, float *per_sample,
                        unsigned long long *counters, cudaStream_t stream) {
  Device &d = g.devs[0];
  DeviceScene *ds = first_device_scene(scene);
  if (!ds) return 1;
  const size_t n_paths = (size_t)n_rays * (size_t)samples;
  WorkspaceRequest r;
  if (n_paths > 0)
    r = {rt_cast_rays_workspace_bytes(n_paths, (int)max_bounces, false), rt_cast_rays_workspace_bytes(n_paths, (int)max_bounces, true)};
  if (workspace_begin(d, *ds, r, true, stream)) return 1;
  int e = rt_launch_cast_rays(ds->dev, reinterpret_cast<const float *>(rays), keys, (int)n_rays, (int)sample_begin,
                              (int)samples, (int)max_bounces, user_seed, accumulate, radiance, per_sample, counters,
                              d.sm_count, d.d_workspace, d.workspace_bytes, stream, &g.last_launches);
  return workspace_end(d, "cast_rays", e, stream);
}

}  // namespace

extern "C" {

int rt_gpu_cast_rays_device(Scene const *scene, Ray const *d_rays, u32 const *d_keys, isize n_rays, isize sample_begin,
                            isize samples, isize max_bounces, u32 user_seed, i32 accumulate, f32 *d_radiance,
                            f32 *d_per_sample, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (cast_rays_validate("cast_rays", scene, d_rays, n_rays, sample_begin, samples, max_bounces, d_radiance)) return 1;
  if (n_rays == 0) return 0;
  return cast_rays_on_device(scene, d_rays, d_keys, n_rays, sample_begin, samples, max_bounces, user_seed, accumulate,
                             d_radiance, d_per_sample, reinterpret_cast<unsigned long long *>(d_counters),
                             static_cast<cudaStream_t>(stream));
}

// Host memory: rays, keys (and the sums to continue from) up, cast, results back.
int rt_gpu_cast_rays(Scene const *scene, Ray const *rays, u32 const *keys, isize n_rays, isize sample_begin, isize samples,
                     isize max_bounces, u32 user_seed, i32 accumulate, f32 *radiance, f32 *per_sample) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  if (cast_rays_validate("cast_rays", scene, rays, n_rays, sample_begin, samples, max_bounces, radiance)) return 1;
  if (n_rays == 0) return 0;
  const size_t n = (size_t)n_rays;
  return host_call({HostPart{n * 3 * sizeof(float), accumulate ? radiance : nullptr, radiance},
                    {per_sample ? n * (size_t)samples * 3 * sizeof(float) : 0, nullptr, per_sample},
                    {n * sizeof(Ray), rays, nullptr},
                    {keys ? n * sizeof(u32) : 0, keys, nullptr}},
                   [&](void **part, cudaStream_t stream) {
                     return cast_rays_on_device(scene, static_cast<Ray *>(part[2]), static_cast<u32 *>(part[3]), n_rays,
                                                sample_begin, samples, max_bounces, user_seed, accumulate,
                                                static_cast<float *>(part[0]), static_cast<float *>(part[1]), nullptr, stream);
                   });
}

// ------------------------------------------------------------- first-surface AOVs
}  // extern "C"

namespace {

// Everything that is refused before a launch of a whole-image camera call (AOV, masked render) writing into `out`;
// afterwards the scene is resident on the first device with the camera the Scene holds now (scene_on_devices
// refreshes it, as for a render).
int camera_validate(const char *what, const Scene *scene, isize width, isize height, isize sample_begin, isize sample_end,
                    isize max_bounces, const void *out, const char *out_name) {
  if (width < 1 || height < 1) return fail("%s: image %lld x %lld is empty", what, (long long)width, (long long)height);
  // one sample of every pixel must fit one chunk of 32-bit path ids
  if (width > INT32_MAX || height > INT32_MAX ||
      (size_t)((width + 7) / 8) * (size_t)((height + 3) / 4) * 32 > ((size_t)1 << 31))
    return fail("%s: image %lld x %lld is too large", what, (long long)width, (long long)height);
  if (sample_begin < 0 || sample_end < sample_begin || sample_end > INT32_MAX)
    return fail("%s: samples [%lld, %lld) must be a range inside [0, INT32_MAX]", what, (long long)sample_begin,
                (long long)sample_end);
  if (check_bounces(what, max_bounces)) return 1;
  if (check_given(what, out, out_name)) return 1;
  return scene_resident(what, scene);
}

// One AOV call on the first device, ordered on `stream`: a workspace user that rewrites the camera-relative copies as
// a render does, and reads texels, so it waits for the scene's texels as well as its geometry.
int aov_on_device(const Scene *scene, isize width, isize height, isize sample_begin, isize sample_end, isize max_bounces,
                  int accumulate, float *aov, unsigned long long *counters, cudaStream_t stream) {
  Device &d = g.devs[0];
  DeviceScene *ds = first_device_scene(scene);
  if (!ds) return 1;
  const isize n_samples = sample_end - sample_begin;
  if (workspace_begin(d, *ds, n_samples > 0 && max_bounces > 0 ? camera_workspace(width, height, n_samples, max_bounces, 1)
                                                               : WorkspaceRequest{}, true, stream))
    return 1;
  int e = rt_launch_aov(ds->dev, (int)width, (int)height, (int)sample_begin, (int)sample_end, (int)max_bounces, accumulate,
                        aov, counters, d.sm_count, d.d_workspace, d.workspace_bytes, stream, &g.last_launches);
  return workspace_end(d, "aov", e, stream);
}

}  // namespace

extern "C" {

int rt_gpu_render_aov_device(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                             isize max_bounces, i32 accumulate, RT_GPU_AOV *d_aov, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (camera_validate("render_aov", scene, width, height, sample_begin, sample_end, max_bounces, d_aov, "aov")) return 1;
  if (reinterpret_cast<uintptr_t>(d_aov) & 15) return fail("render_aov: d_aov is not 16-byte aligned");
  return aov_on_device(scene, width, height, sample_begin, sample_end, max_bounces, accumulate,
                       reinterpret_cast<float *>(d_aov), reinterpret_cast<unsigned long long *>(d_counters),
                       static_cast<cudaStream_t>(stream));
}

// Host memory: the records are computed from zero in a staging part and come back.
int rt_gpu_render_aov(Scene const *scene, isize width, isize height, isize sample_begin, isize sample_end,
                      isize max_bounces, RT_GPU_AOV *aov) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  if (camera_validate("render_aov", scene, width, height, sample_begin, sample_end, max_bounces, aov, "aov")) return 1;
  return host_call({HostPart{(size_t)width * (size_t)height * sizeof(RT_GPU_AOV), nullptr, aov}},
                   [&](void **part, cudaStream_t stream) {
                     return aov_on_device(scene, width, height, sample_begin, sample_end, max_bounces, 0,
                                          static_cast<float *>(part[0]), nullptr, stream);
                   });
}

// ------------------------------------------------------------- masked sample passes
// The renderer itself (render_on_device, whole image, first device) with its primary trace and accumulate swapped for
// their masked builds: the launch sequence, chunking, fast_math and the deferred texel wait are a render's.
int rt_gpu_render_masked_device(Scene const *scene, isize width, isize height, u8 const *d_mask, isize sample_begin,
                                isize sample_end, isize max_bounces, u32 user_seed, i32 accumulate, f32 *d_accum,
                                f32 *d_accum_sq, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (camera_validate("render_masked", scene, width, height, sample_begin, sample_end, max_bounces, d_accum, "accum"))
    return 1;
  const Share share{sample_begin, sample_end, 0, 1};
  return render_on_device(g.devs[0], scene, width, height, share, max_bounces, user_seed, accumulate, d_accum, nullptr,
                          nullptr, reinterpret_cast<unsigned long long *>(d_counters), static_cast<cudaStream_t>(stream),
                          d_mask, d_accum_sq);
}

// ------------------------------------------------------------- many views of a resident scene
}  // extern "C"

namespace {

// Everything that is refused before a launch of a many-view call writing into `out`: camera_validate's refusals, a
// negative view count, NULL cameras for a non-empty call.  The cameras themselves are not checked: a render accepts any.
int views_validate(const char *what, const Scene *scene, i32 n_views, const Camera *cameras, isize width, isize height,
                   isize sample_begin, isize sample_end, isize max_bounces, const void *out, const char *out_name) {
  if (n_views < 0) return fail("%s: n_views = %d, must be >= 0", what, (int)n_views);
  if (camera_validate(what, scene, width, height, sample_begin, sample_end, max_bounces, out, out_name)) return 1;
  if (n_views > 0) return check_given(what, cameras, "cameras");
  return 0;
}

// One many-view call on the first device, ordered on `stream`: the renderer with a camera and a seed per view, each view
// into its W*H*3 slice of d_accum.  The cameras go to the launcher as copies; the resident scene's camera is not touched.
int views_on_device(const Scene *scene, i32 n_views, const Camera *cameras, const u32 *seeds, isize width, isize height,
                    isize sample_begin, isize sample_end, isize max_bounces, int accumulate, float *d_accum,
                    unsigned long long *d_counters, cudaStream_t stream) {
  std::vector<ViewCamera> views((size_t)n_views);
  for (int v = 0; v < n_views; v++) {
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) views[(size_t)v].view[r][c] = cameras[v].view_matrix.rows[r][c];
    views[(size_t)v].focal_length = cameras[v].focal_length;
  }
  const Views vs{(int)n_views, views.data(), seeds};
  const Share share{sample_begin, sample_end, 0, 1};
  return render_on_device(g.devs[0], scene, width, height, share, max_bounces, 0, accumulate, d_accum, nullptr, nullptr,
                          d_counters, stream, nullptr, nullptr, &vs);
}

}  // namespace

extern "C" {

int rt_gpu_render_views_device(Scene const *scene, i32 n_views, Camera const *cameras, u32 const *user_seeds, isize width,
                               isize height, isize sample_begin, isize sample_end, isize max_bounces, i32 accumulate,
                               f32 *d_accum, u64 *d_counters, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (views_validate("render_views", scene, n_views, cameras, width, height, sample_begin, sample_end, max_bounces,
                     d_accum, "accum"))
    return 1;
  if (n_views == 0) return 0;
  return views_on_device(scene, n_views, cameras, user_seeds, width, height, sample_begin, sample_end, max_bounces,
                         accumulate, d_accum, reinterpret_cast<unsigned long long *>(d_counters),
                         static_cast<cudaStream_t>(stream));
}

// Host memory: the sums are computed from zero in a staging part; each view's image is the film of its slice.
int rt_gpu_render_views(Scene const *scene, i32 n_views, Camera const *cameras, u32 const *user_seeds, isize width,
                        isize height, isize sample_begin, isize sample_end, isize max_bounces, f32 *accum, u8 *pixels) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  if (views_validate("render_views", scene, n_views, cameras, width, height, sample_begin, sample_end, max_bounces,
                     accum ? static_cast<const void *>(accum) : pixels, "accum and pixels"))
    return 1;
  if (n_views == 0) return 0;
  const size_t image = (size_t)width * (size_t)height * 3, n = (size_t)n_views * image;
  const isize samples = sample_end - sample_begin;
  return host_call({HostPart{n * sizeof(float), nullptr, accum}, {pixels ? n : 0, nullptr, pixels}},
                   [&](void **part, cudaStream_t stream) {
                     float *d_accum = static_cast<float *>(part[0]);
                     u8 *d_pixels = static_cast<u8 *>(part[1]);
                     if (views_on_device(scene, n_views, cameras, user_seeds, width, height, sample_begin, sample_end,
                                         max_bounces, 0, d_accum, nullptr, stream))
                       return 1;
                     if (!pixels) return 0;
                     if (samples < 1) {            // no samples: black images
                       CUDA_TRY(cudaMemsetAsync(d_pixels, 0, n, stream));
                       return 0;
                     }
                     for (size_t v = 0; v < (size_t)n_views; v++)
                       if (launched("resolve", rt_launch_resolve(d_accum + v * image, (int)width, (int)height, (int)samples,
                                                                 d_pixels + v * image, (int)width, 3, stream)))
                         return 1;
                     return 0;
                   });
}

// ------------------------------------------------------------------ moving geometry (rt_scene.cu: scene_refit)
int rt_gpu_scene_refit_device(Scene const *scene, f32 const *d_positions, f32 const *d_normals, void *stream) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (scene_resident("scene_refit", scene)) return 1;
  if (check_given("scene_refit", d_positions, "positions")) return 1;
  return scene_refit(scene, d_positions, d_normals, 9, static_cast<cudaStream_t>(stream));
}

int rt_gpu_scene_refit(Scene *scene, i32 refit_normals) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (scene_resident("scene_refit", scene)) return 1;
  if (!scene->triangles.x[0] || !scene->triangles.aos) return fail("scene_refit: null positions");
  return scene_refit_host(scene, refit_normals != 0);
}

int rt_gpu_read_nodes(Scene const *scene, BVH_Node *out) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (scene_resident("read_nodes", scene)) return 1;
  if (check_given("read_nodes", out, "output")) return 1;
  return scene_read_nodes(scene, out);
}

// ----------------------------------------------------------------- parity hooks
int rt_gpu_read_accum(f32 *out, isize n_floats) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g.devs.empty() || !g.devs[0].d_accum || (size_t)n_floats > g.last_pixels * 3) return fail("read_accum: no render of that size has run");
  CUDA_TRY(cudaSetDevice(g.devs[0].id));
  CUDA_TRY(cudaMemcpy(out, g.devs[0].d_accum, (size_t)n_floats * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int rt_gpu_read_hit_ids(i32 *out, isize n_pixels) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g.devs.empty() || !g.devs[0].d_hit_ids || !g.last_has_hit_ids || (size_t)n_pixels > g.last_pixels)
    return fail("read_hit_ids: the last render did not keep hit ids (RT_GPU_Options.keep_hit_ids)");
  CUDA_TRY(cudaSetDevice(g.devs[0].id));
  CUDA_TRY(cudaMemcpy(out, g.devs[0].d_hit_ids, (size_t)n_pixels * sizeof(int), cudaMemcpyDeviceToHost));
  if (g.last_split_mode == RT_GPU_SPLIT_CHUNKS && g.devs.size() > 1) {
    // chunk split: every device recorded the pixels of its own chunks, INT_MIN elsewhere
    std::vector<int> other((size_t)n_pixels);
    for (size_t k = 1; k < g.devs.size(); k++) {
      CUDA_TRY(cudaSetDevice(g.devs[k].id));
      CUDA_TRY(cudaMemcpy(other.data(), g.devs[k].d_hit_ids, (size_t)n_pixels * sizeof(int), cudaMemcpyDeviceToHost));
      for (isize i = 0; i < n_pixels; i++) if (other[(size_t)i] > out[i]) out[i] = other[(size_t)i];
    }
    CUDA_TRY(cudaSetDevice(g.devs[0].id));
  }
  return 0;
}

// texels (RGBA8, tightly packed) of texture `slot` of a resident scene on the first device; slot order = first use by
// the materials in triangle-slot order, the environment last unless a material uses it.  *width / *height are set;
// out may be NULL to query the size, slot beyond the last returns non-zero.
int rt_gpu_read_texture(Scene const *scene, i32 slot, u8 *out, isize *width, isize *height) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g.devs.empty()) return fail("read_texture: not initialised");
  Device &d = g.devs[0];
  auto it = d.scenes.find(scene);
  if (it == d.scenes.end()) return fail("read_texture: scene is not resident");
  CUDA_TRY(cudaSetDevice(d.id));
  CUDA_TRY(cudaStreamSynchronize(d.copy));
  TextureDev table[64];
  const char *tab = reinterpret_cast<const char *>(it->second.dev.textures);
  const int n = it->second.n_textures;
  if (slot < 0 || slot >= n || n > 64) return fail("read_texture: slot %d of %d", slot, n);
  CUDA_TRY(cudaMemcpy(table, tab, (size_t)n * sizeof(TextureDev), cudaMemcpyDeviceToHost));
  if (width) *width = table[slot].width;
  if (height) *height = table[slot].height;
  if (out) CUDA_TRY(cudaMemcpy(out, table[slot].texels, (size_t)table[slot].width * (size_t)table[slot].height * 4, cudaMemcpyDeviceToHost));
  return 0;
}

// the first n_slots slots of every device's counter block, summed
static int read_counters(u64 *out, int n_slots) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (g.devs.empty() || !g.devs[0].d_counters) return fail("read_counters: no render has run");
  for (int i = 0; i < n_slots; i++) out[i] = 0;
  for (Device &d : g.devs) {
    if (!d.d_counters) continue;
    u64 part[16];
    CUDA_TRY(cudaSetDevice(d.id));
    CUDA_TRY(cudaMemcpy(part, d.d_counters, n_slots * sizeof(u64), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n_slots; i++) out[i] += part[i];
  }
  CUDA_TRY(cudaSetDevice(g.devs[0].id));
  return 0;
}

int rt_gpu_read_counters(u64 out[8]) { return read_counters(out, 8); }

// The library's own 16-slot counter block on the first device: [0..8) as RT_GPU_CTR_*, [8] rays whose whole walk
// was the root-union test (they count as one node visit in [1], as in the reference, but cost 18 instructions),
// [9] primary rays.  Pass it as d_counters to the device-level calls to have the extended slots filled.
int rt_gpu_counters_buffer(u64 **d_counters_out) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (ensure_init()) return 1;
  Device &d = g.devs[0];
  CUDA_TRY(cudaSetDevice(d.id));
  if (!d.d_counters) {
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d.d_counters), 16 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(d.d_counters, 0, 16 * sizeof(unsigned long long)));
  }
  *d_counters_out = reinterpret_cast<u64 *>(d.d_counters);
  return 0;
}

int rt_gpu_counters_reset(void) {
  u64 *p = nullptr;
  if (rt_gpu_counters_buffer(&p)) return 1;
  std::lock_guard<std::mutex> lock(g_mutex);
  CUDA_TRY(cudaSetDevice(g.devs[0].id));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemset(p, 0, 16 * sizeof(u64)));
  return 0;
}

int rt_gpu_read_counters_ex(u64 out[16]) { return read_counters(out, 16); }

int rt_gpu_last_launches(void) { return g.last_launches; }

void rt_gpu_stage_profile_enable(i32 on) {
  std::lock_guard<std::mutex> lock(g_mutex);
  rt_stage_profile_enable(on, g.devs.empty() ? 0 : g.devs[0].id);
}

int rt_gpu_stage_profile_read_bounces(f64 ms[64], i64 launches[64]) {
  std::lock_guard<std::mutex> lock(g_mutex);
  long long n[RT_N_STAGES * RT_STAGE_BOUNCES];
  int e = rt_stage_profile_read(ms, n);
  if (e) return fail("stage profile: %s", cudaGetErrorString((cudaError_t)e));
  for (int i = 0; i < RT_N_STAGES * RT_STAGE_BOUNCES; i++) launches[i] = n[i];
  return 0;
}

int rt_gpu_stage_profile_read(f64 ms[4], i64 launches[4]) {
  f64 all_ms[RT_N_STAGES * RT_STAGE_BOUNCES];
  i64 all_n[RT_N_STAGES * RT_STAGE_BOUNCES];
  if (rt_gpu_stage_profile_read_bounces(all_ms, all_n)) return 1;
  for (int s = 0; s < RT_N_STAGES; s++) {
    ms[s] = 0; launches[s] = 0;
    for (int b = 0; b < RT_STAGE_BOUNCES; b++) { ms[s] += all_ms[s * RT_STAGE_BOUNCES + b]; launches[s] += all_n[s * RT_STAGE_BOUNCES + b]; }
  }
  return 0;
}

f64 rt_gpu_last_kernel_ms(void) { return g.last_kernel_ms; }

void rt_gpu_last_frame_breakdown(f64 out[4]) {
  out[0] = g.last_upload_ms; out[1] = g.last_reduce_ms; out[2] = g.last_d2h_ms; out[3] = (f64)g.last_split_mode;
}

// ------------------------------------------------------- reference entry points
static int render_owner(Rendering_Context *ctx, isize n_chunks) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  if (ensure_init()) return 1;
  const Image &im = ctx->image;
  if (im.components < 3 || im.pixel_type != PT_u8 || !im.pixels.data) return fail("render: image must be u8 with >= 3 components");
  if (im.width < 1 || im.height < 1 || im.stride < im.width) return fail("render: empty image or stride < width");
  if (ctx->samples < 1) return fail("render: samples must be >= 1");
  if (!ctx->scene) return fail("render: null scene");
  const size_t n_dev = g.devs.size();
  if (n_dev > 1 && enable_peers()) return 1;
  const size_t n_pixels = (size_t)im.width * (size_t)im.height;
  const size_t image_bytes = (size_t)im.stride * (size_t)im.height * (size_t)im.components;
  const RT_GPU_Options opt = g.options;

  double t0 = now_ms();
  bool was_resident = true;
  for (Device &d : g.devs) was_resident &= d.scenes.find(ctx->scene) != d.scenes.end();
  if (scene_on_devices(ctx->scene)) return 1;
  g.last_upload_ms = was_resident ? 0.0 : now_ms() - t0;

  for (Device &d : g.devs)
    if (ensure_frame_buffers(d, n_pixels, opt.keep_hit_ids != 0)) return 1;
  Device &d0 = g.devs[0];
  CUDA_TRY(cudaSetDevice(d0.id));
  if (image_buffers(d0, image_bytes)) return 1;

  // the samples this call renders (a multi-process host narrows them per rank), then their split over the devices
  isize s_begin = opt.sample_begin, s_end = opt.sample_end;
  if (!opt.sample_range_set && s_end <= 0) s_end = ctx->samples;
  if (s_begin < 0) s_begin = 0;
  if (s_end > ctx->samples) s_end = ctx->samples;
  if (s_end < s_begin) s_end = s_begin;
  const i32 mode = n_dev > 1 ? rt_gpu_shard_mode((i32)(s_end - s_begin), (i32)n_dev, opt.split_mode) : RT_GPU_SPLIT_SAMPLES;

  // samples per progress slice: as asked, or as many as one wavefront chunk holds (fewer, larger chunks are faster)
  isize slice = opt.slice_samples;
  if (slice <= 0) {
    const int world = n_dev > 1 && mode == RT_GPU_SPLIT_CHUNKS ? (int)n_dev : (opt.pixel_world > 1 ? opt.pixel_world : 1);
    slice = (isize)rt_render_chunk_samples((int)im.width, (int)im.height, world);
    if (slice < 1) slice = 1;
  }
  g.last_pixels = n_pixels;
  g.last_has_hit_ids = opt.keep_hit_ids != 0;
  g.last_split_mode = mode;
  // rows padded by stride keep whatever the caller had there
  if ((im.stride != im.width || im.components != 3) && image_to_device(d0, im.pixels.data, image_bytes)) return 1;

  CUDA_TRY(cudaEventRecord(d0.ev0, d0.stream));
  std::vector<Share> shares(n_dev);
  isize max_slices = 0;
  for (size_t k = 0; k < n_dev; k++) {
    Share &sh = shares[k];
    sh = Share{s_begin, s_end, opt.pixel_rank, opt.pixel_world};
    if (n_dev > 1) {
      if (mode == RT_GPU_SPLIT_SAMPLES) {
        i32 a = 0, b = 0;
        rt_gpu_shard_samples((i32)k, (i32)n_dev, (i32)(s_end - s_begin), &a, &b);
        sh.s_begin = s_begin + a; sh.s_end = s_begin + b;
      } else {
        sh.split_rank = (int)k; sh.split_world = (int)n_dev;
      }
    }
    const isize n_slices = (sh.s_end - sh.s_begin + slice - 1) / slice;
    if (n_slices > max_slices) max_slices = n_slices;
  }
  // Path-queue workspaces first, for every device, before anything is launched: with peer access enabled a
  // cudaMalloc maps the new block into every peer and waits for whatever those peers are running.
  for (size_t k = 0; k < n_dev; k++) {
    Device &d = g.devs[k];
    const Share &sh = shares[k];
    const isize n = sh.s_end - sh.s_begin < slice ? sh.s_end - sh.s_begin : slice;
    if (n <= 0) continue;
    CUDA_TRY(cudaSetDevice(d.id));
    if (ensure_workspace(d, camera_workspace(im.width, im.height, n, ctx->max_bounces, sh.split_world), d.stream)) return 1;
  }
  // slices round-robin over the devices, so the host's progress bar (driver.c:810-818) follows all of them
  for (size_t k = 0; k < n_dev; k++) {
    Device &d = g.devs[k];
    CUDA_TRY(cudaSetDevice(d.id));
    CUDA_TRY(cudaMemsetAsync(d.d_counters, 0, 16 * sizeof(unsigned long long), d.stream));
    if (opt.keep_hit_ids && shares[k].split_world > 1)
      CUDA_TRY(cudaMemsetAsync(d.d_hit_ids, 0x80, n_pixels * sizeof(int), d.stream));      // 0x80808080 < -1: "not mine"
    if (shares[k].s_end <= shares[k].s_begin) {
      // an empty share still defines its accumulator: zero
      const Share empty{shares[k].s_begin, shares[k].s_begin, shares[k].split_rank, shares[k].split_world};
      if (render_on_device(d, ctx->scene, im.width, im.height, empty, ctx->max_bounces, opt.user_seed, 0, d.d_accum,
                           nullptr, nullptr, d.d_counters, d.stream))
        return 1;
    }
  }
  for (isize j = 0; j < max_slices; j++) {
    for (size_t k = 0; k < n_dev; k++) {
      const Share &sh = shares[k];
      const isize a = sh.s_begin + j * slice;
      if (a >= sh.s_end) continue;
      const Share part{a, a + slice < sh.s_end ? a + slice : sh.s_end, sh.split_rank, sh.split_world};
      Device &d = g.devs[k];
      const bool first = j == 0;
      if (render_on_device(d, ctx->scene, im.width, im.height, part, ctx->max_bounces, opt.user_seed, first ? 0 : 1, d.d_accum,
                           nullptr, (opt.keep_hit_ids && first && (k == 0 || sh.split_world > 1)) ? d.d_hit_ids : nullptr,
                           d.d_counters, d.stream))
        return 1;
    }
    if (max_slices > 1 && (j % 4 == 3)) {
      // progress for the host's bar; never reaches n_chunks early
      for (Device &d : g.devs) { CUDA_TRY(cudaSetDevice(d.id)); CUDA_TRY(cudaStreamSynchronize(d.stream)); }
      isize progress = n_chunks * (j + 1) / max_slices;
      if (progress >= n_chunks) progress = n_chunks - 1;
      if (progress > ctx->_current_chunk) ctx->_current_chunk = (i32)progress;
    }
  }
  CUDA_TRY(cudaSetDevice(d0.id));
  CUDA_TRY(cudaEventRecord(d0.ev1, d0.stream));

  // ---- film: combine the devices' accumulators on the first one and resolve (raytracer.c:700-716)
  cudaEvent_t r0 = nullptr, r1 = nullptr;
  if (n_dev > 1) {
    for (size_t k = 1; k < n_dev; k++) {
      CUDA_TRY(cudaSetDevice(g.devs[k].id));
      CUDA_TRY(cudaEventRecord(g.devs[k].done, g.devs[k].stream));
    }
    CUDA_TRY(cudaSetDevice(d0.id));
    CUDA_TRY(cudaEventCreate(&r0));
    CUDA_TRY(cudaEventCreate(&r1));
    for (size_t k = 1; k < n_dev; k++) CUDA_TRY(cudaStreamWaitEvent(d0.stream, g.devs[k].done, 0));
    CUDA_TRY(cudaEventRecord(r0, d0.stream));
  }
  if (n_dev > 1 && opt.reduce_mode == RT_GPU_REDUCE_NCCL) {
    if (nccl_reduce_to_first(n_pixels * 3)) return 1;
    CUDA_TRY(cudaSetDevice(d0.id));
    if (launched("resolve", rt_launch_resolve(d0.d_accum, (int)im.width, (int)im.height, (int)ctx->samples, d0.d_image,
                                              (int)im.stride, im.components, d0.stream)))
      return 1;
  } else {
    ReduceParts parts{};
    parts.n = (int)n_dev;
    for (size_t k = 0; k < n_dev; k++) parts.part[k] = g.devs[k].d_accum;
    // one device: the same kernel with a single part (x + nothing) — one film code path for every N
    if (launched("reduce+resolve", rt_launch_reduce_resolve(parts, n_dev > 1 ? d0.d_accum : nullptr, (int)im.width,
                                                            (int)im.height, (int)ctx->samples, d0.d_image, (int)im.stride,
                                                            im.components, d0.stream)))
      return 1;
  }
  if (r1) CUDA_TRY(cudaEventRecord(r1, d0.stream));
  if (image_to_pinned(d0, d0.d_image, image_bytes)) return 1;
  t0 = now_ms();
  memcpy(im.pixels.data, d0.h_pinned, image_bytes);
  g.last_d2h_ms = now_ms() - t0;
  // peers keep their accumulators untouched until the reduce has read them: it has, the stream is drained
  for (size_t k = 1; k < n_dev; k++) {
    CUDA_TRY(cudaSetDevice(g.devs[k].id));
    CUDA_TRY(cudaStreamSynchronize(g.devs[k].stream));
  }
  CUDA_TRY(cudaSetDevice(d0.id));
  float ms = 0;
  cudaEventElapsedTime(&ms, d0.ev0, d0.ev1);
  g.last_kernel_ms = ms;
  g.last_reduce_ms = 0;
  if (r0 && r1) {
    cudaEventElapsedTime(&ms, r0, r1);
    g.last_reduce_ms = ms;
    cudaEventDestroy(r0);
    cudaEventDestroy(r1);
  }
  cudaError_t late = cudaGetLastError();
  if (late != cudaSuccess) return fail("render: %s", cudaGetErrorString(late));
  return 0;
}

void render_thread_proc(Rendering_Context *ctx) {
  const isize chunks_x = (ctx->image.width + RT_CHUNK_SIZE - 1) / RT_CHUNK_SIZE;
  const isize chunks_y = (ctx->image.height + RT_CHUNK_SIZE - 1) / RT_CHUNK_SIZE;
  const isize n_chunks = chunks_x * chunks_y;
  // raytracer.c:620: claim a chunk; whoever gets chunk 0 launches the whole frame
  i32 c = __atomic_fetch_add(const_cast<i32 *>(&ctx->_current_chunk), 1, __ATOMIC_SEQ_CST);
  if (c == 0) {
    report_status("render_thread_proc", [&] { return render_owner(ctx, n_chunks); });
    __atomic_store_n(const_cast<i32 *>(&ctx->_current_chunk), (i32)n_chunks + 1, __ATOMIC_SEQ_CST);
  }
  // raytracer.c:622
  __atomic_fetch_add(const_cast<i32 *>(&ctx->n_threads), -1, __ATOMIC_SEQ_CST);
}

bool rendering_context_is_finished(Rendering_Context *ctx) {
  return __atomic_load_n(const_cast<i32 *>(&ctx->n_threads), __ATOMIC_SEQ_CST) == 0;
}

void rendering_context_finish(Rendering_Context *ctx) {
  while (__atomic_load_n(const_cast<i32 *>(&ctx->n_threads), __ATOMIC_SEQ_CST) > 0) sched_yield();
}

// raytracer.h:56 / raytracer.c:722-784 on the GPU (first device): the kernels are in rt_render.cu.  values_out
// (optional, W*H*3 f32) receives accumulated / samples of every written texel before the u8 store, owner_out
// (optional, W*H i32) the slot of the triangle that owns each texel (-1 = untouched; such texels keep their bytes).
int rt_gpu_lightmap_bake(Image const *lightmap, Scene const *scene, isize samples, f32 *values_out, i32 *owner_out) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g.last_launches = 0;
  if (ensure_init()) return 1;
  if (!lightmap || !scene) return fail("lightmap_bake: null argument");
  if (lightmap->pixel_type != PT_u8 || lightmap->components < 3 || !lightmap->pixels.data)      // raytracer.c:723-724
    return fail("lightmap_bake: the lightmap must be u8 with >= 3 components");
  if (lightmap->width < 1 || lightmap->height < 1 || lightmap->stride < lightmap->width) return fail("lightmap_bake: empty image or stride < width");
  if (samples < 1) return fail("lightmap_bake: samples must be >= 1");
  if (scene_on_devices(scene)) return 1;
  Device &d = g.devs[0];
  DeviceScene *ds = first_device_scene(scene);
  if (!ds) return 1;
  const int W = (int)lightmap->width, H = (int)lightmap->height;
  const size_t n_texels = (size_t)W * (size_t)H;
  const size_t image_bytes = (size_t)lightmap->stride * (size_t)H * (size_t)lightmap->components;
  const int max_bounces = 8;                                        // raytracer.c:773: cast_ray(scene, r, 8)

  CUDA_TRY(cudaStreamSynchronize(d.stream));
  CUDA_TRY(cudaStreamSynchronize(d.copy));
  if (image_buffers(d, image_bytes)) return 1;
  const size_t scratch_bytes = rt_lightmap_workspace_bytes(W, H) + (values_out ? n_texels * 3 * sizeof(float) : 0) +
                               (owner_out ? n_texels * sizeof(int) : 0);
  if (grow(&d.d_texel_stage, &d.texel_stage_bytes, scratch_bytes)) return 1;       // the upload's raw-texel block doubles as scratch
  char *scratch = static_cast<char *>(d.d_texel_stage);
  float *d_values = values_out ? reinterpret_cast<float *>(scratch + rt_lightmap_workspace_bytes(W, H)) : nullptr;
  int *d_owner = owner_out ? reinterpret_cast<int *>(scratch + rt_lightmap_workspace_bytes(W, H) + (values_out ? n_texels * 3 * sizeof(float) : 0)) : nullptr;
  const WorkspaceRequest r{rt_lightmap_paths_workspace_bytes(n_texels, (int)samples, max_bounces, false),
                           rt_lightmap_paths_workspace_bytes(n_texels, (int)samples, max_bounces, true)};
  if (workspace_begin(d, *ds, r, true, d.stream)) return 1;
  if (image_to_device(d, lightmap->pixels.data, image_bytes)) return 1;      // untouched texels keep their bytes
  if (d_values) CUDA_TRY(cudaMemsetAsync(d_values, 0, n_texels * 3 * sizeof(float), d.stream));
  unsigned n_jobs = 0;
  int e = rt_launch_lightmap(ds->dev, W, H, (int)samples, max_bounces, g.options.user_seed, d.d_image, (int)lightmap->stride,
                             lightmap->components, d_values, d_owner, scratch, d.sm_count, d.d_workspace, d.workspace_bytes,
                             d.stream, &g.last_launches, &n_jobs);
  if (workspace_end(d, "lightmap", e, d.stream)) return 1;
  if (image_from_device(d, d.d_image, image_bytes, lightmap->pixels.data)) return 1;
  if (values_out) CUDA_TRY(cudaMemcpy(values_out, d_values, n_texels * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  if (owner_out) CUDA_TRY(cudaMemcpy(owner_out, d_owner, n_texels * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

void lightmap_bake(Image const *lightmap, Scene const *scene, isize samples) {
  report_status("lightmap_bake", [&] { return rt_gpu_lightmap_bake(lightmap, scene, samples, nullptr, nullptr); });
}

void denoise_image(Image const *src, Image const *dst, isize n_threads) {
  (void)n_threads;
  report_status("denoise_image", [&]() -> int {
    std::lock_guard<std::mutex> lock(g_mutex);
    g.last_launches = 0;
    if (ensure_init()) return 1;
    if (!src->pixels.data || !dst->pixels.data) return fail("denoise: null pixel buffer");
    if (src->pixels.data == dst->pixels.data) return fail("denoise: src and dst must differ (reference denoiser.c:130)");
    if (src->width != dst->width || src->height != dst->height || src->components != dst->components)
      return fail("denoise: src and dst shapes differ (reference denoiser.c:131-132)");
    Device &d = g.devs[0];
    CUDA_TRY(cudaSetDevice(d.id));
    const size_t src_bytes = (size_t)src->stride * (size_t)src->height * (size_t)src->components;
    const size_t dst_bytes = (size_t)dst->stride * (size_t)dst->height * (size_t)dst->components;
    CUDA_TRY(cudaStreamSynchronize(d.stream));
    if (grow(reinterpret_cast<void **>(&d.d_image), &d.image_bytes, src_bytes)) return 1;
    if (grow(reinterpret_cast<void **>(&d.d_image2), &d.image2_bytes, dst_bytes)) return 1;
    if (grow_pinned(d, src_bytes > dst_bytes ? src_bytes : dst_bytes)) return 1;
    if (image_to_device(d, src->pixels.data, src_bytes)) return 1;
    if (dst->stride != dst->width) CUDA_TRY(cudaMemsetAsync(d.d_image2, 0, dst_bytes, d.stream));
    CUDA_TRY(cudaEventRecord(d.ev0, d.stream));
    if (launched("denoise", rt_launch_denoise(d.d_image, d.d_image2, (int)src->width, (int)src->height, (int)src->stride,
                                              (int)dst->stride, src->components, d.stream)))
      return 1;
    CUDA_TRY(cudaEventRecord(d.ev1, d.stream));
    if (dst->stride == dst->width) {
      if (image_from_device(d, d.d_image2, dst_bytes, dst->pixels.data)) return 1;
    } else {
      if (image_to_pinned(d, d.d_image2, dst_bytes)) return 1;
      for (isize y = 0; y < dst->height; y++)
        memcpy(dst->pixels.data + (size_t)y * (size_t)dst->stride * (size_t)dst->components,
               d.h_pinned + (size_t)y * (size_t)dst->stride * (size_t)dst->components,
               (size_t)dst->width * (size_t)dst->components);
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, d.ev0, d.ev1);
    g.last_kernel_ms = ms;
    return 0;
  });
}

}  // extern "C"
