// rt_state.h — host-side state of libraytracer_gpu.so, shared by its translation units only
// (rt_cabi.cu: entry points; rt_scene.cu: scene residency and upload; rt_multi.cu: multi-GPU plumbing).
//
// One process drives 1..N CUDA devices (rt_gpu_init / rt_gpu_init_devices).  Everything a device owns —
// streams, events, resident scenes, path-queue workspace, accumulator, staging — lives in its `Device`;
// nothing device-specific is global.  All entry points serialise on g_mutex (host side); work on the
// devices is ordered by streams and events.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <map>
#include <mutex>
#include <vector>

#include "rt_gpu.h"
#include "rt_kernels.h"

namespace rt {

struct Block { void *p; size_t bytes; };

// what identifies the host buffers a resident scene was built from (a host that rebuilds a Scene at the same
// address must not be served the old geometry)
struct Fingerprint {
  const void *nodes = nullptr, *aos = nullptr, *x0 = nullptr, *background = nullptr;
  long n_nodes = 0, n_slots = 0, depth = 0;
  bool operator==(const Fingerprint &o) const {
    return nodes == o.nodes && aos == o.aos && x0 == o.x0 && background == o.background && n_nodes == o.n_nodes &&
           n_slots == o.n_slots && depth == o.depth;
  }
};

struct DeviceScene {
  SceneDev dev{};
  std::vector<Block> blocks;          // every device allocation of this scene, in upload order
  size_t bytes = 0;                   // resident on the device
  size_t h2d_bytes = 0;               // copied host -> device by the upload (0 for a peer fan-out copy)
  size_t p2p_bytes = 0;               // copied device -> device over NVLink by the upload
  cudaEvent_t geom_ready = nullptr;   // nodes, triangles, materials, texture table complete
  cudaEvent_t tex_ready = nullptr;    // texels (incl. the environment) complete
  void  *hot_base = nullptr;          // head of the arena: environment texels, nodes, triangles (persisting-L2 window)
  size_t hot_bytes = 0;
  int    n_textures = 0;
  Fingerprint fp;
};

// pinned staging ring for pageable host sources: the host memcpy of piece k+1 overlaps the DMA of piece k
struct StagingRing {
  static constexpr int kSlots = 4;
  static constexpr size_t kSlotBytes = 8u << 20;
  unsigned char *base = nullptr;
  cudaEvent_t drained[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  int next = 0;
};

struct Device {
  int          id = -1;               // CUDA ordinal
  int          sm_count = 0;
  cudaStream_t stream = nullptr;      // kernels
  cudaStream_t copy = nullptr;        // scene upload (DMA + texel repack)
  cudaEvent_t  ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t  busy = nullptr;        // after the last kernel that touches workspace / camera-relative copies
  cudaEvent_t  done = nullptr;        // this device's share of a multi-device frame
  bool         busy_valid = false;
  std::map<const Scene *, DeviceScene> scenes;
  std::multimap<size_t, void *> block_pool;       // device blocks of released scenes, reused by exact size
  StagingRing  ring;
  float *d_accum = nullptr;   size_t accum_floats = 0;
  int   *d_hit_ids = nullptr; size_t hit_pixels = 0;
  unsigned long long *d_counters = nullptr;
  void  *d_texel_stage = nullptr; size_t texel_stage_bytes = 0;
  void  *d_workspace = nullptr;   size_t workspace_bytes = 0;
  size_t workspace_denied = 0;                    // a request at least this large failed before: do not retry it
  unsigned char *d_image = nullptr, *d_image2 = nullptr; size_t image_bytes = 0, image2_bytes = 0;
  unsigned char *h_pinned = nullptr; size_t pinned_bytes = 0;
  // ray queries (rt_gpu_closest_hit* / rt_gpu_occluded*): the kernel's work counter, the event that serialises queries
  // on this device (they share the counter)
  unsigned *d_query_fetch = nullptr;
  cudaEvent_t query_busy = nullptr;
  bool  query_busy_valid = false;
  // staging of the host-memory queries, rt_gpu_cast_rays and rt_gpu_render_aov (rt_cabi.cu: stage)
  void *d_stage = nullptr; size_t stage_bytes = 0;
  bool l2_window_set = false;
  size_t l2_persist_max = 0, l2_window_max = 0;    // device limits (persistingL2CacheMaxSize, accessPolicyMaxWindowSize)
  cudaStream_t l2_stream = nullptr; const void *l2_base = nullptr;   // where the window was last set
};

struct State {
  bool ready = false;
  std::vector<Device> devs;           // devs[0] owns the image (resolve, denoise, D2H)
  bool peers_enabled = false;
  std::vector<Shader_Proc>     pbr_procs;
  std::vector<Background_Proc> bg_procs;
  RT_GPU_Options options{};
  int    last_launches = 0;
  double last_kernel_ms = 0;
  double last_upload_ms = 0, last_reduce_ms = 0, last_d2h_ms = 0;
  bool   last_has_hit_ids = false;
  size_t last_pixels = 0;
  int    last_split_mode = 0;
};

extern State g;
extern std::mutex g_mutex;

int fail(const char *fmt, ...);
void clear_error();

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) return rt::fail("%s failed: %s", #expr, cudaGetErrorString(e_));    \
  } while (0)

// ---- rt_scene.cu
int grow(void **ptr, size_t *have, size_t want);
int grow_pinned(Device &d, size_t want);
int scene_on_devices(const Scene *scene);                     // resident (and current) on every device of g.devs
int scene_upload_all(const Scene *scene);                     // (re-)upload: device 0 over PCIe, peers over NVLink
void scene_release_all(const Scene *scene);
void release_device(Device &d);                               // everything the device owns (shutdown)
void set_l2_window(Device &d, const DeviceScene &ds, cudaStream_t stream);

// ---- rt_jpeg_gpu.cu
int jpeg_begin_batch(cudaStream_t stream);
int jpeg_decode_device(const unsigned char *bytes, size_t len, int width, int height, unsigned char *d_rgb, cudaStream_t stream);
void jpeg_shutdown();

// ---- rt_multi.cu
int enable_peers();                                           // device 0 <-> every other device
int nccl_prepare();                                           // load libnccl, one communicator per device
int nccl_reduce_to_first(size_t n_floats);                    // d_accum of every device summed into devs[0].d_accum
void nccl_shutdown();
void ipc_close_all();

}  // namespace rt
