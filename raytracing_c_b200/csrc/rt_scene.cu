// rt_scene.cu — scene residency: the host Scene (reference scene.h:84-97) flattened into the device layout of
// rt_device.cuh and kept resident per device, keyed by the Scene pointer.
//
// What happens to the reference's data on the way (driver.c:756-775 builds it, raytracer.c reads it):
//   * BVH nodes go up byte for byte; triangle positions are regrouped per slot with the two edge vectors the
//     reference recomputes per ray (raytracer.c:116-122); Triangle_AOS loses its Shader pointer pair to a material
//     index (materials de-duplicated by Shader.data, textures by Image*); RGB8 texels become RGBA8 on the device.
//   * The upload is a pipeline, not a barrier: geometry first, then texels on the copy stream, each with its own
//     event.  A render waits for `geom_ready` before its primary trace and for `tex_ready` only before the first
//     kernel that samples a texture (rt_render.cu), so the 50+ MB of texels travel while rays are already in flight.
//   * Host sources in pinned memory (rt_gpu_host_alloc) are DMA-read in place; pageable ones pass through a ring of
//     pinned 8 MB slots, the host memcpy of one piece overlapping the DMA of the previous one.
//   * With several devices the scene crosses PCIe once: device 0 takes the upload, its peers copy the finished
//     device blocks (texels already RGBA8) over NVLink with cudaMemcpyPeerAsync.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "rt_state.h"

namespace rt {

// ---------------------------------------------------------------- small allocators
int grow(void **ptr, size_t *have, size_t want) {
  if (*have >= want && *ptr) return 0;
  if (*ptr) cudaFree(*ptr);            // cudaFree synchronises the device: no kernel still reads the old block
  *ptr = nullptr;
  *have = 0;
  CUDA_TRY(cudaMalloc(ptr, want));
  *have = want;
  return 0;
}

int grow_pinned(Device &d, size_t want) {
  if (d.pinned_bytes >= want && d.h_pinned) return 0;
  CUDA_TRY(cudaStreamSynchronize(d.stream));      // an async copy may still use the old buffer
  if (d.h_pinned) cudaFreeHost(d.h_pinned);
  d.h_pinned = nullptr;
  d.pinned_bytes = 0;
  CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&d.h_pinned), want));
  d.pinned_bytes = want;
  return 0;
}

// Device blocks of released scenes are kept and handed out again by exact size: re-uploading a scene (per frame
// in an interactive host, per step in bench.py's end-to-end leg) then costs no cudaMalloc / cudaFree.
static int pool_alloc(Device &d, DeviceScene &ds, size_t bytes, void **out) {
  const size_t alloc = bytes ? bytes : 16;
  auto it = d.block_pool.find(alloc);
  if (it != d.block_pool.end()) {
    *out = it->second;
    d.block_pool.erase(it);
  } else {
    CUDA_TRY(cudaMalloc(out, alloc));
  }
  ds.blocks.push_back({*out, alloc});
  ds.bytes += bytes;
  return 0;
}

static void release_scene(Device &d, DeviceScene &ds) {
  for (Block &b : ds.blocks) d.block_pool.emplace(b.bytes, b.p);
  ds.blocks.clear();
  if (ds.geom_ready) cudaEventDestroy(ds.geom_ready);
  if (ds.tex_ready) cudaEventDestroy(ds.tex_ready);
  ds.geom_ready = ds.tex_ready = nullptr;
}

void release_device(Device &d) {
  cudaSetDevice(d.id);
  cudaDeviceSynchronize();
  for (auto &kv : d.scenes) release_scene(d, kv.second);
  d.scenes.clear();
  for (auto &kv : d.block_pool) cudaFree(kv.second);
  d.block_pool.clear();
  cudaFree(d.d_accum); cudaFree(d.d_hit_ids); cudaFree(d.d_counters); cudaFree(d.d_workspace); cudaFree(d.d_texel_stage);
  cudaFree(d.d_image); cudaFree(d.d_image2); cudaFree(d.d_query_fetch); cudaFree(d.d_stage);
  if (d.h_pinned) cudaFreeHost(d.h_pinned);
  if (d.ring.base) cudaFreeHost(d.ring.base);
  for (cudaEvent_t e : d.ring.drained) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : {d.ev0, d.ev1, d.busy, d.done, d.query_busy}) if (e) cudaEventDestroy(e);
  if (d.stream) cudaStreamDestroy(d.stream);
  if (d.copy) cudaStreamDestroy(d.copy);
  d = Device{};
}

// ---------------------------------------------------------------- host -> device
// Host-side staging copy, split over a few threads above 2 MB: one core copies ~10 GB/s, PCIe 5 takes 50.
static void staged_copy(void *dst, const void *src, size_t n) {
  const size_t kMin = 2u << 20;
  if (n < kMin) { memcpy(dst, src, n); return; }
  const int parts = 4;
  std::thread workers[parts - 1];
  const size_t step = ((n / parts) + 63) & ~(size_t)63;
  for (int i = 1; i < parts; i++) {
    const size_t off = step * i, len = off < n ? (off + step < n && i + 1 < parts ? step : n - off) : 0;
    workers[i - 1] = std::thread([=] { if (len) memcpy(static_cast<char *>(dst) + off, static_cast<const char *>(src) + off, len); });
  }
  memcpy(dst, src, step < n ? step : n);
  for (auto &t : workers) t.join();
}

static bool is_pinned(const void *p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

static int ring_init(Device &d) {
  if (d.ring.base) return 0;
  CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&d.ring.base), StagingRing::kSlots * StagingRing::kSlotBytes));
  for (cudaEvent_t &e : d.ring.drained) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}

// asynchronous on d.copy; returns when the last piece is staged (pageable source) or at once (pinned source)
static int h2d(Device &d, DeviceScene &ds, void *dst, const void *src, size_t n) {
  if (!n) return 0;
  ds.h2d_bytes += n;
  if (is_pinned(src)) {
    CUDA_TRY(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, d.copy));
    return 0;
  }
  if (ring_init(d)) return 1;
  for (size_t off = 0; off < n; off += StagingRing::kSlotBytes) {
    const size_t len = n - off < StagingRing::kSlotBytes ? n - off : StagingRing::kSlotBytes;
    const int slot = d.ring.next;
    d.ring.next = (slot + 1) % StagingRing::kSlots;
    CUDA_TRY(cudaEventSynchronize(d.ring.drained[slot]));        // the DMA that last read this slot
    unsigned char *stage = d.ring.base + (size_t)slot * StagingRing::kSlotBytes;
    staged_copy(stage, static_cast<const char *>(src) + off, len);
    CUDA_TRY(cudaMemcpyAsync(static_cast<char *>(dst) + off, stage, len, cudaMemcpyHostToDevice, d.copy));
    CUDA_TRY(cudaEventRecord(d.ring.drained[slot], d.copy));
  }
  return 0;
}

// ---------------------------------------------------------------- host-side flattening (once per upload)
struct HostScene {
  // geometry goes up from the host's own buffers (in-place DMA when they are pinned); what the host has to compute
  // is one material index per triangle slot — the per-slot regrouping is rt_scene_pack_kernel's job on the device
  const float             *nodes = nullptr;        // scene->bvh.nodes.data, n_internal * 48 floats
  const float             *soa = nullptr;          // nine vertex arrays of n_slots floats, one block
  std::vector<float>       soa_copy;               // only if the host's nine arrays are not one block
  const Triangle_AOS      *aos = nullptr;
  std::vector<int>         mat_index;              // [n_slots]
  std::vector<MaterialDev> materials;
  std::vector<const Image *> images;
  int   env_slot = -1;
  int   depth = 0, n_internal = 0, n_slots = 0;
  float root_lo[3], root_hi[3];
  int   root_upper_empty = 0;             // children 4..7 of the root are padding (lo == hi on every axis)
  Fingerprint fp;
};

static Fingerprint fingerprint(const Scene *scene) {
  Fingerprint f;
  f.nodes = scene->bvh.nodes.data; f.aos = scene->triangles.aos; f.x0 = scene->triangles.x[0];
  f.background = scene->background.data;
  f.n_nodes = (long)scene->bvh.nodes.len; f.n_slots = (long)scene->triangles.len; f.depth = (long)scene->bvh.depth;
  return f;
}

static int flatten(const Scene *scene, HostScene &hs) {
  const isize depth = scene->bvh.depth;
  if (depth < 1 || depth > RT_MAX_DEPTH) return fail("scene: BVH depth %ld outside [1,%d]", (long)depth, RT_MAX_DEPTH);
  const isize n_nodes = scene->bvh.nodes.len, n_slots = scene->triangles.len;
  if (n_nodes != bvh_n_internal_nodes(depth) || n_slots != bvh_n_leaf_nodes(depth) * RT_SIMD_WIDTH)
    return fail("scene: node/slot counts do not describe a complete 8-ary tree of depth %ld", (long)depth);
  if (!scene->bvh.nodes.data || !scene->triangles.aos || !scene->triangles.x[0]) return fail("scene: null node or triangle buffer");
  hs.fp = fingerprint(scene);
  hs.depth = (int)depth; hs.n_internal = (int)n_nodes; hs.n_slots = (int)n_slots;

  hs.nodes = reinterpret_cast<const float *>(scene->bvh.nodes.data);
  hs.aos = scene->triangles.aos;
  // scene_init lays the nine vertex arrays out as one block x0 x1 x2 y0 y1 y2 z0 z1 z2 (scene.h:62-63, scene.c:86-96);
  // a host that assembled them differently gets them gathered into that order
  {
    const float *arrays[9] = { scene->triangles.x[0], scene->triangles.x[1], scene->triangles.x[2],
                               scene->triangles.y[0], scene->triangles.y[1], scene->triangles.y[2],
                               scene->triangles.z[0], scene->triangles.z[1], scene->triangles.z[2] };
    bool one_block = true;
    for (int a = 0; a < 9; a++) one_block &= arrays[a] == arrays[0] + (size_t)a * (size_t)n_slots;
    if (one_block) {
      hs.soa = arrays[0];
    } else {
      hs.soa_copy.resize((size_t)n_slots * 9);
      for (int a = 0; a < 9; a++) {
        if (!arrays[a]) return fail("scene: null vertex array");
        memcpy(hs.soa_copy.data() + (size_t)a * (size_t)n_slots, arrays[a], (size_t)n_slots * sizeof(float));
      }
      hs.soa = hs.soa_copy.data();
    }
  }

  // materials / textures, de-duplicated by host pointer
  std::map<const void *, int> material_index, texture_index;
  auto texture_slot = [&](const Image *im) -> int {
    if (!im) return -1;
    auto it = texture_index.find(im);
    if (it != texture_index.end()) return it->second;
    int slot = (int)hs.images.size();
    hs.images.push_back(im);
    texture_index[im] = slot;
    return slot;
  };

  hs.mat_index.assign((size_t)n_slots, 0);
  const void *last_data = nullptr;
  int last_mat = 0;
  Shader_Proc last_proc = nullptr;
  for (isize s = 0; s < n_slots; s++) {
    const Triangle_AOS &a = scene->triangles.aos[s];
    if (!a.shader.proc && !a.shader.data) continue;
    if (a.shader.proc != last_proc) {
      bool known = false;
      for (Shader_Proc p : g.pbr_procs) known |= (p == a.shader.proc);
      if (!known) return fail("scene: triangle slot %ld uses a Shader_Proc that was not registered with rt_gpu_register_pbr_shader", (long)s);
      last_proc = a.shader.proc;
    }
    if (!a.shader.data) return fail("scene: triangle slot %ld has a registered Shader_Proc but no PBR_Shader_Data", (long)s);
    if (a.shader.data != last_data) {
      auto it = material_index.find(a.shader.data);
      if (it == material_index.end()) {
        const PBR_Shader_Data *m = static_cast<const PBR_Shader_Data *>(a.shader.data);
        MaterialDev d{};
        for (int c = 0; c < 3; c++) { d.base[c] = m->base_color.data[c]; d.emission[c] = m->emission.data[c]; }
        d.roughness = m->roughness; d.metalness = m->metalness; d.normal_strength = m->normal_map_strength;
        d.sheen = m->sheen; d.sheen_tint = m->sheen_tint; d.aniso = m->anisotropic_strength;
        d.tex_albedo = texture_slot(m->texture_albedo);
        d.tex_normal = texture_slot(m->texture_normal);
        d.tex_mr = texture_slot(m->texture_metal_roughness);
        d.tex_emission = texture_slot(m->texture_emission);
        last_mat = (int)hs.materials.size();
        hs.materials.push_back(d);
        material_index[a.shader.data] = last_mat;
      } else {
        last_mat = it->second;
      }
      last_data = a.shader.data;
    }
    hs.mat_index[(size_t)s] = last_mat;
  }
  if (hs.materials.empty()) hs.materials.push_back(MaterialDev{});

  // environment
  bool bg_known = false;
  for (Background_Proc p : g.bg_procs) bg_known |= (p == scene->background.proc);
  if (!bg_known || !scene->background.data)
    return fail("scene: Scene.background.proc was not registered with rt_gpu_register_background (or its Image is null)");
  hs.env_slot = texture_slot(static_cast<const Image *>(scene->background.data));
  for (size_t i = 0; i < hs.images.size(); i++)
    if (hs.images[i]->components < 3 || !hs.images[i]->pixels.data || hs.images[i]->width < 1 || hs.images[i]->height < 1 ||
        (hs.images[i]->pixel_type != PT_u8 && hs.images[i]->pixel_type != PT_RT_JPEG_BYTES))
      return fail("scene: texture %zu needs >= 3 u8 components (or compressed JPEG bytes) and a non-empty pixel buffer", i);

  // union of the root's child boxes; all-zero padding slots (lo == hi) can never be entered (enter >= leave)
  for (int a = 0; a < 3; a++) { hs.root_lo[a] = INFINITY; hs.root_hi[a] = -INFINITY; }
  hs.root_upper_empty = 1;
  for (int j = 0; j < 8; j++) {
    const float *n0 = hs.nodes;
    bool empty = true;
    for (int a = 0; a < 3; a++) empty &= (n0[a * 8 + j] == n0[(3 + a) * 8 + j]);
    if (empty) continue;
    if (j >= 4) hs.root_upper_empty = 0;
    for (int a = 0; a < 3; a++) {
      hs.root_lo[a] = fminf(hs.root_lo[a], n0[a * 8 + j]);
      hs.root_hi[a] = fmaxf(hs.root_hi[a], n0[(3 + a) * 8 + j]);
    }
  }
  return 0;
}

static void fill_common(const HostScene &hs, SceneDev &dev) {
  dev.env_texture = hs.env_slot;
  dev.depth = hs.depth; dev.n_internal = hs.n_internal; dev.n_slots = hs.n_slots;
  for (int a = 0; a < 3; a++) { dev.root_lo[a] = hs.root_lo[a]; dev.root_hi[a] = hs.root_hi[a]; }
  dev.root_upper_empty = hs.root_upper_empty;
  dev.srgb_of_zero = rt_powf_positive((0.0f + 0.055f) / 1.055f, 2.4f);      // rt_math.h: the same bits on host and device
}

static int make_events(DeviceScene &ds) {
  CUDA_TRY(cudaEventCreateWithFlags(&ds.geom_ready, cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&ds.tex_ready, cudaEventDisableTiming));
  return 0;
}

// One arena per scene and device (one cudaMalloc, one persisting-L2 window, two peer copies):
//   [ environment texels | nodes | tri_pos | tri_rec | materials ]  [ texture table ] [ nodes_rel | tri_rel ] [ other texels ]
//   [ environment texels as floats ]     (built on each device by a kernel, not copied: beyond `total`)
// The first bracket is what every ray re-reads; the persisting window (set_l2_window) starts there.
struct ArenaLayout {
  size_t env, nodes, tri_pos, tri_rec, materials, tri_soa, hot_end, table, nodes_rel, tri_rel, texels_begin, total;
  size_t env_f32, alloc_total;       // total = end of what travels host -> device / device -> device
  std::vector<size_t> texel_off;     // per image slot
};

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static ArenaLayout layout_of(const HostScene &hs) {
  ArenaLayout L{};
  L.texel_off.resize(hs.images.size());
  auto texel_bytes = [&](size_t i) { return (size_t)hs.images[i]->width * (size_t)hs.images[i]->height * sizeof(uchar4); };
  size_t off = 0;
  L.env = off;
  if (hs.env_slot >= 0) { L.texel_off[(size_t)hs.env_slot] = off; off = align256(off + texel_bytes((size_t)hs.env_slot)); }
  L.nodes = off;     off = align256(off + (size_t)hs.n_internal * 48 * sizeof(float));
  L.tri_pos = off;   off = align256(off + (size_t)hs.n_slots * 3 * sizeof(float4));
  L.tri_rec = off;   off = align256(off + (size_t)hs.n_slots * 7 * sizeof(float4));
  L.materials = off; off = align256(off + hs.materials.size() * sizeof(MaterialDev));
  L.tri_soa = off;   off = align256(off + (size_t)hs.n_slots * 9 * sizeof(float));
  L.hot_end = off;
  L.table = off;     off = align256(off + hs.images.size() * sizeof(TextureDev) + 16);
  L.nodes_rel = off; off = align256(off + (size_t)hs.n_internal * 48 * sizeof(float));
  L.tri_rel = off;   off = align256(off + (size_t)hs.n_slots * 4 * sizeof(float4));
  L.texels_begin = off;
  for (size_t i = 0; i < hs.images.size(); i++) {
    if ((int)i == hs.env_slot) continue;
    L.texel_off[i] = off;
    off = align256(off + texel_bytes(i));
  }
  L.total = off;
  L.env_f32 = off;
  if (hs.env_slot >= 0) off = align256(off + (size_t)hs.images[(size_t)hs.env_slot]->width * (size_t)hs.images[(size_t)hs.env_slot]->height * sizeof(float4));
  L.alloc_total = off;
  return L;
}

static void bind_arena(char *base, const ArenaLayout &L, const HostScene &hs, DeviceScene &ds, std::vector<TextureDev> &table) {
  ds.dev.nodes     = reinterpret_cast<const float *>(base + L.nodes);
  ds.dev.tri_pos   = reinterpret_cast<const float4 *>(base + L.tri_pos);
  ds.dev.tri_rec   = reinterpret_cast<const float4 *>(base + L.tri_rec);
  ds.dev.materials = reinterpret_cast<const MaterialDev *>(base + L.materials);
  ds.dev.tri_soa   = reinterpret_cast<const float *>(base + L.tri_soa);
  ds.dev.textures  = reinterpret_cast<const TextureDev *>(base + L.table);
  ds.dev.nodes_rel = reinterpret_cast<float *>(base + L.nodes_rel);
  ds.dev.tri_rel   = reinterpret_cast<float4 *>(base + L.tri_rel);
  table.resize(hs.images.size());
  for (size_t i = 0; i < hs.images.size(); i++) {
    table[i].texels = reinterpret_cast<const uchar4 *>(base + L.texel_off[i]);
    table[i].width = (int)hs.images[i]->width;
    table[i].height = (int)hs.images[i]->height;
    table[i].texels_f32 = (int)i == hs.env_slot ? reinterpret_cast<const float4 *>(base + L.env_f32) : nullptr;
  }
  ds.hot_base = base;
  ds.hot_bytes = L.hot_end;
  ds.n_textures = (int)hs.images.size();
}

// device 0: over PCIe from the host buffers
static int upload_primary(Device &d, const HostScene &hs, const ArenaLayout &L, DeviceScene &ds) {
  CUDA_TRY(cudaSetDevice(d.id));
  if (make_events(ds)) return 1;
  ds.fp = hs.fp;
  fill_common(hs, ds.dev);
  void *arena = nullptr;
  if (pool_alloc(d, ds, L.alloc_total, &arena)) return 1;
  char *base = static_cast<char *>(arena);
  std::vector<TextureDev> table;
  bind_arena(base, L, hs, ds, table);
  // raw block = the larger of: every image's raw rows, the Triangle_AOS records + material indices awaiting the pack kernel
  const size_t aos_bytes = (size_t)hs.n_slots * sizeof(Triangle_AOS), idx_bytes = (size_t)hs.n_slots * sizeof(int);
  size_t raw_max = align256(aos_bytes) + idx_bytes;
  for (const Image *im : hs.images) {
    const size_t raw = im->pixel_type == PT_RT_JPEG_BYTES ? (size_t)im->width * (size_t)im->height * 3
                                                          : (size_t)im->stride * (size_t)im->height * (size_t)im->components;
    if (raw > raw_max) raw_max = raw;
  }
  if (raw_max > d.texel_stage_bytes) {
    CUDA_TRY(cudaStreamSynchronize(d.copy));
    if (grow(&d.d_texel_stage, &d.texel_stage_bytes, raw_max)) return 1;
  }
  char *raw_block = static_cast<char *>(d.d_texel_stage);
  if (h2d(d, ds, base + L.nodes, hs.nodes, (size_t)hs.n_internal * 48 * sizeof(float))) return 1;
  if (h2d(d, ds, base + L.tri_soa, hs.soa, (size_t)hs.n_slots * 9 * sizeof(float))) return 1;
  if (h2d(d, ds, raw_block, hs.aos, aos_bytes)) return 1;
  if (h2d(d, ds, raw_block + align256(aos_bytes), hs.mat_index.data(), idx_bytes)) return 1;
  if (h2d(d, ds, base + L.materials, hs.materials.data(), hs.materials.size() * sizeof(MaterialDev))) return 1;
  if (h2d(d, ds, base + L.table, table.data(), table.size() * sizeof(TextureDev))) return 1;
  {
    int e = rt_launch_scene_pack(reinterpret_cast<const float *>(base + L.tri_soa), reinterpret_cast<const float4 *>(raw_block),
                                 reinterpret_cast<const int *>(raw_block + align256(aos_bytes)), hs.n_slots,
                                 reinterpret_cast<float4 *>(base + L.tri_pos), reinterpret_cast<float4 *>(base + L.tri_rec), d.copy);
    if (e) return fail("scene pack launch failed: %s", cudaGetErrorString((cudaError_t)e));
  }
  CUDA_TRY(cudaEventRecord(ds.geom_ready, d.copy));
  // texels: raw rows go up as they are (3 B per texel for RGB8); the RGBA8 layout the samplers read (one 32-bit load
  // per tap) is produced by a kernel on the same stream.  The environment goes first: the miss kernel of bounce 0 is
  // its first consumer.  Two raw staging blocks alternate, so the DMA of one image overlaps the repack of the previous.
  bool any_jpeg = false;
  for (const Image *im : hs.images) any_jpeg |= im->pixel_type == PT_RT_JPEG_BYTES;
  if (any_jpeg && jpeg_begin_batch(d.copy)) return 1;
  std::vector<size_t> order;
  if (hs.env_slot >= 0) order.push_back((size_t)hs.env_slot);
  for (size_t i = 0; i < hs.images.size(); i++) if ((int)i != hs.env_slot) order.push_back(i);
  for (size_t i : order) {
    const Image *im = hs.images[i];
    int e = 0;
    if (im->pixel_type == PT_RT_JPEG_BYTES) {
      // compressed on the host: nvJPEG decodes on the copy stream into the raw block (interleaved RGB), see rt_jpeg_gpu.cu
      ds.h2d_bytes += (size_t)im->pixels.len;
      if (jpeg_decode_device(im->pixels.data, (size_t)im->pixels.len, (int)im->width, (int)im->height,
                             static_cast<unsigned char *>(d.d_texel_stage), d.copy))
        return 1;
      e = rt_launch_texel_repack(static_cast<const unsigned char *>(d.d_texel_stage), (int)im->width, (int)im->height,
                                 (int)im->width, 3, reinterpret_cast<uchar4 *>(base + L.texel_off[i]), d.copy);
    } else {
      const size_t raw = (size_t)im->stride * (size_t)im->height * (size_t)im->components;
      if (h2d(d, ds, d.d_texel_stage, im->pixels.data, raw)) return 1;
      e = rt_launch_texel_repack(static_cast<const unsigned char *>(d.d_texel_stage), (int)im->width, (int)im->height,
                                 (int)im->stride, im->components, reinterpret_cast<uchar4 *>(base + L.texel_off[i]), d.copy);
    }
    if (e) return fail("texel repack launch failed: %s", cudaGetErrorString((cudaError_t)e));
    if ((int)i == hs.env_slot) {
      e = rt_launch_texel_expand(reinterpret_cast<const uchar4 *>(base + L.texel_off[i]), (size_t)im->width * (size_t)im->height,
                                 reinterpret_cast<float4 *>(base + L.env_f32), d.copy);
      if (e) return fail("texel expand launch failed: %s", cudaGetErrorString((cudaError_t)e));
    }
  }
  CUDA_TRY(cudaEventRecord(ds.tex_ready, d.copy));
  return 0;
}

// devices 1..N-1: the finished arena of device 0 (texels already RGBA8), over NVLink
static int upload_peer(Device &d, const Device &src_dev, const DeviceScene &src, const HostScene &hs, const ArenaLayout &L,
                       DeviceScene &ds) {
  CUDA_TRY(cudaSetDevice(d.id));
  if (make_events(ds)) return 1;
  ds.fp = hs.fp;
  fill_common(hs, ds.dev);
  void *arena = nullptr;
  if (pool_alloc(d, ds, L.alloc_total, &arena)) return 1;
  char *base = static_cast<char *>(arena);
  const char *src_base = static_cast<const char *>(src.blocks[0].p);
  std::vector<TextureDev> table;
  bind_arena(base, L, hs, ds, table);
  const size_t env_bytes = L.nodes;      // the environment's texels lead the arena
  CUDA_TRY(cudaStreamWaitEvent(d.copy, src.geom_ready, 0));
  CUDA_TRY(cudaMemcpyPeerAsync(base + L.nodes, d.id, src_base + L.nodes, src_dev.id, L.hot_end - L.nodes, d.copy));
  ds.p2p_bytes += L.hot_end - L.nodes;
  if (h2d(d, ds, base + L.table, table.data(), table.size() * sizeof(TextureDev))) return 1;      // pointers differ per device
  CUDA_TRY(cudaEventRecord(ds.geom_ready, d.copy));
  CUDA_TRY(cudaStreamWaitEvent(d.copy, src.tex_ready, 0));
  if (env_bytes) {
    CUDA_TRY(cudaMemcpyPeerAsync(base, d.id, src_base, src_dev.id, env_bytes, d.copy));
    const Image *env = hs.images[(size_t)hs.env_slot];
    int e = rt_launch_texel_expand(reinterpret_cast<const uchar4 *>(base), (size_t)env->width * (size_t)env->height,
                                   reinterpret_cast<float4 *>(base + L.env_f32), d.copy);
    if (e) return fail("texel expand launch failed: %s", cudaGetErrorString((cudaError_t)e));
  }
  if (L.total > L.texels_begin)
    CUDA_TRY(cudaMemcpyPeerAsync(base + L.texels_begin, d.id, src_base + L.texels_begin, src_dev.id, L.total - L.texels_begin, d.copy));
  ds.p2p_bytes += env_bytes + (L.total - L.texels_begin);
  CUDA_TRY(cudaEventRecord(ds.tex_ready, d.copy));
  return 0;
}

// Scene data is re-read by every kernel of every bounce while gigabytes of path-queue records stream through the
// same 126 MB L2 (round-1 ncu: the miss kernel read 1.31 GB from DRAM for 0.27 GB of records at an L2 hit rate of
// 5.8 % — the 8 MB environment was being evicted by the queue stream).  A persisting access-policy window over the
// head of the arena — environment texels, nodes, triangle records — pins what every ray touches; the queue
// streams around it.
void set_l2_window(Device &d, const DeviceScene &ds, cudaStream_t stream) {
  if (!ds.hot_base || !ds.hot_bytes) return;
  // measured (profiles/r02_summary.md): no effect with the 13 MB head, -7 % with the whole arena — the kernels that read
  // the scene are issue-bound, not waiting for evicted lines.  Off unless RT_GPU_L2_WINDOW=hot|all asks for it.
  static int mode = -1;
  if (mode < 0) { const char *e = getenv("RT_GPU_L2_WINDOW"); mode = !e ? 0 : !strcmp(e, "all") ? 2 : !strcmp(e, "hot") ? 1 : 0; }
  if (mode == 0) return;
  if (!d.l2_persist_max || !d.l2_window_max) return;
  if (d.l2_stream == stream && d.l2_base == ds.hot_base) return;
  size_t want = ds.hot_bytes;
  if (mode == 2 && !ds.blocks.empty()) want = ds.blocks[0].bytes;        // the whole arena (all texels) instead of its head
  if (want > d.l2_window_max) want = d.l2_window_max;
  const size_t carve = want < d.l2_persist_max ? want : d.l2_persist_max;
  if (!d.l2_window_set) { cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve); d.l2_window_set = true; }
  d.l2_stream = stream; d.l2_base = ds.hot_base;
  cudaStreamAttrValue attr{};
  attr.accessPolicyWindow.base_ptr = ds.hot_base;
  attr.accessPolicyWindow.num_bytes = want;
  attr.accessPolicyWindow.hitRatio = want <= carve ? 1.0f : (float)carve / (float)want;
  attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &attr);
  cudaGetLastError();
}

int scene_upload_all(const Scene *scene) {
  HostScene hs;
  if (flatten(scene, hs)) return 1;
  // blocks of an earlier upload of this Scene* are reused below: nothing may still read them
  for (Device &d : g.devs) {
    auto it = d.scenes.find(scene);
    if (it == d.scenes.end()) continue;
    CUDA_TRY(cudaSetDevice(d.id));
    CUDA_TRY(cudaDeviceSynchronize());
    release_scene(d, it->second);
    d.scenes.erase(it);
  }
  const ArenaLayout L = layout_of(hs);
  Device &d0 = g.devs[0];
  DeviceScene first;
  if (upload_primary(d0, hs, L, first)) { release_scene(d0, first); return 1; }
  auto it0 = d0.scenes.emplace(scene, std::move(first)).first;
  for (size_t k = 1; k < g.devs.size(); k++) {
    Device &d = g.devs[k];
    DeviceScene ds;
    if (upload_peer(d, d0, it0->second, hs, L, ds)) { release_scene(d, ds); return 1; }
    d.scenes.emplace(scene, std::move(ds));
  }
  CUDA_TRY(cudaSetDevice(d0.id));
  return 0;
}

int scene_on_devices(const Scene *scene) {
  bool resident = true;
  const Fingerprint now = fingerprint(scene);
  for (Device &d : g.devs) {
    auto it = d.scenes.find(scene);
    resident &= (it != d.scenes.end() && it->second.fp == now);
  }
  if (!resident && scene_upload_all(scene)) return 1;
  for (Device &d : g.devs) {
    SceneDev &dev = d.scenes.find(scene)->second.dev;      // the camera is cheap and may change between frames
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) dev.view[r][c] = scene->camera.view_matrix.rows[r][c];
    dev.focal_length = scene->camera.focal_length;
  }
  return 0;
}

void scene_release_all(const Scene *scene) {
  for (Device &d : g.devs) {
    auto it = d.scenes.find(scene);
    if (it == d.scenes.end()) continue;
    cudaSetDevice(d.id);
    cudaDeviceSynchronize();
    release_scene(d, it->second);
    d.scenes.erase(it);
  }
  if (!g.devs.empty()) cudaSetDevice(g.devs[0].id);
}

}  // namespace rt
