"""Host-side mirror of the reference's driver.c flow (driver.c:730-878) on top of the C ABI.

    load background -> default camera -> load_model_file -> scene_init
    -> Rendering_Context + render_thread_proc -> (denoise_image) -> save

Everything that computes is native: librt_host.so (C: loaders, BVH build, codecs) and
libraytracer_gpu.so (sm_100a kernels).  This module only wires pointers together, so the
parity tests can drive the same entry points a C host would.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _ffi
from ._ffi import (Camera, GPUOptions, Image, Model, RenderingContext, Scene, Vec3, gpu_check, gpu_lib, host_lib)

# driver.c:733-742
DEFAULT_WIDTH, DEFAULT_HEIGHT, DEFAULT_SAMPLES, DEFAULT_BOUNCES, DEFAULT_THREADS = 1024, 1024, 16, 8, 1
BACKGROUND_SIZE = (2048, 1024)


def fn_address(fn) -> int:
    return C.cast(fn, C.c_void_p).value


@dataclass
class LoadedScene:
    """Owns the host buffers a Scene points into (model, textures, environment image)."""
    model: Model
    scene: Scene
    background: Image
    shader_proc: int
    background_proc: int
    path: str
    n_triangles: int
    foreign_builder: bool = False      # scene buffers came from a test's builder (plain aligned_alloc), not scene_init
    _closed: bool = field(default=False)

    def close(self) -> None:
        if self._closed:
            return
        self._closed = True
        if _ffi._gpu is not None:
            gpu_lib().rt_gpu_scene_release(C.byref(self.scene))
        host = host_lib()
        if self.foreign_builder:
            libc = C.CDLL(None)
            libc.free.argtypes = [C.c_void_p]
            libc.free(self.scene.bvh.nodes.data)
            libc.free(self.scene.triangles.x[0])
        else:
            host.scene_destroy(C.byref(self.scene))
        host.rt_model_free(C.byref(self.model))
        host.rt_image_free(C.byref(self.background))


def use_pinned_host_buffers(on: bool = True) -> None:
    """Texels, BVH nodes, the triangle block and images loaded from now on live in pinned memory
    (rt_gpu_host_alloc), so rt_gpu_scene_upload DMA-reads them in place instead of staging them."""
    if on:
        gpu = gpu_lib()
        host_lib().rt_host_set_buffer_allocator(fn_address(gpu.rt_gpu_host_alloc), fn_address(gpu.rt_gpu_host_free))
    else:
        host_lib().rt_host_set_buffer_allocator(None, None)


def defer_jpeg_decode(on: bool = True) -> None:
    """Models loaded from now on keep their JPEG textures compressed; rt_gpu_scene_upload decodes them on the device
    (nvJPEG).  Such scenes can only be rendered by the GPU library."""
    host_lib().rt_host_defer_jpeg_decode(bool(on))


def read_texture(loaded: "LoadedScene", slot: int) -> np.ndarray:
    """RGBA8 texels of texture `slot` as resident on the first device."""
    w, h = _ffi.isize(), _ffi.isize()
    gpu_check(gpu_lib().rt_gpu_read_texture(C.byref(loaded.scene), slot, None, C.byref(w), C.byref(h)))
    out = np.zeros((h.value, w.value, 4), dtype=np.uint8)
    gpu_check(gpu_lib().rt_gpu_read_texture(C.byref(loaded.scene), slot, out.ctypes.data, C.byref(w), C.byref(h)))
    return out


def look_at(eye, target, up=(0.0, 1.0, 0.0), fov_degrees: float = 70.0) -> Camera:
    cam = Camera()
    host_lib().rt_camera_look_at(C.byref(cam), Vec3(*eye), Vec3(*target), Vec3(*up),
                                 C.c_float(np.deg2rad(fov_degrees)))
    return cam


def load_scene(path: str, shader_proc: Optional[int] = None, background_proc: Optional[int] = None,
               background_path: Optional[str] = None, camera: Optional[Camera] = None,
               builder=None) -> LoadedScene:
    """driver.c:756-775.  `shader_proc`/`background_proc` default to the GPU library's own
    identities; tests pass the oracle's CPU callbacks so ONE Scene feeds both sides.
    `builder` replaces scene_init (tests use the oracle's builder to compare layouts)."""
    host = host_lib()
    if shader_proc is None or background_proc is None:
        gpu = gpu_lib()
        shader_proc = shader_proc or fn_address(gpu.rt_gpu_pbr_shader_proc)
        background_proc = background_proc or fn_address(gpu.rt_gpu_background_proc)

    background = Image()
    if background_path:
        if not host.rt_load_texture(background_path.encode(), C.byref(background)):
            raise RuntimeError(f"Failed to load texture: '{background_path}': {host.rt_host_last_error().decode()}")
    else:
        host.rt_generate_background(C.byref(background), *BACKGROUND_SIZE)

    scene = Scene()
    host.rt_camera_default(C.byref(scene.camera))
    model = Model()
    if not host.rt_load_model_file(path.encode(), shader_proc, C.byref(model), C.byref(scene.camera)):
        host.rt_image_free(C.byref(background))
        raise RuntimeError(f"Failed to load model '{path}': {host.rt_host_last_error().decode()}")
    if camera is not None:
        scene.camera = camera
    scene.background.proc = background_proc
    loaded = LoadedScene(model=model, scene=scene, background=background, shader_proc=shader_proc,
                         background_proc=background_proc, path=path, n_triangles=model.triangles.len,
                         foreign_builder=builder is not None)
    loaded.scene.background.data = C.addressof(loaded.background)
    (builder or host.scene_init)(C.byref(loaded.scene), model.triangles)
    return loaded


def register_callbacks(loaded: LoadedScene) -> None:
    gpu = gpu_lib()
    gpu.rt_gpu_register_pbr_shader(loaded.shader_proc)
    gpu.rt_gpu_register_background(loaded.background_proc)


def image_view(pixels: np.ndarray) -> Image:
    """Image header over a contiguous (H, W, C) uint8 array (driver.c:747-754)."""
    assert pixels.dtype == np.uint8 and pixels.ndim == 3 and pixels.flags["C_CONTIGUOUS"]
    im = Image()
    im.pixels.data = pixels.ctypes.data
    im.pixels.len = pixels.size
    im.height, im.width, im.components = pixels.shape
    im.stride = im.width
    im.pixel_type = 0
    return im


def set_options(user_seed: int = 0, sample_begin: int = 0, sample_end: int = 0, slice_samples: int = 0,
                keep_hit_ids: bool = False, sample_range_set: bool = False, split_mode: int = 0, reduce_mode: int = 0,
                pixel_rank: int = 0, pixel_world: int = 0, fast_math: bool = False) -> None:
    opt = GPUOptions(user_seed, sample_begin, sample_end, slice_samples, int(keep_hit_ids), int(sample_range_set),
                     split_mode, reduce_mode, pixel_rank, pixel_world, int(fast_math))
    gpu_lib().rt_gpu_set_options(C.byref(opt))


def init_devices(n: int, devices=None) -> None:
    """rt_gpu_init_devices: this process drives `n` GPUs (the host program's --gpus N)."""
    ids = (C.c_int * n)(*devices) if devices is not None else None
    gpu_check(gpu_lib().rt_gpu_init_devices(n, ids))


def render(loaded: LoadedScene, width: int = DEFAULT_WIDTH, height: int = DEFAULT_HEIGHT,
           samples: int = DEFAULT_SAMPLES, max_bounces: int = DEFAULT_BOUNCES,
           n_threads: int = DEFAULT_THREADS, out: Optional[np.ndarray] = None) -> np.ndarray:
    """driver.c:793-819 through the reference's own entry points with HOST buffers:
    n_threads OS threads all enter render_thread_proc with one context, the caller polls
    rendering_context_is_finished."""
    gpu = gpu_lib()
    register_callbacks(loaded)
    pixels = out if out is not None else np.zeros((height, width, 3), dtype=np.uint8)
    ctx = RenderingContext()
    ctx.image = image_view(pixels)
    ctx.scene = C.pointer(loaded.scene)
    ctx.samples, ctx.max_bounces = samples, max_bounces
    ctx.n_threads, ctx._current_chunk = n_threads, 0
    threads = [threading.Thread(target=gpu.render_thread_proc, args=(C.byref(ctx),)) for _ in range(n_threads)]
    for t in threads:
        t.start()
    gpu.rendering_context_finish(C.byref(ctx))
    for t in threads:
        t.join()
    if not gpu.rendering_context_is_finished(C.byref(ctx)):
        raise RuntimeError("render did not finish")
    if gpu.rt_gpu_last_status() != 0:         # the entry points return void (raytracer.h:51-56)
        raise RuntimeError("libraytracer_gpu: " + gpu.rt_gpu_last_error().decode())
    return pixels


def denoise(src: np.ndarray, n_threads: int = 1) -> np.ndarray:
    """driver.c:827-837 through denoise_image (host buffers)."""
    gpu = gpu_lib()
    src = np.ascontiguousarray(src)
    dst = np.zeros_like(src)
    a, b = image_view(src), image_view(dst)
    gpu.denoise_image(C.byref(a), C.byref(b), n_threads)
    if gpu.rt_gpu_last_status() != 0:
        raise RuntimeError("libraytracer_gpu: " + gpu.rt_gpu_last_error().decode())
    return dst


def lightmap_bake(loaded: LoadedScene, width: int, height: int, samples: int, out: Optional[np.ndarray] = None,
                  want_values: bool = False):
    """raytracer.h's lightmap_bake (reference raytracer.c:722-784) on the GPU.  Returns the u8 lightmap, or — with
    want_values — a dict with the f32 values before the u8 store and the owning triangle slot per texel."""
    gpu = gpu_lib()
    register_callbacks(loaded)
    pixels = out if out is not None else np.zeros((height, width, 3), dtype=np.uint8)
    im = image_view(pixels)
    if not want_values:
        gpu.lightmap_bake(C.byref(im), C.byref(loaded.scene), samples)
        if gpu.rt_gpu_last_status() != 0:
            raise RuntimeError("libraytracer_gpu: " + gpu.rt_gpu_last_error().decode())
        return pixels
    values = np.zeros((height, width, 3), dtype=np.float32)
    owner = np.full((height, width), -1, dtype=np.int32)
    gpu_check(gpu.rt_gpu_lightmap_bake(C.byref(im), C.byref(loaded.scene), samples, values.ctypes.data, owner.ctypes.data))
    return dict(pixels=pixels, values=values, owner=owner)


def _query_rays(origins, directions, t_max):
    """(n, 6) float32 rays (the C Ray: position, direction) and the optional (n,) float32 t_max, both contiguous."""
    o = np.asarray(origins, dtype=np.float32).reshape(-1, 3)
    d = np.asarray(directions, dtype=np.float32).reshape(-1, 3)
    if o.shape != d.shape:
        raise ValueError(f"origins {o.shape} and directions {d.shape} differ")
    rays = np.ascontiguousarray(np.concatenate([o, d], axis=1))
    if t_max is not None:
        t_max = np.ascontiguousarray(np.broadcast_to(np.asarray(t_max, dtype=np.float32), (len(rays),)))
    return rays, t_max


def closest_hit(loaded: LoadedScene, origins, directions, t_max=None, surface: bool = False) -> dict:
    """Closest hit of each ray (rt_gpu_closest_hit; semantics in include/rt_gpu.h): the reference's ray_scene_hit with
    hit.distance = t_max (None = +inf; a scalar applies to every ray).  Returns t, u, v (float32) and slot (int32,
    -1 = miss); with surface, also point, normal (interpolated, not normalised), normal_geo (n, 3) and tex_coords (n, 2)."""
    register_callbacks(loaded)
    rays, t_max = _query_rays(origins, directions, t_max)
    n = len(rays)
    hits = np.zeros(n, dtype=[("t", np.float32), ("u", np.float32), ("v", np.float32), ("slot", np.int32)])
    surf = np.zeros((n, 11), dtype=np.float32) if surface else None
    gpu_check(gpu_lib().rt_gpu_closest_hit(C.byref(loaded.scene), rays.ctypes.data,
                                           t_max.ctypes.data if t_max is not None else None, n, hits.ctypes.data,
                                           surf.ctypes.data if surf is not None else None))
    out = {k: np.ascontiguousarray(hits[k]) for k in ("t", "u", "v", "slot")}
    if surf is not None:
        out.update(point=surf[:, 0:3], normal=surf[:, 3:6], normal_geo=surf[:, 6:9], tex_coords=surf[:, 9:11])
    return out


def occluded(loaded: LoadedScene, origins, directions, t_max=None) -> np.ndarray:
    """Whether any triangle lies along each ray before t_max (rt_gpu_occluded): exactly closest_hit(...)["slot"] >= 0
    for the same rays and t_max, with a walk that stops at the first accepted triangle."""
    register_callbacks(loaded)
    rays, t_max = _query_rays(origins, directions, t_max)
    out = np.zeros(len(rays), dtype=np.uint8)
    gpu_check(gpu_lib().rt_gpu_occluded(C.byref(loaded.scene), rays.ctypes.data,
                                        t_max.ctypes.data if t_max is not None else None, len(rays), out.ctypes.data))
    return out.astype(bool)


def cast_rays(loaded: LoadedScene, origins, directions, samples: int, max_bounces: int = 8, sample_begin: int = 0,
              user_seed: int = 0, keys=None, per_sample: bool = False):
    """Path-traced radiance along each ray (rt_gpu_cast_rays; semantics in include/rt_gpu.h): the reference's cast_ray
    for samples [sample_begin, sample_begin + samples), the shader generator of path (i, s) seeded to
    rt_path_seed(keys[i] (default i), s, user_seed).  Directions are used as given.  Uploads the scene if it is not
    resident.  Returns the (n, 3) float32 sums over the samples (not divided); with per_sample, also the
    (n, samples, 3) radiance of every path, as (radiance, per_sample)."""
    gpu = gpu_lib()
    register_callbacks(loaded)
    rays, _ = _query_rays(origins, directions, None)
    n = len(rays)
    if keys is not None:
        keys = np.ascontiguousarray(np.asarray(keys, dtype=np.uint32).reshape(-1))
        if len(keys) != n:
            raise ValueError(f"{len(keys)} keys for {n} rays")
    if gpu.rt_gpu_scene_device_bytes(C.byref(loaded.scene)) == 0:
        gpu_check(gpu.rt_gpu_scene_upload(C.byref(loaded.scene)))
    radiance = np.zeros((n, 3), dtype=np.float32)
    per = np.zeros((n, samples, 3), dtype=np.float32) if per_sample else None
    gpu_check(gpu.rt_gpu_cast_rays(C.byref(loaded.scene), rays.ctypes.data, keys.ctypes.data if keys is not None else None,
                                   n, sample_begin, samples, max_bounces, user_seed, 0, radiance.ctypes.data,
                                   per.ctypes.data if per is not None else None))
    return (radiance, per) if per_sample else radiance


def render_aov(loaded: LoadedScene, width: int, height: int, samples: int, max_bounces: int = 8,
               sample_begin: int = 0) -> dict:
    """First-surface AOVs of the renderer's camera samples [sample_begin, sample_begin + samples) (rt_gpu_render_aov;
    semantics in include/rt_gpu.h): per pixel, the sums over the samples of albedo, shading normal, position and
    emission ((H, W, 3) float32) and of coverage, depth, roughness and metalness ((H, W) float32), at the first front
    face each sample's path shades.  The sums are not divided: divide by coverage for the mean over the covered samples.
    Uploads the scene if it is not resident."""
    gpu = gpu_lib()
    register_callbacks(loaded)
    if gpu.rt_gpu_scene_device_bytes(C.byref(loaded.scene)) == 0:
        gpu_check(gpu.rt_gpu_scene_upload(C.byref(loaded.scene)))
    floats = C.sizeof(_ffi.GPUAOV) // 4
    records = np.zeros((height, width, floats), dtype=np.float32)
    gpu_check(gpu.rt_gpu_render_aov(C.byref(loaded.scene), width, height, sample_begin, sample_begin + samples,
                                    max_bounces, records.ctypes.data))
    out = {}
    for name, ctype in _ffi.GPUAOV._fields_:
        first = getattr(_ffi.GPUAOV, name).offset // 4
        out[name] = records[:, :, first:first + 3].copy() if ctype is Vec3 else records[:, :, first].copy()
    return out


def render_masked(loaded: LoadedScene, accum, sample_begin: int, sample_end: int, mask=None, accum_sq=None,
                  max_bounces: int = 8, user_seed: int = 0, accumulate: bool = False, counters=None, stream=None) -> None:
    """Samples [sample_begin, sample_end) of the pixels `mask` selects (rt_gpu_render_masked_device; semantics in
    include/rt_gpu.h), enqueued on `stream` (default: torch's current stream).  `accum` and `accum_sq` (optional) are
    contiguous (H, W, 3) float32 CUDA tensors: the sums and the per-channel sums of squares in sample order, continued
    with `accumulate`.  `mask` is an (H, W) bool or uint8 CUDA tensor (None = every pixel); `counters` an optional
    8-element int64 CUDA tensor the work counters are added to.  Uploads the scene if it is not resident."""
    import torch
    gpu = gpu_lib()
    height, width = accum.shape[0], accum.shape[1]

    def check(t, shape, dtypes, what):
        if t.device.type != "cuda" or t.dtype not in dtypes or tuple(t.shape) != shape or not t.is_contiguous():
            raise ValueError(f"{what}: a contiguous CUDA tensor of shape {shape} and dtype {dtypes[0]} is required")
    check(accum, (height, width, 3), (torch.float32,), "accum")
    if accum_sq is not None:
        check(accum_sq, (height, width, 3), (torch.float32,), "accum_sq")
    if mask is not None:
        check(mask, (height, width), (torch.uint8, torch.bool), "mask")
    if counters is not None:
        check(counters, (8,), (torch.int64,), "counters")
    register_callbacks(loaded)
    if gpu.rt_gpu_scene_device_bytes(C.byref(loaded.scene)) == 0:
        gpu_check(gpu.rt_gpu_scene_upload(C.byref(loaded.scene)))
    st = stream or torch.cuda.current_stream()
    gpu_check(gpu.rt_gpu_render_masked_device(
        C.byref(loaded.scene), width, height, mask.data_ptr() if mask is not None else None, sample_begin, sample_end,
        max_bounces, user_seed, int(accumulate), accum.data_ptr(), accum_sq.data_ptr() if accum_sq is not None else None,
        counters.data_ptr() if counters is not None else None, st.cuda_stream))


def resolve_counts(accum, samples, stream=None):
    """The film with a sample count per pixel (rt_gpu_resolve_counts_device): `accum` an (H, W, 3) float32 and `samples`
    an (H, W) int32 CUDA tensor; returns the (H, W, 3) uint8 CUDA image, enqueued on `stream` (default: torch's current
    stream).  A count <= 0 gives black."""
    import torch
    height, width = accum.shape[0], accum.shape[1]
    if accum.dtype != torch.float32 or tuple(accum.shape) != (height, width, 3) or not accum.is_contiguous() \
            or accum.device.type != "cuda":
        raise ValueError("accum: a contiguous (H, W, 3) float32 CUDA tensor is required")
    if samples.dtype != torch.int32 or tuple(samples.shape) != (height, width) or not samples.is_contiguous() \
            or samples.device != accum.device:
        raise ValueError("samples: a contiguous (H, W) int32 tensor on the device of accum is required")
    pixels = torch.empty((height, width, 3), dtype=torch.uint8, device=accum.device)
    st = stream or torch.cuda.current_stream()
    gpu_check(gpu_lib().rt_gpu_resolve_counts_device(accum.data_ptr(), samples.data_ptr(), width, height,
                                                     pixels.data_ptr(), width, 3, st.cuda_stream))
    return pixels


def read_accum(width: int, height: int) -> np.ndarray:
    out = np.empty((height, width, 3), dtype=np.float32)
    gpu_check(gpu_lib().rt_gpu_read_accum(out.ctypes.data, out.size))
    return out


def read_hit_ids(width: int, height: int) -> np.ndarray:
    out = np.empty((height, width), dtype=np.int32)
    gpu_check(gpu_lib().rt_gpu_read_hit_ids(out.ctypes.data, out.size))
    return out


def read_counters() -> dict:
    out = np.zeros(8, dtype=np.uint64)
    gpu_check(gpu_lib().rt_gpu_read_counters(out.ctypes.data))
    names = ["rays", "nodes", "leaves", "accepts", "shades", "misses", "passthrough", "samples"]
    return {k: int(v) for k, v in zip(names, out)}


def save_image(path: str, pixels: np.ndarray) -> None:
    im = image_view(np.ascontiguousarray(pixels))
    if not host_lib().rt_save_image(path.encode(), C.byref(im)):
        raise RuntimeError("Failed to encode output file: " + host_lib().rt_host_last_error().decode())
