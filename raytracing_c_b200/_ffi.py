"""ctypes view of the C ABI (include/*.h) and loaders for the two in-tree libraries.

The structure definitions mirror include/rt_base.h, scene.h, raytracer.h, rt_pbr.h,
rt_gpu.h and host/rt_host.h field for field.  Loading fails loudly: there is no
Python or CPU fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HOST_LIB = os.path.join(HERE, "host", "librt_host.so")
GPU_LIB = os.environ.get("RT_GPU_LIB", os.path.join(HERE, "csrc", "libraytracer_gpu.so"))   # override: kernel experiments only

isize = C.c_ssize_t


class Vec2(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float)]


class Vec3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class ByteSlice(C.Structure):
    _fields_ = [("data", C.c_void_p), ("len", isize)]


class Image(C.Structure):
    _fields_ = [("pixels", ByteSlice), ("width", isize), ("height", isize), ("stride", isize),
                ("components", C.c_int32), ("pixel_type", C.c_int32)]


class Shader(C.Structure):
    _fields_ = [("data", C.c_void_p), ("proc", C.c_void_p)]


class Triangle(C.Structure):
    _fields_ = [("positions", Vec3 * 3), ("normals", Vec3 * 3), ("tex_coords", Vec2 * 3), ("shader", Shader)]


class TriangleSlice(C.Structure):
    _fields_ = [("data", C.POINTER(Triangle)), ("len", isize)]


class Camera(C.Structure):
    _fields_ = [("view_matrix", (C.c_float * 4) * 4), ("fov", C.c_float), ("focal_length", C.c_float)]


class PBRShaderData(C.Structure):
    _fields_ = [("base_color", Vec3), ("emission", Vec3),
                ("roughness", C.c_float), ("metalness", C.c_float), ("normal_map_strength", C.c_float),
                ("sheen", C.c_float), ("sheen_tint", C.c_float), ("anisotropic_strength", C.c_float),
                ("texture_albedo", C.POINTER(Image)), ("texture_normal", C.POINTER(Image)),
                ("texture_metal_roughness", C.POINTER(Image)), ("texture_emission", C.POINTER(Image))]


class Model(C.Structure):
    _fields_ = [("triangles", TriangleSlice), ("materials", C.POINTER(PBRShaderData)), ("n_materials", isize),
                ("images", C.POINTER(Image)), ("n_images", isize)]


class NodeSlice(C.Structure):
    _fields_ = [("data", C.c_void_p), ("len", isize)]


class BVH(C.Structure):
    _fields_ = [("nodes", NodeSlice), ("depth", isize), ("last_row_offset", isize)]


class Triangles(C.Structure):
    _fields_ = [("x", C.c_void_p * 3), ("y", C.c_void_p * 3), ("z", C.c_void_p * 3),
                ("aos", C.c_void_p), ("len", C.c_int32)]


class Background(C.Structure):
    _fields_ = [("proc", C.c_void_p), ("data", C.c_void_p)]


class Scene(C.Structure):
    _fields_ = [("bvh", BVH), ("camera", Camera), ("triangles", Triangles), ("background", Background)]


class RenderingContext(C.Structure):
    _fields_ = [("image", Image), ("scene", C.POINTER(Scene)), ("samples", isize), ("max_bounces", isize),
                ("n_threads", C.c_int32), ("_current_chunk", C.c_int32)]


class GPUOptions(C.Structure):
    _fields_ = [("user_seed", C.c_uint32), ("sample_begin", C.c_int32), ("sample_end", C.c_int32),
                ("slice_samples", C.c_int32), ("keep_hit_ids", C.c_int32), ("sample_range_set", C.c_int32),
                ("split_mode", C.c_int32), ("reduce_mode", C.c_int32), ("pixel_rank", C.c_int32),
                ("pixel_world", C.c_int32), ("fast_math", C.c_int32)]


class Ray(C.Structure):
    _fields_ = [("position", Vec3), ("direction", Vec3)]


class GPUHit(C.Structure):
    _fields_ = [("t", C.c_float), ("u", C.c_float), ("v", C.c_float), ("slot", C.c_int32)]


class GPUSurface(C.Structure):
    _fields_ = [("point", Vec3), ("normal", Vec3), ("normal_geo", Vec3), ("tex_coords", Vec2)]


class GPUAOV(C.Structure):
    """RT_GPU_AOV: per-pixel sums of the first-surface AOVs (64 B)."""
    _fields_ = [("albedo", Vec3), ("coverage", C.c_float), ("normal", Vec3), ("depth", C.c_float),
                ("position", Vec3), ("roughness", C.c_float), ("emission", Vec3), ("metalness", C.c_float)]


SPLIT_AUTO, SPLIT_SAMPLES, SPLIT_CHUNKS = 0, 1, 2
REDUCE_P2P, REDUCE_NCCL = 0, 1


TRIANGLE_AOS_BYTES = 112
BVH_NODE_BYTES = 192

GPU_EXPORTS = [
    # reference entry points (raytracer.h:51-56, denoiser.h:4)
    "render_thread_proc", "rendering_context_is_finished", "rendering_context_finish", "lightmap_bake",
    "denoise_image",
    # rt_gpu.h
    "rt_gpu_init", "rt_gpu_init_devices", "rt_gpu_device_count", "rt_gpu_visible_devices", "rt_gpu_shutdown",
    "rt_gpu_last_error", "rt_gpu_last_status", "rt_gpu_sm_count", "rt_gpu_measure_fp32_issue",
    "rt_gpu_host_alloc", "rt_gpu_host_free", "rt_gpu_prepare_frame", "rt_gpu_last_frame_breakdown",
    "rt_gpu_shard_samples", "rt_gpu_shard_mode", "rt_gpu_shard_chunks",
    "rt_gpu_render_shard_device", "rt_gpu_accum_buffer", "rt_gpu_ipc_export", "rt_gpu_ipc_open",
    "rt_gpu_reduce_resolve_device", "rt_gpu_lightmap_bake",
    "rt_gpu_scene_device_bytes", "rt_gpu_scene_upload_bytes",
    "rt_gpu_register_pbr_shader", "rt_gpu_register_background", "rt_gpu_pbr_shader_proc", "rt_gpu_background_proc",
    "rt_gpu_scene_upload", "rt_gpu_scene_release", "rt_gpu_set_options", "rt_gpu_get_options",
    "rt_gpu_read_accum", "rt_gpu_read_hit_ids", "rt_gpu_read_counters", "rt_gpu_counters_buffer", "rt_gpu_counters_reset", "rt_gpu_read_texture",
    "rt_gpu_read_counters_ex", "rt_gpu_last_launches",
    "rt_gpu_last_kernel_ms", "rt_gpu_stage_profile_enable", "rt_gpu_stage_profile_read", "rt_gpu_stage_profile_read_bounces",
    "rt_gpu_render_accum_device", "rt_gpu_resolve_device", "rt_gpu_denoise_device",
    "rt_gpu_closest_hit_device", "rt_gpu_occluded_device", "rt_gpu_closest_hit", "rt_gpu_occluded",
    "rt_gpu_cast_rays_device", "rt_gpu_cast_rays",
    "rt_gpu_render_aov_device", "rt_gpu_render_aov",
    "rt_gpu_render_masked_device", "rt_gpu_resolve_counts_device",
]

HOST_EXPORTS = [
    "scene_init", "scene_destroy", "rt_load_model_file", "rt_model_free", "rt_camera_default", "rt_camera_look_at",
    "rt_image_decode", "rt_load_texture", "rt_image_free", "rt_image_alloc", "rt_generate_background",
    "rt_save_image", "rt_save_png", "rt_save_qoi", "rt_save_ppm", "rt_host_last_error",
    "rt_host_set_buffer_allocator", "rt_host_buffer_alloc", "rt_host_buffer_free", "rt_host_defer_jpeg_decode",
    "scene_save_file", "scene_load_file",
]


def build_native(verbose: bool = False) -> None:
    """Compile both libraries in-tree (gcc + nvcc -gencode arch=compute_100a,code=sm_100a)."""
    out = subprocess.run(["make", "-C", HERE, "all"], capture_output=True, text=True)
    if verbose or out.returncode:
        print(out.stdout)
        print(out.stderr)
    if out.returncode:
        raise RuntimeError("building the native libraries failed")


_host = None
_gpu = None


def host_lib() -> C.CDLL:
    global _host
    if _host is None:
        if not os.path.exists(HOST_LIB):
            raise RuntimeError(f"{HOST_LIB} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        lib = C.CDLL(HOST_LIB)
        lib.rt_load_model_file.restype = C.c_bool
        lib.rt_load_model_file.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(Model), C.POINTER(Camera)]
        lib.rt_model_free.argtypes = [C.POINTER(Model)]
        lib.scene_init.argtypes = [C.POINTER(Scene), TriangleSlice]
        lib.scene_destroy.argtypes = [C.POINTER(Scene)]
        lib.rt_camera_default.argtypes = [C.POINTER(Camera)]
        lib.rt_camera_look_at.argtypes = [C.POINTER(Camera), Vec3, Vec3, Vec3, C.c_float]
        lib.rt_image_decode.restype = C.c_bool
        lib.rt_image_decode.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(Image)]
        lib.rt_load_texture.restype = C.c_bool
        lib.rt_load_texture.argtypes = [C.c_char_p, C.POINTER(Image)]
        lib.rt_image_free.argtypes = [C.POINTER(Image)]
        lib.rt_image_alloc.restype = Image
        lib.rt_image_alloc.argtypes = [isize, isize, C.c_int32]
        lib.rt_generate_background.argtypes = [C.POINTER(Image), isize, isize]
        for name in ("rt_save_image", "rt_save_png", "rt_save_qoi", "rt_save_ppm"):
            getattr(lib, name).restype = C.c_bool
            getattr(lib, name).argtypes = [C.c_char_p, C.POINTER(Image)]
        lib.rt_host_last_error.restype = C.c_char_p
        lib.rt_host_set_buffer_allocator.argtypes = [C.c_void_p, C.c_void_p]
        lib.rt_host_set_buffer_allocator.restype = None
        lib.scene_save_file.restype = C.c_bool
        lib.scene_save_file.argtypes = [C.c_char_p, C.POINTER(Scene), C.POINTER(PBRShaderData), isize]
        lib.scene_load_file.restype = C.c_bool
        lib.scene_load_file.argtypes = [C.c_char_p, C.POINTER(Scene), C.POINTER(PBRShaderData), isize, C.c_void_p]
        lib.rt_host_defer_jpeg_decode.argtypes = [C.c_bool]
        lib.rt_host_defer_jpeg_decode.restype = None
        _host = lib
    return _host


def gpu_lib() -> C.CDLL:
    global _gpu
    if _gpu is None:
        if not os.path.exists(GPU_LIB):
            raise RuntimeError(f"{GPU_LIB} is missing: the CUDA extension must be built (no CPU fallback exists)")
        lib = C.CDLL(GPU_LIB)
        lib.rt_gpu_init.argtypes = [C.c_int]
        lib.rt_gpu_init_devices.argtypes = [C.c_int, C.POINTER(C.c_int)]
        lib.rt_gpu_prepare_frame.argtypes = [isize, isize, isize, isize]
        lib.rt_gpu_host_alloc.restype = C.c_void_p
        lib.rt_gpu_host_alloc.argtypes = [C.c_size_t]
        lib.rt_gpu_host_free.argtypes = [C.c_void_p]
        lib.rt_gpu_host_free.restype = None
        lib.rt_gpu_last_frame_breakdown.argtypes = [C.POINTER(C.c_double * 4)]
        lib.rt_gpu_last_frame_breakdown.restype = None
        lib.rt_gpu_shard_samples.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        lib.rt_gpu_shard_samples.restype = None
        lib.rt_gpu_shard_mode.argtypes = [C.c_int32, C.c_int32, C.c_int32]
        lib.rt_gpu_shard_mode.restype = C.c_int32
        lib.rt_gpu_shard_chunks.argtypes = [C.c_int32, C.c_int32, isize, isize]
        lib.rt_gpu_shard_chunks.restype = C.c_int32
        lib.rt_gpu_render_shard_device.argtypes = [C.POINTER(Scene), isize, isize, isize, isize, C.c_uint32, C.c_int32,
                                                   C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p,
                                                   C.c_void_p]
        lib.rt_gpu_lightmap_bake.argtypes = [C.POINTER(Image), C.POINTER(Scene), isize, C.c_void_p, C.c_void_p]
        lib.lightmap_bake.argtypes = [C.POINTER(Image), C.POINTER(Scene), isize]
        lib.lightmap_bake.restype = None
        lib.rt_gpu_accum_buffer.argtypes = [isize, isize, C.POINTER(C.c_void_p)]
        lib.rt_gpu_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
        lib.rt_gpu_ipc_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        lib.rt_gpu_reduce_resolve_device.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, isize, isize, isize,
                                                     C.c_void_p, isize, C.c_int32, C.c_void_p]
        lib.rt_gpu_last_error.restype = C.c_char_p
        lib.rt_gpu_measure_fp32_issue.restype = C.c_double
        lib.rt_gpu_scene_device_bytes.restype = isize
        lib.rt_gpu_scene_device_bytes.argtypes = [C.POINTER(Scene)]
        lib.rt_gpu_scene_upload_bytes.restype = isize
        lib.rt_gpu_scene_upload_bytes.argtypes = [C.POINTER(Scene)]
        lib.rt_gpu_register_pbr_shader.argtypes = [C.c_void_p]
        lib.rt_gpu_register_background.argtypes = [C.c_void_p]
        lib.rt_gpu_scene_upload.argtypes = [C.POINTER(Scene)]
        lib.rt_gpu_scene_release.argtypes = [C.POINTER(Scene)]
        lib.rt_gpu_set_options.argtypes = [C.POINTER(GPUOptions)]
        lib.rt_gpu_get_options.argtypes = [C.POINTER(GPUOptions)]
        lib.rt_gpu_read_accum.argtypes = [C.c_void_p, isize]
        lib.rt_gpu_read_hit_ids.argtypes = [C.c_void_p, isize]
        lib.rt_gpu_read_counters.argtypes = [C.c_void_p]
        lib.rt_gpu_counters_buffer.argtypes = [C.POINTER(C.c_void_p)]
        lib.rt_gpu_read_counters_ex.argtypes = [C.c_void_p]
        lib.rt_gpu_read_texture.argtypes = [C.POINTER(Scene), C.c_int32, C.c_void_p, C.POINTER(isize), C.POINTER(isize)]
        lib.rt_gpu_last_kernel_ms.restype = C.c_double
        lib.rt_gpu_stage_profile_enable.argtypes = [C.c_int32]
        lib.rt_gpu_stage_profile_enable.restype = None
        lib.rt_gpu_stage_profile_read.argtypes = [C.POINTER(C.c_double * 4), C.POINTER(C.c_int64 * 4)]
        lib.rt_gpu_stage_profile_read_bounces.argtypes = [C.POINTER(C.c_double * 64), C.POINTER(C.c_int64 * 64)]
        lib.rt_gpu_render_accum_device.argtypes = [C.POINTER(Scene), isize, isize, isize, isize, isize, C.c_uint32,
                                                   C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_gpu_resolve_device.argtypes = [C.c_void_p, isize, isize, isize, C.c_void_p, isize, C.c_int32, C.c_void_p]
        lib.rt_gpu_denoise_device.argtypes = [C.c_void_p, C.c_void_p, isize, isize, isize, isize, C.c_int32, C.c_void_p]
        lib.rt_gpu_closest_hit_device.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
        lib.rt_gpu_occluded_device.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, C.c_void_p, C.c_void_p,
                                               C.c_void_p]
        lib.rt_gpu_closest_hit.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, C.c_void_p, C.c_void_p]
        lib.rt_gpu_occluded.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, C.c_void_p]
        lib.rt_gpu_cast_rays_device.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, isize, isize, isize,
                                                C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_gpu_cast_rays.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, isize, isize, isize, C.c_uint32,
                                         C.c_int32, C.c_void_p, C.c_void_p]
        lib.rt_gpu_render_aov_device.argtypes = [C.POINTER(Scene), isize, isize, isize, isize, isize, C.c_int32, C.c_void_p,
                                                 C.c_void_p, C.c_void_p]
        lib.rt_gpu_render_aov.argtypes = [C.POINTER(Scene), isize, isize, isize, isize, isize, C.c_void_p]
        lib.rt_gpu_render_masked_device.argtypes = [C.POINTER(Scene), isize, isize, C.c_void_p, isize, isize, isize,
                                                    C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_gpu_resolve_counts_device.argtypes = [C.c_void_p, C.c_void_p, isize, isize, C.c_void_p, isize, C.c_int32,
                                                     C.c_void_p]
        lib.render_thread_proc.argtypes = [C.POINTER(RenderingContext)]
        lib.render_thread_proc.restype = None
        lib.rendering_context_is_finished.argtypes = [C.POINTER(RenderingContext)]
        lib.rendering_context_is_finished.restype = C.c_bool
        lib.rendering_context_finish.argtypes = [C.POINTER(RenderingContext)]
        lib.rendering_context_finish.restype = None
        lib.denoise_image.argtypes = [C.POINTER(Image), C.POINTER(Image), isize]
        lib.denoise_image.restype = None
        _gpu = lib
    return _gpu


def gpu_check(rc: int) -> None:
    if rc:
        raise RuntimeError("libraytracer_gpu: " + gpu_lib().rt_gpu_last_error().decode())
