"""ctypes bindings of oracle/_ref/libref.so — the reference's OWN raytracer.c / scene.c / denoiser.c /
driver.c compiled unmodified over the Codin stand-in (oracle/codin_shim).  TEST INFRASTRUCTURE ONLY.

The library can only be (re)built from a checkout of the reference named by RT_REFERENCE_DIR.
available() says whether the tests that need it can run.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from raytracing_c_b200._ffi import Image, RenderingContext, Scene, TriangleSlice, Vec2, Vec3, isize
from oracle_ffi import Ray, ORACLE_DIR

REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libref.so")


class RefHit(C.Structure):
    _fields_ = [("distance", C.c_float), ("normal", Vec3), ("normal_geo", Vec3), ("point", Vec3),
                ("tangent", Vec3), ("bitangent", Vec3), ("tex_coords", Vec2), ("shader_data", C.c_void_p)]


def available() -> bool:
    if os.path.exists(REF_LIB):
        return True
    if os.path.isdir(os.environ.get("RT_REFERENCE_DIR", "")):
        return subprocess.run(["make", "-C", ORACLE_DIR, "ref"], capture_output=True).returncode == 0
    return False


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        assert available(), "oracle/_ref/libref.so is missing and RT_REFERENCE_DIR names no reference checkout"
        r = C.CDLL(REF_LIB)
        r.ref_scene_init.argtypes = [C.POINTER(Scene), TriangleSlice]
        r.render_thread_proc.argtypes = [C.POINTER(RenderingContext)]
        r.denoise_image.argtypes = [C.POINTER(Image), C.POINTER(Image), isize]
        r.ref_cast_ray.argtypes = [C.POINTER(Scene), Ray, isize]
        r.ref_cast_ray.restype = Vec3
        r.ref_trace_ray.argtypes = [C.POINTER(Scene), Ray, C.POINTER(RefHit)]
        r.ref_hash12.argtypes = [C.c_float, C.c_float]
        r.ref_hash12.restype = C.c_float
        r.ref_shader_proc.restype = C.c_void_p
        r.ref_background_proc.restype = C.c_void_p
        r.ref_random_state.restype = C.POINTER(C.c_uint32)
        r.ref_sample_texture_bilinear.argtypes = [C.POINTER(Image), Vec2]
        r.ref_sample_texture_bilinear.restype = Vec3
        r.ref_sample_background.argtypes = [C.POINTER(Image), Vec3]
        r.ref_sample_background.restype = Vec3
        for name in ("ref_sizeof_triangle", "ref_sizeof_triangle_aos", "ref_sizeof_scene", "ref_sizeof_context",
                     "ref_sizeof_bvh_node"):
            getattr(r, name).restype = isize
        _lib = r
    return _lib


def scene_builder():
    return lib().ref_scene_init


def render_reference_mode(loaded, width, height, samples, max_bounces=8):
    """The reference's render_thread_proc on ONE thread with its shader stream starting at 0."""
    from raytracing_c_b200.driver import image_view
    pixels = np.zeros((height, width, 3), dtype=np.uint8)
    ctx = RenderingContext()
    ctx.image = image_view(pixels)
    ctx.scene = C.pointer(loaded.scene)
    ctx.samples, ctx.max_bounces, ctx.n_threads, ctx._current_chunk = samples, max_bounces, 1, 0
    lib().ref_random_state()[0] = 0
    lib().render_thread_proc(C.byref(ctx))
    assert ctx.n_threads == 0
    return pixels


def cast_rays_per_sample(loaded, width, height, samples, max_bounces=8, user_seed=0):
    """The reference's cast_ray per (pixel, sample) with rt_path_seed seeding and exact primary rays."""
    import oracle_ffi
    o = oracle_ffi.lib()
    o.oracle_primary_ray.restype = Ray
    o.oracle_primary_ray.argtypes = [C.c_void_p, isize, isize, isize, isize, isize]
    o.oracle_path_seed.restype = C.c_uint32
    o.oracle_path_seed.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
    r = lib()
    state = r.ref_random_state()
    out = np.zeros((height, width, samples, 3), dtype=np.float32)
    cam = C.addressof(loaded.scene.camera)
    scene = C.byref(loaded.scene)
    for y in range(height):
        for x in range(width):
            for s in range(samples):
                ray = o.oracle_primary_ray(cam, width, height, x, y, s)
                state[0] = o.oracle_path_seed(y * width + x, s, user_seed)
                c = r.ref_cast_ray(scene, ray, max_bounces)
                out[y, x, s] = (c.x, c.y, c.z)
    return out


def denoise(src: np.ndarray) -> np.ndarray:
    from raytracing_c_b200.driver import image_view
    src = np.ascontiguousarray(src)
    dst = np.zeros_like(src)
    a, b = image_view(src), image_view(dst)
    lib().denoise_image(C.byref(a), C.byref(b), 1)
    return dst


def lightmap_bake(loaded, width, height, samples, dir_state=0, shader_state=0):
    """The reference's own lightmap_bake (raytracer.c:722-784), both generator copies started where asked.
    It writes texels at x == width / y == height when a UV is exactly 1.0 (out of bounds): the image handed to it
    has 8 spare columns (stride) and 8 spare rows for those; the in-range region is returned."""
    from raytracing_c_b200.driver import image_view
    r = lib()
    r.ref_rt_random_state.restype = C.POINTER(C.c_uint32)
    r.lightmap_bake.argtypes = [C.POINTER(Image), C.c_void_p, isize]
    r.lightmap_bake.restype = None
    padded = np.zeros((height + 8, width + 8, 3), dtype=np.uint8)
    im = image_view(padded)
    im.width, im.height, im.stride = width, height, width + 8
    r.ref_rt_random_state()[0] = dir_state
    r.ref_random_state()[0] = shader_state
    r.lightmap_bake(C.byref(im), C.byref(loaded.scene), samples)
    return np.ascontiguousarray(padded[:height, :width])
