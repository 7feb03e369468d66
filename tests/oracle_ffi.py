"""ctypes bindings of the CPU oracle (oracle/liboracle.so) — TEST INFRASTRUCTURE ONLY.

Imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs; never by raytracing_c_b200/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from raytracing_c_b200._ffi import (Image, RenderingContext, Scene, TriangleSlice, Vec2, Vec3, isize)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "liboracle.so")

SEED_REFERENCE, SEED_PER_SAMPLE = 0, 1
COUNTER_NAMES = ["rays", "nodes", "leaves", "accepts", "shades", "misses", "passthrough", "samples"]


class Ray(C.Structure):
    _fields_ = [("position", Vec3), ("direction", Vec3)]


class OracleOptions(C.Structure):
    _fields_ = [("seed_mode", C.c_int32), ("user_seed", C.c_uint32), ("approx_rsqrt", C.c_int32),
                ("sample_begin", C.c_int32), ("sample_end", C.c_int32),
                ("accum", C.c_void_p), ("per_sample", C.c_void_p), ("hit_ids", C.c_void_p),
                ("counters", C.c_uint64 * 8), ("pixel_mask", C.c_void_p)]


class OracleLightmapOptions(C.Structure):
    _fields_ = [("seed_mode", C.c_int32), ("user_seed", C.c_uint32), ("dir_state", C.c_uint32), ("shader_state", C.c_uint32),
                ("values", C.c_void_p), ("owner", C.c_void_p), ("texels_written", C.c_int64)]


def build_oracle() -> None:
    out = subprocess.run(["make", "-C", ORACLE_DIR, "all"], capture_output=True, text=True)
    if out.returncode:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_LIB):
            build_oracle()
        o = C.CDLL(ORACLE_LIB)
        o.oracle_scene_init.argtypes = [C.POINTER(Scene), TriangleSlice]
        o.oracle_scene_destroy.argtypes = [C.POINTER(Scene)]
        o.oracle_render.argtypes = [C.POINTER(RenderingContext), C.POINTER(OracleOptions), C.c_int32]
        o.oracle_trace_ray.argtypes = [C.POINTER(Scene), Ray, C.POINTER(C.c_float)]
        o.oracle_trace_ray.restype = C.c_int32
        o.oracle_hash12.argtypes = [C.c_float, C.c_float]
        o.oracle_hash12.restype = C.c_float
        o.oracle_denoise_image.argtypes = [C.POINTER(Image), C.POINTER(Image), isize]
        o.oracle_resolve.argtypes = [C.c_void_p, isize, isize, C.c_void_p]
        o.oracle_sample_texture_bilinear.argtypes = [C.POINTER(Image), Vec2]
        o.oracle_sample_texture_bilinear.restype = Vec3
        o.oracle_sample_background.argtypes = [C.c_void_p, Vec3]
        o.oracle_sample_background.restype = Vec3
        o.oracle_shader_random_state.restype = C.POINTER(C.c_uint32)
        o.oracle_lightmap_bake.argtypes = [C.POINTER(Image), C.POINTER(Scene), isize, C.POINTER(OracleLightmapOptions)]
        o.oracle_lightmap_bake.restype = None
        _lib = o
    return _lib


def shader_proc() -> int:
    return C.cast(lib().oracle_disney_shader_proc, C.c_void_p).value


def background_proc() -> int:
    return C.cast(lib().oracle_sample_background, C.c_void_p).value


def render(loaded, width, height, samples, max_bounces=8, n_threads=1, seed_mode=SEED_PER_SAMPLE, user_seed=0,
           sample_begin=0, sample_end=0, want_accum=True, want_per_sample=False, want_hit_ids=False,
           approx_rsqrt=False, pixel_mask=None):
    """Runs the oracle's render_thread_proc restatement; returns a dict of numpy arrays.
    `pixel_mask` (H, W) uint8: only pixels with a non-zero byte are rendered (the others stay 0)."""
    from raytracing_c_b200.driver import image_view
    pixels = np.zeros((height, width, 3), dtype=np.uint8)
    ctx = RenderingContext()
    ctx.image = image_view(pixels)
    ctx.scene = C.pointer(loaded.scene)
    ctx.samples, ctx.max_bounces = samples, max_bounces
    opt = OracleOptions()
    opt.seed_mode, opt.user_seed, opt.approx_rsqrt = seed_mode, user_seed, int(approx_rsqrt)
    opt.sample_begin, opt.sample_end = sample_begin, sample_end
    n_s = (sample_end or samples) - sample_begin
    out = {"pixels": pixels}
    if want_accum:
        out["accum"] = np.zeros((height, width, 3), dtype=np.float32)
        opt.accum = out["accum"].ctypes.data
    if want_per_sample:
        out["per_sample"] = np.zeros((height, width, n_s, 3), dtype=np.float32)
        opt.per_sample = out["per_sample"].ctypes.data
    if want_hit_ids:
        out["hit_ids"] = np.full((height, width), -1, dtype=np.int32)
        opt.hit_ids = out["hit_ids"].ctypes.data
    if pixel_mask is not None:
        pixel_mask = np.ascontiguousarray(pixel_mask, dtype=np.uint8)
        assert pixel_mask.shape == (height, width)
        opt.pixel_mask = pixel_mask.ctypes.data
    lib().oracle_render(C.byref(ctx), C.byref(opt), n_threads)
    out["counters"] = {k: int(v) for k, v in zip(COUNTER_NAMES, opt.counters)}
    return out


def denoise(src: np.ndarray, n_threads: int = 1) -> np.ndarray:
    from raytracing_c_b200.driver import image_view
    src = np.ascontiguousarray(src)
    dst = np.zeros_like(src)
    a, b = image_view(src), image_view(dst)
    lib().oracle_denoise_image(C.byref(a), C.byref(b), n_threads)
    return dst


def rsqrt_ps(x: np.ndarray) -> np.ndarray:
    """_mm256_rsqrt_ps of every element on this CPU (the approximation of reference seed mode's primary rays)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty_like(x)
    lib().oracle_rsqrt_ps_array(x.ctypes.data, out.ctypes.data, C.c_ssize_t(x.size))
    return out


def resolve(accum: np.ndarray, samples: int) -> np.ndarray:
    accum = np.ascontiguousarray(accum, dtype=np.float32)
    out = np.zeros(accum.shape, dtype=np.uint8)
    lib().oracle_resolve(accum.ctypes.data, accum.size // 3, samples, out.ctypes.data)
    return out


def lightmap_bake(loaded, width, height, samples, seed_mode=SEED_PER_SAMPLE, user_seed=0, dir_state=0, shader_state=0):
    """oracle_lightmap_bake (raytracer.c:722-784): returns the u8 lightmap, the f32 values before the u8 store,
    the slot that wrote each texel last (-1 = untouched) and the number of stores."""
    from raytracing_c_b200.driver import image_view
    pixels = np.zeros((height, width, 3), dtype=np.uint8)
    values = np.zeros((height, width, 3), dtype=np.float32)
    owner = np.full((height, width), -1, dtype=np.int32)
    im = image_view(pixels)
    opt = OracleLightmapOptions()
    opt.seed_mode, opt.user_seed, opt.dir_state, opt.shader_state = seed_mode, user_seed, dir_state, shader_state
    opt.values, opt.owner = values.ctypes.data, owner.ctypes.data
    lib().oracle_lightmap_bake(C.byref(im), C.byref(loaded.scene), samples, C.byref(opt))
    return dict(pixels=pixels, values=values, owner=owner, stores=int(opt.texels_written),
                dir_state=int(opt.dir_state), shader_state=int(opt.shader_state))
