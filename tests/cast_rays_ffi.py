"""Radiance for caller rays, for the tests: the batch CPU reference (oracle_cast_rays, tests/csrc/cast_rays_oracle.c), the
oracle's per-ray cast_ray seeded by hand, the renderer's camera rays restated on the CPU (tests/csrc/camera_rays.c) and
the device-level GPU call on torch tensors.  TEST INFRASTRUCTURE ONLY.

Both C files are compiled on first use into a private temporary directory (the tree is never written).  Rays are (n, 6)
float32 arrays laid out as the C Ray (position, direction); keys are (n,) uint32 or None (the ray's index).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle_ffi
from raytracing_c_b200._ffi import Scene, isize

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tests", "csrc")

_build_dir = None
_camera_lib = None
_cast_lib = None


def _ptr(a):
    return a.ctypes.data if a is not None else None


def _compile(name, args):
    global _build_dir
    if _build_dir is None:
        _build_dir = tempfile.mkdtemp(prefix="rt_cast_rays_")
    out = os.path.join(_build_dir, name)
    r = subprocess.run(["gcc", *args, "-shared", "-fPIC", "-o", out], capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f"building {name} failed:\n{r.stdout}{r.stderr}")
    return out


def cast_lib() -> C.CDLL:
    """oracle_cast_rays, built with the oracle's flags over its unmodified oracle_trace.c, linked against liboracle.so
    (whose shading callbacks the scenes of the tests carry)."""
    global _cast_lib
    if _cast_lib is None:
        oracle_ffi.lib()                                   # builds liboracle.so if it is missing
        o = oracle_ffi.ORACLE_DIR
        path = _compile("libcast_rays_oracle.so", [
            "-O2", "-std=gnu11", "-mavx2", "-mfma", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), "-I", o,
            os.path.join(CSRC, "cast_rays_oracle.c"), "-L", o, "-loracle", f"-Wl,-rpath,{o}", "-lpthread", "-lm"])
        lib = C.CDLL(path)
        lib.oracle_cast_rays.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, isize, isize, isize, C.c_uint32,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        lib.oracle_cast_rays.restype = None
        _cast_lib = lib
    return _cast_lib


def oracle_lib() -> C.CDLL:
    o = oracle_ffi.lib()
    o.oracle_cast_ray.argtypes = [C.POINTER(Scene), oracle_ffi.Ray, isize]
    o.oracle_cast_ray.restype = oracle_ffi.Vec3
    o.oracle_path_seed.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
    o.oracle_path_seed.restype = C.c_uint32
    return o


def oracle_cast_rays(loaded, rays, samples, max_bounces=8, sample_begin=0, user_seed=0, keys=None, n_threads=8) -> dict:
    """oracle_cast_rays (tests/csrc/cast_rays_oracle.c): per-ray sums (n, 3), per-sample radiance (n, samples, 3) and the
    eight counters."""
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = len(rays)
    if keys is not None:
        keys = np.ascontiguousarray(keys, dtype=np.uint32)
    sums = np.zeros((n, 3), dtype=np.float32)
    per = np.zeros((n, samples, 3), dtype=np.float32)
    ctr = np.zeros(8, dtype=np.uint64)
    cast_lib().oracle_cast_rays(C.byref(loaded.scene), rays.ctypes.data, _ptr(keys), n, sample_begin, samples, max_bounces,
                                user_seed, sums.ctypes.data, per.ctypes.data, ctr.ctypes.data, n_threads)
    return {"radiance": sums, "per_sample": per, "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr)))}


def _ray(r):
    ray = oracle_ffi.Ray()
    ray.position.x, ray.position.y, ray.position.z, ray.direction.x, ray.direction.y, ray.direction.z = map(float, r)
    return ray


def oracle_cast_ray_seeded(loaded, ray, key, sample, max_bounces, user_seed=0):
    """The oracle's single cast_ray with its shader generator set to rt_path_seed(key, sample, user_seed) by hand."""
    o = oracle_lib()
    o.oracle_shader_random_state()[0] = o.oracle_path_seed(int(key), int(sample), int(user_seed))
    c = o.oracle_cast_ray(C.byref(loaded.scene), _ray(ray), max_bounces)
    return np.array([c.x, c.y, c.z], dtype=np.float32)


def ref_cast_ray_seeded(loaded, ray, key, sample, max_bounces, user_seed=0):
    """The reference's own cast_ray (oracle/ref_glue_rt.c) with its shader generator seeded the same way."""
    import ref_ffi
    r = ref_ffi.lib()
    r.ref_random_state()[0] = oracle_lib().oracle_path_seed(int(key), int(sample), int(user_seed))
    c = r.ref_cast_ray(C.byref(loaded.scene), _ray(ray), max_bounces)
    return np.array([c.x, c.y, c.z], dtype=np.float32)


def camera_lib() -> C.CDLL:
    global _camera_lib
    if _camera_lib is None:
        lib = C.CDLL(_compile("libcamera_rays.so", ["-O2", "-std=gnu11", "-ffp-contract=off", "-I",
                                                    os.path.join(ROOT, "include"), os.path.join(CSRC, "camera_rays.c"),
                                                    "-lm"]))
        lib.camera_rays.argtypes = [C.c_void_p, isize, isize, isize, C.c_void_p]
        lib.camera_rays.restype = None
        _camera_lib = lib
    return _camera_lib


def camera_rays(loaded, width, height, sample) -> np.ndarray:
    """The renderer's camera ray of every pixel (row-major) for sample index `sample`: (width * height, 6) float32."""
    out = np.zeros((width * height, 6), dtype=np.float32)
    camera_lib().camera_rays(C.addressof(loaded.scene.camera), width, height, sample, out.ctypes.data)
    return out


def device_cast_rays(loaded, rays, samples, max_bounces=8, sample_begin=0, user_seed=0, keys=None, per_sample=True,
                     radiance=None, accumulate=False, stream=None) -> dict:
    """rt_gpu_cast_rays_device on torch tensors, on `stream` (default: torch's current stream).  `rays` and `keys` may be
    numpy arrays or CUDA tensors; `radiance` (a CUDA tensor, (n, 3)) is continued from with accumulate.  Returns numpy
    radiance, per-sample radiance and the eight counters."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    r = rays if isinstance(rays, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(rays, dtype=np.float32)).cuda()
    k = None
    if keys is not None:
        k = keys if isinstance(keys, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(keys, dtype=np.uint32).view(np.int32)).cuda()
    n = r.shape[0]
    rad = radiance if radiance is not None else torch.full((max(n, 1), 3), 7.0, dtype=torch.float32, device="cuda")
    per = torch.full((max(n * samples, 1), 3), 7.0, dtype=torch.float32, device="cuda") if per_sample else None
    ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
    st = stream or torch.cuda.current_stream()
    driver.register_callbacks(loaded)
    gpu_check(gpu_lib().rt_gpu_cast_rays_device(C.byref(loaded.scene), r.data_ptr(), k.data_ptr() if k is not None else None,
                                                n, sample_begin, samples, max_bounces, user_seed, int(accumulate),
                                                rad.data_ptr(), per.data_ptr() if per is not None else None, ctr.data_ptr(),
                                                st.cuda_stream))
    st.synchronize()
    out = {"radiance": rad[:n].cpu().numpy(), "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy())))}
    if per is not None:
        out["per_sample"] = per[:n * samples].cpu().numpy().reshape(n, samples, 3)
    return out


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
