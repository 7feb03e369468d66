"""Many views of a resident scene, for the tests: the device-level GPU call on torch tensors, the single renders it
replaces (rt_gpu_render_accum_device with scene->camera set per view), and the camera sets the tests use.
TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

import oracle_ffi
from helpers import bits  # noqa: F401  (bits is re-exported)
from raytracing_c_b200._ffi import Camera

CTR16_NAMES = oracle_ffi.COUNTER_NAMES + [f"ex{i}" for i in range(8)]


def copy_camera(cam) -> Camera:
    out = Camera()
    C.memmove(C.addressof(out), C.addressof(cam), C.sizeof(Camera))
    return out


def camera_bytes(cam) -> bytes:
    return C.string_at(C.addressof(cam), C.sizeof(Camera))


def _counters(n_slots):
    """(tensor, pointer): a zeroed 8-slot torch counter block, or the library's own 16-slot block, reset."""
    import torch
    from raytracing_c_b200 import gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    if n_slots == 8:
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        return ctr, ctr.data_ptr()
    p = C.c_void_p()
    gpu_check(gpu_lib().rt_gpu_counters_buffer(C.byref(p)))
    gpu_check(gpu_lib().rt_gpu_counters_reset())
    return None, p.value


def _read_counters(ctr, n_slots) -> dict:
    from raytracing_c_b200 import gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    if ctr is not None:
        return dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy())))
    out = np.zeros(16, dtype=np.uint64)
    gpu_check(gpu_lib().rt_gpu_read_counters_ex(out.ctypes.data))
    return dict(zip(CTR16_NAMES, map(int, out)))


def device_views(loaded, cameras, width, height, sample_begin, sample_end, max_bounces=8, user_seeds=None, accum=None,
                 accumulate=False, n_counters=8, stream=None) -> dict:
    """rt_gpu_render_views_device on `stream` (default: torch's current stream).  `accum` (a CUDA float32 tensor of
    V * H * W * 3) is continued from with accumulate; a fresh one is filled with 7.0 first, so a value the call does not
    write shows.  n_counters 8: a torch block; 16: the library's own block, reset first.  Returns the (V, H, W, 3)
    accumulator, the counters and the kernels launched."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    n = len(cameras)
    acc = accum if accum is not None else torch.full((max(n, 1) * width * height * 3,), 7.0, dtype=torch.float32,
                                                     device="cuda")
    cams = (Camera * max(n, 1))(*cameras)
    seeds = None if user_seeds is None else np.ascontiguousarray(user_seeds, dtype=np.uint32)
    driver.register_callbacks(loaded)
    torch.cuda.synchronize()
    ctr, ctr_ptr = _counters(n_counters)
    st = stream or torch.cuda.current_stream()
    gpu = gpu_lib()
    before = gpu.rt_gpu_last_launches()
    gpu_check(gpu.rt_gpu_render_views_device(C.byref(loaded.scene), n, cams, seeds.ctypes.data if seeds is not None else None,
                                             width, height, sample_begin, sample_end, max_bounces, int(accumulate),
                                             acc.data_ptr(), ctr_ptr, st.cuda_stream))
    launches = gpu.rt_gpu_last_launches() - before
    st.synchronize()
    return {"accum": acc.cpu().numpy()[:n * width * height * 3].reshape(n, height, width, 3),
            "counters": _read_counters(ctr, n_counters), "launches": launches}


def device_single(loaded, camera, width, height, sample_begin, sample_end, max_bounces=8, user_seed=0, accum=None,
                  accumulate=False, n_counters=8) -> dict:
    """rt_gpu_render_accum_device with scene->camera = camera (restored afterwards), from zero on a fresh buffer unless
    `accum` is given: the accumulator, counters and kernels launched."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    acc = accum if accum is not None else torch.full((width * height * 3,), 7.0, dtype=torch.float32, device="cuda")
    driver.register_callbacks(loaded)
    torch.cuda.synchronize()
    ctr, ctr_ptr = _counters(n_counters)
    own = copy_camera(loaded.scene.camera)
    gpu = gpu_lib()
    try:
        if camera is not None:
            loaded.scene.camera = copy_camera(camera)
        before = gpu.rt_gpu_last_launches()
        gpu_check(gpu.rt_gpu_render_accum_device(C.byref(loaded.scene), width, height, sample_begin, sample_end,
                                                 max_bounces, user_seed, int(accumulate), acc.data_ptr(), None, None,
                                                 ctr_ptr, torch.cuda.current_stream().cuda_stream))
        launches = gpu.rt_gpu_last_launches() - before
        torch.cuda.synchronize()
    finally:
        loaded.scene.camera = own
    return {"accum": acc.cpu().numpy().reshape(height, width, 3), "counters": _read_counters(ctr, n_counters),
            "launches": launches}


def singles(loaded, cameras, width, height, sample_begin, sample_end, max_bounces=8, user_seeds=None, n_counters=8):
    """The per-view renders a views call replaces: (V, H, W, 3) accumulators and the summed counters."""
    outs = [device_single(loaded, cam, width, height, sample_begin, sample_end, max_bounces,
                          0 if user_seeds is None else int(user_seeds[v]), n_counters=n_counters)
            for v, cam in enumerate(cameras)]
    total = {k: sum(o["counters"][k] for o in outs) for k in outs[0]["counters"]} if outs else {}
    return {"accum": np.stack([o["accum"] for o in outs]) if outs else None, "counters": total,
            "launches": [o["launches"] for o in outs]}


def bounds(loaded):
    """(lo, hi) of the scene's occupied triangle slots (float64)."""
    from raytracing_c_b200 import driver
    p = driver.scene_positions(loaded).astype(np.float64)          # [axis][vertex][slot]
    occupied = np.any(p != 0, axis=(0, 1))
    pts = p[:, :, occupied].reshape(3, -1)
    return pts.min(axis=1), pts.max(axis=1)


def orbit(loaded, n, radius_scale=2.5, fov=60.0, height=0.3):
    """n cameras on a circle around the scene's bounds, looking at its centre."""
    from raytracing_c_b200 import driver
    lo, hi = bounds(loaded)
    c = (lo + hi) / 2
    r = max(float(np.linalg.norm(hi - lo)) / 2, 1e-3)
    cams = []
    for k in range(n):
        a = 2 * np.pi * k / n + 0.3
        eye = c + radius_scale * r * np.array([np.sin(a), height, np.cos(a)])
        cams.append(driver.look_at(tuple(map(float, eye)), tuple(map(float, c)), fov_degrees=fov))
    return cams


def all_sky_camera(loaded):
    """A camera whose view holds no geometry: far from the scene, the scene in front of its plane but 50 degrees off its
    axis, looking along (1, 1, 1) so no direction component comes near zero over a 40-degree field of view (every tile
    can be sky)."""
    from raytracing_c_b200 import driver
    lo, hi = bounds(loaded)
    c = (lo + hi) / 2
    r = max(float(np.linalg.norm(hi - lo)) / 2, 1e-3)
    d = np.ones(3) / np.sqrt(3)
    w = np.array([1.0, -1.0, 0.0]) / np.sqrt(2)
    to_scene = d + np.tan(np.deg2rad(50)) * w
    to_scene /= np.linalg.norm(to_scene)
    eye = c - 12 * r * to_scene
    return driver.look_at(tuple(map(float, eye)), tuple(map(float, eye + d)), fov_degrees=40.0)


def inside_camera(loaded):
    """A camera at the centre of the scene's bounds (no tile can be sky)."""
    from raytracing_c_b200 import driver
    lo, hi = bounds(loaded)
    c = (lo + hi) / 2
    return driver.look_at(tuple(map(float, c)), tuple(map(float, c + np.array([0.3, -0.2, -1.0]))), fov_degrees=80.0)


def camera_set(loaded):
    """The scene's own camera, two orbit cameras with different fields of view (so different focal lengths), a duplicate
    of the scene's camera, an all-sky view and a view from inside the bounds."""
    own = copy_camera(loaded.scene.camera)
    a = orbit(loaded, 2, fov=35.0)
    b = orbit(loaded, 3, radius_scale=1.8, fov=95.0)
    return [own, a[0], copy_camera(own), all_sky_camera(loaded), b[1], inside_camera(loaded)]
