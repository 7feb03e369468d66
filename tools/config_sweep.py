"""Renders every BASELINE.json config on the visible GPU and prints one JSON line per run.

    python tools/config_sweep.py [--quick]

configs: spheres.glb 1024^2 x16 (driver defaults) | quad / fov_test 1024^2 x1 (hit ids) | helmet.glb 1080p x1024 |
sheen.glb 1024^2 x16 + denoise | tower.obj 3840x2160, spp in {1,4,16,64,256,1024}.
Times are CUDA-event times of the render (device buffers, scene resident); the denoise pass is timed separately.
"""
import argparse
import ctypes as C
import json
import os

import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
from helpers import upload
from raytracing_c_b200 import driver
from raytracing_c_b200._ffi import gpu_check

ap = argparse.ArgumentParser()
ap.add_argument("--quick", action="store_true", help="cap spp at 64")
args = ap.parse_args()

CAMERAS = {"quad.obj": dict(eye=(3.0, 0.0, 0.0), target=(0.0, 0.0, 0.0)),
           "tower.obj": dict(eye=(0.0, 12.5, 40.0), target=(0.0, 12.5, 0.0))}
RUNS = [("spheres.glb", 1024, 1024, [16], False), ("quad.obj", 1024, 1024, [1], False),
        ("fov_test.obj", 1024, 1024, [1], False), ("helmet.glb", 1920, 1080, [1024], False),
        ("sheen.glb", 1024, 1024, [16], True), ("tower.obj", 3840, 2160, [1, 4, 16, 64, 256, 1024], False)]

gpu = benchkit.init()
torch.cuda.set_device(0)
stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
for model, W, H, spps, denoise in RUNS:
    cam = driver.look_at(**CAMERAS[model]) if model in CAMERAS else None
    loaded = driver.load_scene(os.path.join(benchkit.ROOT, "assets", "models", model), camera=cam)
    if model == "sheen.glb":                       # the asset declares no sheen: inject it (SURVEY fact 7)
        for i in range(loaded.model.n_materials):
            loaded.model.materials[i].sheen, loaded.model.materials[i].sheen_tint = 1.0, 0.5
    upload(loaded)
    scene = C.byref(loaded.scene)
    accum = torch.zeros(W * H * 3, dtype=torch.float32, device="cuda")
    pixels = torch.zeros(W * H * 3, dtype=torch.uint8, device="cuda")
    pixels2 = torch.zeros(W * H * 3, dtype=torch.uint8, device="cuda")
    for spp in spps:
        if args.quick and spp > 64:
            continue
        driver.set_options(slice_samples=spp)
        best = None
        for rep in range(3 if spp <= 64 else 2):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            gpu_check(gpu.rt_gpu_render_accum_device(scene, W, H, 0, spp, 8, 0, 0, accum.data_ptr(), None, None, None, stream))
            gpu_check(gpu.rt_gpu_resolve_device(accum.data_ptr(), W, H, spp, pixels.data_ptr(), W, 3, stream))
            e1.record()
            if denoise:
                gpu_check(gpu.rt_gpu_denoise_device(pixels.data_ptr(), pixels2.data_ptr(), W, H, W, W, 3, stream))
            e2.record()
            torch.cuda.synchronize()
            ms, dms = e0.elapsed_time(e1), e1.elapsed_time(e2)
            if rep and (best is None or ms < best[0]):
                best = (ms, dms)
        print(json.dumps({"model": model, "width": W, "height": H, "spp": spp, "triangles": int(loaded.n_triangles),
                          "render_ms": round(best[0], 3), "Msamples_per_s": round(W * H * spp / best[0] / 1e3, 1),
                          "denoise_ms": round(best[1], 3) if denoise else None}), flush=True)
    loaded.close()
