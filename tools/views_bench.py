#!/usr/bin/env python
"""views_bench.py — many views of one resident scene: one rt_gpu_render_views_device call against a loop of per-view
rt_gpu_render_accum_device calls, on helmet.glb with 8 bounces and cameras on an orbit around the model.

    python tools/views_bench.py [--reps 7] [--out profiles/r12_views_bench.json] [--quick]

Workloads: (a) 64 views of 256x256 at 16 spp; (b) 4 views of 1920x1080 at 64 spp (--quick: small sizes, for a dry run).
Arms, alternating in one run after a warm-up of each: the batched call, and the loop (scene->camera rewritten before
each view's render, every render into its own slice).  Each arm is timed with CUDA events around the whole call or loop
(the host's enqueue included), and the median of `reps` is reported with ms, Msamples/s (views * W * H * spp per second)
and loop / batched.  Every timed batched result is compared bit for bit with the loop's.  The card name and power
limit are read in the same run.
"""
from __future__ import annotations

import ctypes as C
import json

import numpy as np
import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
from raytracing_c_b200 import driver
from raytracing_c_b200._ffi import Camera, gpu_check
from views_ffi import copy_camera

BOUNCES = 8
WORKLOADS = {"a": dict(views=64, width=256, height=256, spp=16), "b": dict(views=4, width=1920, height=1080, spp=64)}
QUICK = {"a": dict(views=8, width=64, height=64, spp=4), "b": dict(views=2, width=192, height=108, spp=4)}


def orbit_cameras(driver, loaded, n):
    """n cameras on a circle at 1.6 bounding radii around the model, 15 degrees above its centre, looking at it."""
    p = driver.scene_positions(loaded).astype(np.float64)
    pts = p[:, :, np.any(p != 0, axis=(0, 1))].reshape(3, -1)
    lo, hi = pts.min(axis=1), pts.max(axis=1)
    c, r = (lo + hi) / 2, float(np.linalg.norm(hi - lo)) / 2
    cams = []
    for k in range(n):
        a = 2 * np.pi * k / n
        eye = c + 1.6 * r * np.array([np.cos(np.deg2rad(15)) * np.sin(a), np.sin(np.deg2rad(15)), np.cos(np.deg2rad(15)) * np.cos(a)])
        cams.append(driver.look_at(tuple(map(float, eye)), tuple(map(float, c)), fov_degrees=60.0))
    return cams


def main() -> None:
    ap = benchkit.parser(reps=7)
    ap.add_argument("--quick", action="store_true", help="small workloads (a dry run of the script)")
    args = ap.parse_args()
    gpu = benchkit.init()
    loaded = benchkit.resident("helmet.glb")
    scene = C.byref(loaded.scene)
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    own_camera = copy_camera(loaded.scene.camera)
    result = {"card": benchkit.card(), "model": "helmet.glb", "max_bounces": BOUNCES, "reps": args.reps,
              "cameras": "orbit at 1.6 bounding radii, 15 degrees up, 60-degree field of view",
              "timing": "CUDA events around the batched call / the whole loop, host enqueue included; median of reps",
              "workloads": {}}
    all_identical = True

    for key, wl in (QUICK if args.quick else WORKLOADS).items():
        n, w, h, spp = wl["views"], wl["width"], wl["height"], wl["spp"]
        cams = orbit_cameras(driver, loaded, n)
        carr = (Camera * n)(*cams)
        batched = torch.empty((n, h, w, 3), dtype=torch.float32, device="cuda")
        looped = torch.empty_like(batched)

        def views():
            gpu_check(gpu.rt_gpu_render_views_device(scene, n, carr, None, w, h, 0, spp, BOUNCES, 0, batched.data_ptr(),
                                                     None, st))

        def loop():
            for v in range(n):
                loaded.scene.camera = cams[v]
                gpu_check(gpu.rt_gpu_render_accum_device(scene, w, h, 0, spp, BOUNCES, 0, 0, looped[v].data_ptr(), None,
                                                         None, None, st))
            loaded.scene.camera = own_camera

        views(); loop()                                       # warm-up: workspace, modules, pools
        torch.cuda.synchronize()
        t_views, t_loop, identical = [], [], True
        for _ in range(args.reps):
            t_views.append(benchkit.window_ms(views, stream))
            t_loop.append(benchkit.window_ms(loop, stream))
            identical &= bool(torch.equal(batched.view(torch.int32), looped.view(torch.int32)))
        samples = n * w * h * spp
        mv, ml = float(np.median(t_views)), float(np.median(t_loop))
        r = {"views": n, "frame": f"{w}x{h}", "spp": spp, "samples": samples,
             "batched_ms": [round(t, 3) for t in t_views], "loop_ms": [round(t, 3) for t in t_loop],
             "batched_median_ms": round(mv, 3), "loop_median_ms": round(ml, 3),
             "batched_Msamples_per_s": round(samples / (mv * 1e-3) / 1e6, 1),
             "loop_Msamples_per_s": round(samples / (ml * 1e-3) / 1e6, 1),
             "loop_over_batched": round(ml / mv, 4), "bitwise_identical": identical}
        all_identical &= identical
        result["workloads"][key] = r
        print(json.dumps({key: r}), flush=True)

    result["parity_ok"] = all_identical
    benchkit.finish(args, result, ("parity_ok",), loaded)


if __name__ == "__main__":
    main()
