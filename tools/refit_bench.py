#!/usr/bin/env python
"""refit_bench.py — what moving the geometry of a resident scene costs: the refit (rt_gpu_scene_refit_device /
rt_gpu_scene_refit) against rebuilding and re-uploading (scene_init + rt_gpu_scene_upload), and what a refit costs in
trace work, on helmet.glb and tower.obj.

    python tools/refit_bench.py [--reps 20] [--out refit_bench.json]

Per model:
1. Device refit: CUDA events around rt_gpu_scene_refit_device on torch's current stream (the call synchronises before
   it returns, so the host wall-clock time is given beside it), median over `reps` calls after 3 warm-up calls,
   alternating two deformed position sets so every call changes the geometry.
2. Host refit (rt_gpu_scene_refit): host wall clock around the call (staging, refit, write-back), median.
3. Rebuild: scene_init of the same deformed mesh on a new Scene, then rt_gpu_scene_upload of it and a device
   synchronise; host wall clock of each part, median over `reps // 4` (at least 3) rebuilds.
4. Trace work: node visits and leaf visits per ray of a 480x270, 4 spp, 8-bounce render (the counters of the render)
   on the original mesh, after a sequence of 8 refits of growing deformation (p += a * sin(3 p.yzx), a up to 0.2 of
   the model's extent), and on a fresh scene_init of the final deformed mesh.
The card name and power limit are read in the same run.
"""
from __future__ import annotations

import ctypes as C
import json
import time

import numpy as np
import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
from raytracing_c_b200 import driver, host_lib
from raytracing_c_b200._ffi import Scene, gpu_check
from refit_ffi import deform

MODELS = {"helmet.glb": None, "tower.obj": dict(eye=(0.0, 12.5, 40.0), target=(0.0, 12.5, 0.0))}
W, H, SPP, BOUNCES = 480, 270, 4, 8


def main() -> None:
    args = benchkit.parser(reps=20).parse_args()
    gpu, host = benchkit.init(), host_lib()
    result = {"card": benchkit.card(), "reps": args.reps, "frame": f"{W}x{H}", "spp": SPP, "max_bounces": BOUNCES,
              "models": {}}
    stream = torch.cuda.current_stream()

    def trace_work(loaded):
        driver.render(loaded, W, H, SPP, BOUNCES)
        c = driver.read_counters()
        return {"nodes_per_ray": round(c["nodes"] / c["rays"], 3), "leaves_per_ray": round(c["leaves"] / c["rays"], 3)}

    for name, cam in MODELS.items():
        loaded = benchkit.resident(name, camera=driver.look_at(**cam) if cam else None)
        n_tri, slots = loaded.n_triangles, loaded.scene.triangles.len
        p0 = driver.scene_positions(loaded)
        src = np.ctypeslib.as_array((C.c_float * (n_tri * 28)).from_address(C.addressof(loaded.model.triangles.data.contents)))
        src = src.reshape(n_tri, 28)
        src_p0 = src[:, :9].copy()
        extent = float((p0.max(axis=(1, 2)) - p0.min(axis=(1, 2))).max())
        r = {"triangles": n_tri, "slots": slots, "nodes": int(loaded.scene.bvh.nodes.len), "extent": round(extent, 3),
             "original": trace_work(loaded)}

        # 1. device refit
        sets = [torch.from_numpy(deform(p0, 0.01 * extent, 3.0 / extent)).cuda(),
                torch.from_numpy(deform(p0, 0.02 * extent, 3.0 / extent)).cuda()]
        for i in range(3):
            driver.refit_device(loaded, sets[i % 2])
        ev, wall = [], []
        for i in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(stream)
            driver.refit_device(loaded, sets[i % 2])
            e1.record(stream)
            t1 = time.perf_counter()
            torch.cuda.synchronize()
            ev.append(e0.elapsed_time(e1))
            wall.append((t1 - t0) * 1e3)
        r["refit_device_ms"] = round(float(np.median(ev)), 4)
        r["refit_device_wall_ms"] = round(float(np.median(wall)), 4)

        # 2. host refit
        host_sets = [s.cpu().numpy() for s in sets]
        wall = []
        for i in range(args.reps):
            t0 = time.perf_counter()
            driver.refit(loaded, host_sets[i % 2])
            wall.append((time.perf_counter() - t0) * 1e3)
        r["refit_host_wall_ms"] = round(float(np.median(wall)), 4)
        driver.refit(loaded, p0)

        # 3. rebuild + re-upload of the same change
        src[:, :9] = deform(src_p0.reshape(n_tri, 3, 3).transpose(2, 1, 0), 0.02 * extent, 3.0 / extent) \
            .transpose(2, 1, 0).reshape(n_tri, 9)
        init_ms, upload_ms = [], []
        for _ in range(max(3, args.reps // 4)):
            fresh = Scene()
            fresh.camera, fresh.background = loaded.scene.camera, loaded.scene.background
            t0 = time.perf_counter()
            host.scene_init(C.byref(fresh), loaded.model.triangles)
            t1 = time.perf_counter()
            gpu_check(gpu.rt_gpu_scene_upload(C.byref(fresh)))
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            init_ms.append((t1 - t0) * 1e3)
            upload_ms.append((t2 - t1) * 1e3)
            gpu.rt_gpu_scene_release(C.byref(fresh))
            host.scene_destroy(C.byref(fresh))
        r["scene_init_ms"] = round(float(np.median(init_ms)), 3)
        r["scene_upload_ms"] = round(float(np.median(upload_ms)), 3)
        src[:, :9] = src_p0

        # 4. trace work after a deformation sequence, against a fresh build of the final mesh
        steps = [0.025 * (k + 1) * extent for k in range(8)]
        for a in steps:
            driver.refit(loaded, deform(p0, a, 3.0 / extent))
        r["refit_after_sequence"] = dict(trace_work(loaded), amount=round(steps[-1], 4))
        src[:, :9] = deform(src_p0.reshape(n_tri, 3, 3).transpose(2, 1, 0), steps[-1], 3.0 / extent) \
            .transpose(2, 1, 0).reshape(n_tri, 9)
        rebuilt = driver.LoadedScene(model=loaded.model, scene=Scene(), background=loaded.background,
                                     shader_proc=loaded.shader_proc, background_proc=loaded.background_proc,
                                     path=loaded.path, n_triangles=n_tri)
        rebuilt.scene.camera, rebuilt.scene.background = loaded.scene.camera, loaded.scene.background
        host.scene_init(C.byref(rebuilt.scene), loaded.model.triangles)
        r["rebuilt"] = trace_work(rebuilt)
        gpu.rt_gpu_scene_release(C.byref(rebuilt.scene))
        host.scene_destroy(C.byref(rebuilt.scene))
        src[:, :9] = src_p0

        result["models"][name] = r
        print(json.dumps({name: r}), flush=True)
        loaded.close()

    benchkit.finish(args, result, ())


if __name__ == "__main__":
    main()
