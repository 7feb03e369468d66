#!/usr/bin/env python
"""cast_rays_bench.py — throughput of radiance for caller rays (rt_gpu_cast_rays_device) on helmet.glb, with the
renderer's own frame of the same size and sample count beside it in the same run.

    python tools/cast_rays_bench.py [--reps 20] [--out profiles/r04_cast_rays_bench.json]

Workloads (8 bounces; inputs generated from fixed seeds):
  camera   one pixel-centre ray per pixel of the scene camera at 1920x1080, 64 samples each (keys = pixel): 132.7 M paths,
           beside rt_gpu_render_accum_device rendering the same frame at 64 spp
  probes   1 M rays from points uniform in the root box, directions uniform on the sphere, 256 samples each: 268 M paths
The rays themselves (50 MB and 24 MB) are read once per chunk; what each call streams is its path queues, 128 B per path
(17 GB and 34 GB), far beyond the 126 MB L2.  Per workload: Msamples/s over CUDA events around `reps` back-to-back calls
after one warm-up call, and a parity check of a seeded subset of rays, cast alone with their own keys, against the CPU
oracle (oracle_cast_rays) and against the same rays inside the full batch (sums bit-exact).  The card name and power
limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H = 1920, 1080
FRAME_SPP, PROBES, PROBE_SPP, BOUNCES = 64, 1 << 20, 256, 8
PARITY_RAYS = 1024


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in out[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()

    import torch
    import cast_rays_ffi as R
    import query_ffi as Q
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check

    gpu = gpu_lib()
    gpu_check(gpu.rt_gpu_init(0))
    loaded = driver.load_scene(os.path.join(ROOT, "assets", "models", "helmet.glb"))
    oracle_scene = driver.load_scene(os.path.join(ROOT, "assets", "models", "helmet.glb"),
                                     shader_proc=R.oracle_ffi.shader_proc(), background_proc=R.oracle_ffi.background_proc())
    driver.register_callbacks(loaded)
    gpu_check(gpu.rt_gpu_scene_upload(C.byref(loaded.scene)))
    scene = C.byref(loaded.scene)
    stream = torch.cuda.current_stream()
    dev = "cuda"
    result = {"card": card(), "model": "helmet.glb", "max_bounces": BOUNCES, "reps": args.reps, "workloads": {}}

    def cast(rays, keys, samples, radiance, counters=None):
        return gpu.rt_gpu_cast_rays_device(scene, rays.data_ptr(), keys.data_ptr() if keys is not None else None,
                                           rays.shape[0], 0, samples, BOUNCES, 0, 0, radiance.data_ptr(), None,
                                           counters.data_ptr() if counters is not None else None, stream.cuda_stream)

    def timed(fn):
        gpu_check(fn())                                           # warm-up: workspace, kernel modules
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.reps):
            gpu_check(fn())
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.reps

    def measure(name, rays, keys, samples):
        n = rays.shape[0]
        rad = torch.empty((n, 3), dtype=torch.float32, device=dev)
        ctr = torch.zeros(8, dtype=torch.int64, device=dev)
        gpu_check(cast(rays, keys, samples, rad, ctr))
        torch.cuda.synchronize()
        c = dict(zip(R.oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy())))
        ms = timed(lambda: cast(rays, keys, samples, rad))
        w = {"rays": n, "samples_per_ray": samples, "paths": n * samples, "ms": round(ms, 2),
             "Msamples_per_s": round(n * samples / (ms * 1e-3) / 1e6, 1), "rays_traced_per_path": round(c["rays"] / (n * samples), 3),
             "counters_samples_ok": c["samples"] == n * samples}
        # parity: a seeded subset cast alone with its own keys, against the oracle and the full batch
        idx = np.sort(np.random.default_rng(7).choice(n, size=min(PARITY_RAYS, n), replace=False))
        sub_r = rays[torch.from_numpy(idx).to(dev)].cpu().numpy()
        sub_k = (keys.cpu().numpy().view(np.uint32)[idx] if keys is not None else idx.astype(np.uint32))
        got = R.device_cast_rays(loaded, sub_r, samples, BOUNCES, 0, 0, sub_k, per_sample=False)
        want = R.oracle_cast_rays(oracle_scene, sub_r, samples, BOUNCES, 0, 0, sub_k, n_threads=os.cpu_count() or 8)
        w["parity"] = {"rays": len(idx), "oracle": bool(np.array_equal(R.bits(got["radiance"]), R.bits(want["radiance"]))),
                       "counters": got["counters"] == want["counters"],
                       "in_full_batch": bool(np.array_equal(R.bits(rad.cpu().numpy()[idx]), R.bits(got["radiance"])))}
        result["workloads"][name] = w
        print(json.dumps({name: w}), flush=True)
        return rad

    # (a) pixel-centre camera rays, keys = pixel; the renderer's frame at the same size and spp beside it
    cam = torch.from_numpy(Q.camera_rays(loaded.scene, W, H)).to(dev).contiguous()
    pixels = torch.arange(W * H, dtype=torch.int32, device=dev)
    measure("camera_1920x1080x64", cam, pixels, FRAME_SPP)
    del cam, pixels
    torch.cuda.empty_cache()
    accum = torch.empty(W * H * 3, dtype=torch.float32, device=dev)
    ms = timed(lambda: gpu.rt_gpu_render_accum_device(scene, W, H, 0, FRAME_SPP, BOUNCES, 0, 0, accum.data_ptr(), None, None,
                                                      None, stream.cuda_stream))
    result["renderer_frame"] = {"frame": f"helmet.glb {W}x{H}, {FRAME_SPP} spp, {BOUNCES} bounces (rt_gpu_render_accum_device)",
                                "ms": round(ms, 2), "Msamples_per_s": round(W * H * FRAME_SPP / (ms * 1e-3) / 1e6, 1)}
    print(json.dumps({"renderer_frame": result["renderer_frame"]}), flush=True)
    del accum
    torch.cuda.empty_cache()

    # (b) probe rays from interior points
    g = torch.Generator(device=dev).manual_seed(2026)
    lo, hi = Q.root_box(loaded.scene)
    o = torch.tensor(lo, device=dev) + torch.rand(PROBES, 3, device=dev, generator=g) * torch.tensor(hi - lo, device=dev)
    d = torch.randn(PROBES, 3, device=dev, generator=g)
    d = d / d.norm(dim=1, keepdim=True)
    measure("probes_1Mx256", torch.cat([o, d], dim=1).contiguous(), None, PROBE_SPP)

    result["camera_vs_renderer"] = round(result["workloads"]["camera_1920x1080x64"]["Msamples_per_s"] /
                                         result["renderer_frame"]["Msamples_per_s"], 3)
    result["parity_ok"] = all(all(v for k, v in w["parity"].items() if k != "rays") and w["counters_samples_ok"]
                              for w in result["workloads"].values())
    print(json.dumps({"card": result["card"], "camera_vs_renderer": result["camera_vs_renderer"],
                      "parity_ok": result["parity_ok"]}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    oracle_scene.close()
    loaded.close()
    if not result["parity_ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
