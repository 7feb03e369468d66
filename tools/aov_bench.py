#!/usr/bin/env python
"""aov_bench.py — cost of the first-surface AOVs (rt_gpu_render_aov_device) on helmet.glb at 1920x1080, with the
renderer's own frame at the same size and sample count beside it in the same run.

    python tools/aov_bench.py [--reps 20] [--out profiles/r05_aov_bench.json]

Per sample count (1, 16, 64 spp; 8 bounces): milliseconds per call over CUDA events around `reps` back-to-back calls
after one warm-up call, for the AOV pass and for rt_gpu_render_accum_device rendering the same frame.  The AOV path
queues are 128 B per path (0.27 / 4.2 / 17 GB), far beyond the 126 MB L2.  Every AOV result of the run is checked
against the CPU oracle (oracle_render_aov): records and counters bit-exact.  The card name and power limit are read in
the same run.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np
import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
import aov_ffi as A
import helpers
import oracle_ffi
from raytracing_c_b200._ffi import gpu_check

W, H, BOUNCES = 1920, 1080, 8
SPPS = (1, 16, 64)


def main() -> None:
    args = benchkit.parser(reps=20).parse_args()
    gpu = benchkit.init()
    loaded = benchkit.resident("helmet.glb")
    oracle_scene = helpers.load("helmet.glb")
    scene = C.byref(loaded.scene)
    stream = torch.cuda.current_stream()
    aov = torch.empty(W * H * A.FLOATS, dtype=torch.float32, device="cuda")
    accum = torch.empty(W * H * 3, dtype=torch.float32, device="cuda")
    ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
    result = {"card": benchkit.card(), "model": "helmet.glb", "frame": f"{W}x{H}", "max_bounces": BOUNCES,
              "reps": args.reps, "spp": {}}

    for spp in SPPS:
        ctr.zero_()
        gpu_check(gpu.rt_gpu_render_aov_device(scene, W, H, 0, spp, BOUNCES, 0, aov.data_ptr(), ctr.data_ptr(),
                                               stream.cuda_stream))
        torch.cuda.synchronize()
        got = {"records": aov.cpu().numpy().reshape(H, W, A.FLOATS),
               "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy())))}
        want = A.oracle_aov(oracle_scene, W, H, 0, spp, BOUNCES, n_threads=os.cpu_count() or 8)
        parity = {"records": bool(np.array_equal(A.bits(got["records"]), A.bits(want["records"]))),
                  "counters": got["counters"] == want["counters"]}
        calls = (lambda: gpu_check(gpu.rt_gpu_render_aov_device(scene, W, H, 0, spp, BOUNCES, 0, aov.data_ptr(), None,
                                                                stream.cuda_stream)),
                 lambda: gpu_check(gpu.rt_gpu_render_accum_device(scene, W, H, 0, spp, BOUNCES, 0, 0, accum.data_ptr(),
                                                                  None, None, None, stream.cuda_stream)))
        ms = []
        for call in calls:
            call()                                                # warm-up: workspace, kernel modules
            torch.cuda.synchronize()
            ms.append(benchkit.per_call_ms(call, stream, args.reps))
        aov_ms, render_ms = ms
        c = got["counters"]
        r = {"aov_ms": round(aov_ms, 3), "aov_Msamples_per_s": round(W * H * spp / (aov_ms * 1e-3) / 1e6, 1),
             "render_ms": round(render_ms, 3), "render_Msamples_per_s": round(W * H * spp / (render_ms * 1e-3) / 1e6, 1),
             "aov_over_render": round(aov_ms / render_ms, 4),
             "walks_per_sample": round(c["rays"] / c["samples"], 4), "coverage": round(c["shades"] / c["samples"], 4),
             "counters": c, "parity": parity}
        result["spp"][str(spp)] = r
        print(json.dumps({f"{spp}spp": r}), flush=True)

    result["parity_ok"] = all(all(r["parity"].values()) for r in result["spp"].values())
    benchkit.finish(args, result, ("parity_ok",), oracle_scene, loaded)


if __name__ == "__main__":
    main()
