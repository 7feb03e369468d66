#!/usr/bin/env python
"""query_bench.py — throughput of the batched ray queries (rt_gpu_closest_hit_device / rt_gpu_occluded_device) on
helmet.glb, with the renderer's own trace rate of the headline frame beside them.

    python tools/query_bench.py [--reps 20] [--out profiles/query_bench.json]

Families (every array generated on the device from a fixed seed; 1920x1080x16 = 33.2 M rays = 796 MB of rays, far
beyond the 126 MB L2, so no timed pass reads its rays from L2):
  camera   pinhole rays from the scene camera through 16 uniformly jittered points per pixel (unit directions)
  ao       from the camera rays' hits, four per hit: origin = point + EPSILON * normal_geo (normal_geo facing the
           incoming ray), cosine-distributed directions about it; run with t_max = inf and with t_max = 0.5
  interior origins uniform in the root box, directions uniform on the sphere
Per family and query: Mrays/s over CUDA events around `reps` back-to-back calls after one warm-up call, nodes and leaves
per ray from the kernels' counters, and a parity check of 65 536 seeded rays against the CPU oracle (every field and the
four counters bit-exact).  The card name and power limit are read in the same run.
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

W, H, SPP_RAYS = 1920, 1080, 16
AO_PER_HIT = 4
EPS = 0.0001
PARITY_RAYS = 65536


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
    import query_ffi as Q
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check

    gpu = gpu_lib()
    gpu_check(gpu.rt_gpu_init(0))
    loaded = driver.load_scene(os.path.join(ROOT, "assets", "models", "helmet.glb"))
    driver.register_callbacks(loaded)
    gpu_check(gpu.rt_gpu_scene_upload(C.byref(loaded.scene)))
    scene = C.byref(loaded.scene)
    stream = torch.cuda.current_stream()
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(2026)
    result = {"card": card(), "model": "helmet.glb", "reps": args.reps, "families": {}}

    def query(rays, t_max, kind, hits=None, surf=None, occ=None, ctr=None):
        n = rays.shape[0]
        tp = t_max.data_ptr() if t_max is not None else None
        cp = ctr.data_ptr() if ctr is not None else None
        if kind == "occluded":
            return gpu.rt_gpu_occluded_device(scene, rays.data_ptr(), tp, n, occ.data_ptr(), cp, stream.cuda_stream)
        return gpu.rt_gpu_closest_hit_device(scene, rays.data_ptr(), tp, n, hits.data_ptr(),
                                             surf.data_ptr() if (kind == "closest_surface") else None, cp, stream.cuda_stream)

    def measure(name, rays, t_max):
        n = rays.shape[0]
        hits = torch.empty((n, 4), dtype=torch.float32, device=dev)
        surf = torch.empty((n, 11), dtype=torch.float32, device=dev)
        occ = torch.empty(n, dtype=torch.uint8, device=dev)
        fam = {"rays": n, "ray_bytes": n * 24}
        for kind in ("closest", "closest_surface", "occluded"):
            ctr = torch.zeros(4, dtype=torch.int64, device=dev)
            gpu_check(query(rays, t_max, kind, hits, surf, occ, ctr))          # warm-up, and the counters of one pass
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.reps):
                gpu_check(query(rays, t_max, kind, hits, surf, occ))
            e1.record(stream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.reps
            c = ctr.cpu().numpy()
            fam[kind] = {"ms": round(ms, 3), "Mrays_per_s": round(n / (ms * 1e-3) / 1e6, 1),
                         "nodes_per_ray": round(float(c[1]) / n, 3), "leaves_per_ray": round(float(c[2]) / n, 3),
                         "accepts_per_ray": round(float(c[3]) / n, 3)}
        near_hit = (hits[:, 3].view(torch.int32) >= 0)
        fam["hit_fraction"] = round(float(near_hit.float().mean()), 4)
        fam["occluded_equals_closest_slot_ge_0"] = bool(torch.equal(occ.bool(), near_hit))
        fam["occluded_vs_closest_time"] = round(fam["occluded"]["ms"] / fam["closest"]["ms"], 3)

        # parity: a seeded subset, queried on its own on the GPU (for its counters) and by the oracle
        idx = torch.from_numpy(np.sort(np.random.default_rng(7).choice(n, size=min(PARITY_RAYS, n), replace=False))).to(dev)
        sr = rays[idx].contiguous()
        st = t_max[idx].contiguous() if t_max is not None else None
        m = sr.shape[0]
        sh, ss, so = (torch.empty((m, 4), dtype=torch.float32, device=dev), torch.empty((m, 11), dtype=torch.float32, device=dev),
                      torch.empty(m, dtype=torch.uint8, device=dev))
        c1, c2 = torch.zeros(4, dtype=torch.int64, device=dev), torch.zeros(4, dtype=torch.int64, device=dev)
        gpu_check(query(sr, st, "closest_surface", sh, ss, so, c1))
        gpu_check(query(sr, st, "occluded", sh, ss, so, c2))
        torch.cuda.synchronize()
        rn, tn = sr.cpu().numpy(), st.cpu().numpy() if st is not None else None
        want = Q.oracle_query(loaded, rn, tn, surface=True, n_threads=os.cpu_count() or 8)
        want_any = Q.oracle_query(loaded, rn, tn, any_hit=True, n_threads=os.cpu_count() or 8)
        h = sh.cpu().numpy()
        full = hits[idx].cpu().numpy()
        checks = {
            "hits": all(np.array_equal(Q.bits(h[:, k]), Q.bits(want[f])) for k, f in enumerate(("t", "u", "v")))
                    and np.array_equal(h[:, 3].view(np.int32), want["slot"]),
            "hits_in_full_batch": np.array_equal(Q.bits(full), Q.bits(h)),
            "surface": np.array_equal(Q.bits(ss.cpu().numpy()), Q.bits(want["surface"])),
            "occluded": np.array_equal(so.cpu().numpy().astype(bool), want_any["occluded"]),
            "counters": dict(zip(Q.QUERY_COUNTERS, map(int, c1.cpu().numpy()))) == want["counters"]
                        and dict(zip(Q.QUERY_COUNTERS, map(int, c2.cpu().numpy()))) == want_any["counters"],
        }
        fam["parity"] = {"rays": m, **{k: bool(v) for k, v in checks.items()}}
        result["families"][name] = fam
        print(json.dumps({name: fam}), flush=True)
        return hits, surf

    # (a) camera rays: 16 jittered rays per pixel through the pinhole (the renderer's camera model without its hash)
    sc = loaded.scene
    mtx = torch.tensor([[sc.camera.view_matrix[r][c] for c in range(4)] for r in range(3)], dtype=torch.float32, device=dev)
    n = W * H * SPP_RAYS
    pix = torch.arange(n, device=dev) // SPP_RAYS
    jx, jy = torch.rand(n, device=dev, generator=g), torch.rand(n, device=dev, generator=g)
    ux = ((pix % W).float() + jx) * (2.0 / W) - 1.0
    uy = ((pix // W).float() + jy) * (2.0 / H) - 1.0
    cam = torch.stack([ux * (W / H), -uy, torch.full_like(ux, -sc.camera.focal_length)], dim=1)
    d = cam @ mtx[:, :3].T
    d = d / d.norm(dim=1, keepdim=True)
    rays = torch.cat([mtx[:, 3].expand(n, 3), d], dim=1).contiguous()
    del pix, jx, jy, ux, uy, cam, d
    hits, surf = measure("camera", rays, None)

    # (b) ambient-occlusion rays from those hits
    hit = hits[:, 3].view(torch.int32) >= 0
    p, ng, din = (surf[hit, 0:3].repeat_interleave(AO_PER_HIT, dim=0), surf[hit, 6:9].repeat_interleave(AO_PER_HIT, dim=0),
                  rays[hit, 3:6].repeat_interleave(AO_PER_HIT, dim=0))
    ng = torch.where(((ng * din).sum(dim=1, keepdim=True) > 0), -ng, ng)
    ng = ng / ng.norm(dim=1, keepdim=True)
    m = p.shape[0]
    r1, r2 = torch.rand(m, device=dev, generator=g), torch.rand(m, device=dev, generator=g)
    phi, sr = 2 * np.pi * r1, torch.sqrt(r2)
    local = torch.stack([sr * torch.cos(phi), sr * torch.sin(phi), torch.sqrt(1 - r2)], dim=1)
    helper = torch.where((ng[:, 0].abs() > 0.9)[:, None], torch.tensor([0.0, 1.0, 0.0], device=dev), torch.tensor([1.0, 0.0, 0.0], device=dev))
    t1 = torch.linalg.cross(helper, ng)
    t1 = t1 / t1.norm(dim=1, keepdim=True)
    t2 = torch.linalg.cross(ng, t1)
    ao_dir = local[:, 0:1] * t1 + local[:, 1:2] * t2 + local[:, 2:3] * ng
    ao = torch.cat([p + EPS * ng, ao_dir], dim=1).contiguous()
    del hits, surf, rays, hit, p, ng, din, r1, r2, phi, sr, local, helper, t1, t2, ao_dir
    torch.cuda.empty_cache()
    measure("ao_inf", ao, None)
    measure("ao_0.5", ao, torch.full((ao.shape[0],), 0.5, dtype=torch.float32, device=dev))
    del ao
    torch.cuda.empty_cache()

    # (c) interior rays
    lo, hi = Q.root_box(loaded.scene)
    o = torch.tensor(lo, device=dev) + torch.rand(n, 3, device=dev, generator=g) * torch.tensor(hi - lo, device=dev)
    d = torch.randn(n, 3, device=dev, generator=g)
    d = d / d.norm(dim=1, keepdim=True)
    measure("interior", torch.cat([o, d], dim=1).contiguous(), None)
    del o, d
    torch.cuda.empty_cache()

    # reference point: the headline frame (1920x1080, 1024 spp, 8 bounces) rendered once with per-stage timing; the
    # renderer's own trace rate = its rays counter over the CUDA-event time of its trace launches
    driver.render(loaded, W, H, 16, 8)                        # warm-up: workspace, kernel modules
    gpu.rt_gpu_stage_profile_enable(1)
    driver.render(loaded, W, H, 1024, 8)
    stage_ms, stage_n = (C.c_double * 4)(), (C.c_int64 * 4)()
    gpu_check(gpu.rt_gpu_stage_profile_read(C.byref(stage_ms), C.byref(stage_n)))
    gpu.rt_gpu_stage_profile_enable(0)
    ctr = driver.read_counters()
    result["renderer_trace"] = {"frame": "helmet.glb 1920x1080, 1024 spp, 8 bounces", "rays": ctr["rays"],
                                "trace_ms": round(float(stage_ms[0]), 2), "trace_launches": int(stage_n[0]),
                                "Mrays_per_s": round(ctr["rays"] / (float(stage_ms[0]) * 1e-3) / 1e6, 1),
                                "nodes_per_ray": round(ctr["nodes"] / ctr["rays"], 3),
                                "leaves_per_ray": round(ctr["leaves"] / ctr["rays"], 3)}
    print(json.dumps({"renderer_trace": result["renderer_trace"]}), flush=True)
    result["parity_ok"] = all(all(v for k, v in f["parity"].items() if k != "rays") for f in result["families"].values())
    result["occluded_not_slower_at_inf"] = all(f["occluded_vs_closest_time"] <= 1.0 for k, f in result["families"].items()
                                               if k in ("camera", "ao_inf", "interior"))
    print(json.dumps({"card": result["card"], "parity_ok": result["parity_ok"],
                      "occluded_not_slower_at_inf": result["occluded_not_slower_at_inf"]}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    loaded.close()
    if not result["parity_ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
