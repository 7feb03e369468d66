#!/usr/bin/env python
"""bench.py — Msamples/s (pixel*spp/s) of the path-tracing hot path on helmet.glb 1920x1080.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU renderer on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed frame to DIR/*.npy

A step = one full frame of BASELINE.json's headline config (helmet.glb, 1920x1080, 1024 spp, 8 bounces, synthetic
environment) rendered by N GPUs, one process per GPU: every rank renders the share of the frame the library's policy
gives it (rt_gpu_render_shard_device: sample ranges, or the reference's 32x32 chunks when the sample batches do not
divide evenly), rank 0 combines the f32 accumulators with the library's fused reduce+resolve kernel, which reads the
peers' buffers in place over NVLink (CUDA IPC; --reduce nccl swaps in an NCCL reduce), and resolves to u8 sRGB.
The total work is fixed => "scaling": "strong".

Keys beyond the base contract: `roofline` (rt_trace_kernel — BVH traversal, the dominant kernel of the wavefront —
against the measured FP32 issue ceiling, the bound SURVEY 8d derives: not HBM, not tensor; launch time measured live
with CUDA events around every launch of the timed region; `executed` / `traffic` from the committed ncu capture of the
same command; `resolve` / `denoise` = the two HBM-streaming kernels), `parity` (rank 0, after the timed region: the
REDUCED accumulator of the last timed step against the CPU oracle on 4096 random pixels + 4 scanlines at the full sample
count), `cpu_baseline` (the reference's renderer on the host cores on a bounded sample), `e2e` (the same frame with the
scene re-uploaded from host memory and the image read back every step, itemised).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MODELS = os.path.join(ROOT, "assets", "models")
METRIC = "Msamples/s (pixel*spp/s), helmet.glb 1920x1080"
UNIT = "Msamples/s"
# BASELINE.json's other configs, selectable with --workload for the multi-GPU sweeps (the default, and the only
# one the driver's contract names, is the headline helmet frame)
WORKLOADS = {
    "helmet1080p": dict(model="helmet.glb", width=1920, height=1080, spp=1024, camera=None,
                        describe="helmet.glb (15452 triangles, depth-4 8-ary BVH, 4x 2048^2 textures)"),
    "tower4k": dict(model="tower.obj", width=3840, height=2160, spp=1024,
                    camera=dict(eye=(0.0, 12.5, 40.0), target=(0.0, 12.5, 0.0)),
                    describe="tower.obj (4320 triangles, depth-4 8-ary BVH, default material), camera (0,12.5,40)->(0,12.5,0)"),
    "spheres": dict(model="spheres.glb", width=1024, height=1024, spp=1024, camera=None,
                    describe="spheres.glb (4800 triangles, 5 factor-only materials), camera from the file"),
}
COUNTER_NAMES = ["rays", "nodes", "leaves", "accepts", "shades", "misses", "passthrough", "samples"]

# FLOP model of SURVEY §8(d): per box test 25 lane-ops x 8, per triangle 57 x 8, +33 per accepted
# hit, ~700 per textured shade, ~90 per environment lookup, 40 per primary ray.
FLOP_NODE, FLOP_LEAF, FLOP_ACCEPT, FLOP_SHADE, FLOP_ENV, FLOP_RAYGEN = 200.0, 456.0, 33.0, 700.0, 90.0, 40.0
# cache-level bytes per unit of work (same section): 192 B per node, 288 B per leaf, 112 B per
# accepted record, 4 taps x 4 textures x 4 B + 80 B material per shade
BYTES_NODE, BYTES_LEAF, BYTES_ACCEPT, BYTES_SHADE = 192.0, 288.0, 112.0, 144.0
DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs writes at most this much


def algorithmic_flops(c: dict) -> float:
    return (FLOP_RAYGEN * c["samples"] + FLOP_NODE * c["nodes"] + FLOP_LEAF * c["leaves"] +
            FLOP_ACCEPT * c["accepts"] + FLOP_SHADE * c["shades"] + FLOP_ENV * c["misses"])


def workload_config(args, parallelism: str) -> dict:
    wl = WORKLOADS[args.workload]
    return {"workload": f"{wl['model']} {args.width}x{args.height} {args.spp}spp max_bounces {args.bounces}",
            "model": wl["describe"],
            "environment": "procedural equirect 2048x1024 (reference background.png is not in its tree)",
            "seed_mode": "per-(pixel,sample) rt_path_seed, user_seed 0", "parallelism": parallelism}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML, else nvidia-smi)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_flag = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {getattr(pynvml, k): k for k in dir(pynvml) if k.startswith("nvmlClocksThrottleReason")
                     or k.startswith("nvmlClocksEventReason")}
            while not self._stop_flag.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if isinstance(bit, int) and bit and mask & bit and "None" not in name and "All" not in name:
                            self.reasons.add(name.replace("nvmlClocksThrottleReason", "").replace("nvmlClocksEventReason", ""))
                except Exception:
                    pass
                time.sleep(0.2)
        except Exception:
            import subprocess
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            while not self._stop_flag.is_set():
                try:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                    self.samples.append(int(out[0]))
                    self.max_mhz = int(out[1])
                    for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], out[2:]):
                        if "Active" in v and "Not" not in v:
                            self.reasons.add(name)
                except Exception:
                    pass
                time.sleep(0.2)

    def finish(self) -> dict:
        self._stop_flag.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "n_samples": len(s)}


def metric_name(args) -> str:
    return METRIC if args.workload == "helmet1080p" else \
        f"Msamples/s (pixel*spp/s), {WORKLOADS[args.workload]['model']} {args.width}x{args.height}"


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def load_workload(args, **procs):
    from raytracing_c_b200 import driver
    wl = WORKLOADS[args.workload]
    cam = driver.look_at(**wl["camera"]) if wl["camera"] else None
    return driver.load_scene(os.path.join(MODELS, wl["model"]), camera=cam, **procs)


class CpuRenderer:
    """The CPU arm: the reference's OWN raytracer.c / driver.c (oracle/_ref/libref.so — its sources compiled
    unmodified where they lie, over the stand-in for its un-vendored stdlib; built by oracle/Makefile from
    the reference checkout RT_REFERENCE_DIR names) when that file is present, `kind: "reference"`;
    otherwise the oracle port, `kind: "port"`.  Either way N host threads enter render_thread_proc with one
    context and pull 32x32 chunks from its atomic counter, exactly as the reference's driver starts them
    (driver.c:793-803)."""

    def __init__(self, args):
        import oracle_ffi
        self.kind, self._ref = "port", None
        try:
            import ref_ffi
            if os.path.exists(ref_ffi.REF_LIB):
                self._ref = ref_ffi.lib()
                self.kind = "reference"
        except Exception:
            self._ref = None
        if self._ref is not None:
            procs = dict(shader_proc=self._ref.ref_shader_proc(), background_proc=self._ref.ref_background_proc())
        else:
            procs = dict(shader_proc=oracle_ffi.shader_proc(), background_proc=oracle_ffi.background_proc())
        self.loaded = load_workload(args, **procs)
        self.args, self.cores = args, host_threads()
        self.what = ("the reference's raytracer.c + driver.c (oracle/_ref; its own per-thread RNG stream and rsqrt_ps), AVX2" if self._ref is not None
                     else "AVX2 oracle port") + f", reference chunk scheduler, {self.cores} threads"

    def render(self, spp: int) -> float:
        """Seconds for one frame at `spp` samples per pixel."""
        import numpy as np
        a = self.args
        t0 = time.perf_counter()
        if self._ref is None:
            import oracle_ffi
            oracle_ffi.render(self.loaded, a.width, a.height, spp, a.bounces, n_threads=self.cores, want_accum=False)
        else:
            from raytracing_c_b200._ffi import RenderingContext
            from raytracing_c_b200.driver import image_view
            pixels = np.zeros((a.height, a.width, 3), dtype=np.uint8)
            ctx = RenderingContext()
            ctx.image = image_view(pixels)
            ctx.scene = C.pointer(self.loaded.scene)
            ctx.samples, ctx.max_bounces, ctx.n_threads, ctx._current_chunk = spp, a.bounces, self.cores, 0
            threads = [threading.Thread(target=self._ref.render_thread_proc, args=(C.byref(ctx),)) for _ in range(self.cores)]
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            assert ctx.n_threads == 0
        return time.perf_counter() - t0

    def close(self):
        self.loaded.close()


def cpu_reference_rate(args, target_seconds: float = 15.0):
    """Times the CPU arm on all host threads on a bounded sample of the SAME frame: full resolution, reduced spp
    (the rate does not depend on spp)."""
    cpu = CpuRenderer(args)
    try:
        t1 = cpu.render(1)
        spp = max(1, min(256, int(target_seconds / max(t1, 1e-3))))
        dt = cpu.render(spp)
    finally:
        cpu.close()
    rate = args.width * args.height * spp / dt / 1e6
    return {"value": round(rate, 4), "unit": UNIT, "cores": cpu.cores, "kind": cpu.kind,
            "sample": f"{WORKLOADS[args.workload]['model']} {args.width}x{args.height} at {spp} spp ({dt:.1f} s of CPU work; "
                      f"{cpu.what})"}, spp, dt


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpu = CpuRenderer(args)
    spp = args.cpu_spp
    per_step = []
    try:
        for i in range(args.warmup + args.steps):
            dt = cpu.render(spp)
            if i >= args.warmup:
                per_step.append(dt)
    finally:
        cpu.close()
    total = sum(per_step)
    value = args.width * args.height * spp * len(per_step) / total / 1e6
    config = workload_config(args, "cpu")
    config["sample"] = (f"each step renders the same frame at {spp} spp instead of {args.spp} (the rate is spp-independent: "
                        f"every sample is an independent path, raytracer.c:687-696)")
    line = {"impl": "reference", "metric": metric_name(args), "value": round(value, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / len(per_step), 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": cpu.cores, "kind": cpu.kind,
                             "sample": f"each step = the same frame at {spp} spp instead of {args.spp} "
                                       f"(rate is spp-independent); {cpu.what}"},
            "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def parity_mask(W, H, n_random=4096, seed=2026):
    """The pixels of the frame that are checked against the oracle after the timed region: 4096 random ones and
    four full scanlines (per-(pixel,sample) seeds make every pixel independent of the others)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    mask = np.zeros((H, W), dtype=np.uint8)
    mask.reshape(-1)[rng.choice(W * H, size=min(n_random, W * H), replace=False)] = 1
    for y in (H // 8, H // 3, H // 2, (2 * H) // 3):
        mask[y, :] = 1
    return mask


def parity_against_oracle(args, accum_host, pixels_host):
    """rank 0, after the timed region: the REDUCED f32 accumulator of the last step (all GPUs' shares combined) and
    the resolved u8 image against the CPU oracle on `parity_mask` at the full sample count."""
    import numpy as np
    import oracle_ffi
    W, H, SPP, B = args.width, args.height, args.spp, args.bounces
    procs = dict(shader_proc=oracle_ffi.shader_proc(), background_proc=oracle_ffi.background_proc())
    loaded = load_workload(args, **procs)
    try:
        mask = parity_mask(W, H)
        t0 = time.perf_counter()
        ref = oracle_ffi.render(loaded, W, H, SPP, B, n_threads=host_threads(), pixel_mask=mask)
        dt = time.perf_counter() - t0
    finally:
        loaded.close()
    sel = mask.astype(bool)
    a, b = accum_host.reshape(H, W, 3)[sel].astype(np.float64), ref["accum"][sel].astype(np.float64)
    rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-6)
    u8 = (pixels_host.reshape(H, W, 3)[sel] != ref["pixels"][sel])
    d8 = pixels_host.reshape(H, W, 3)[sel].astype(np.float64) / 255 - ref["pixels"][sel].astype(np.float64) / 255
    return {"pixels": int(sel.sum()), "spp": SPP, "max_rel": float(rel.max()), "frac_within_1e-3": float((rel <= 1e-3).mean()),
            "median_rel": float(np.median(rel)), "srgb_rmse": float(np.sqrt(np.mean(d8 ** 2))),
            "bit_identical": bool(np.array_equal(accum_host.reshape(H, W, 3)[sel], ref["accum"][sel])),
            "u8_mismatch": int(u8.any(axis=-1).sum()), "oracle_s": round(dt, 2),
            "what": "NCCL/NVLink-reduced f32 accumulator of the last timed step vs the CPU oracle: 4096 random pixels + 4 scanlines"}


def film_kernel_rates(gpu, gpu_check, torch, W, H, SPP, sptr, peak_gbs):
    """The two HBM-streaming kernels of the frame, timed alone with CUDA events (burst peak applies)."""
    dev = torch.device("cuda", torch.cuda.current_device())
    accum = torch.rand(H * W * 3, dtype=torch.float32, device=dev) * SPP
    px, px2 = torch.zeros(H * W * 3, dtype=torch.uint8, device=dev), torch.zeros(H * W * 3, dtype=torch.uint8, device=dev)
    ptrs = (C.c_void_p * 1)(accum.data_ptr())
    out = {}
    for name, call, nbytes in (
            ("resolve", lambda: gpu.rt_gpu_reduce_resolve_device(ptrs, 1, None, W, H, SPP, px.data_ptr(), W, 3, sptr), W * H * 15),
            ("denoise", lambda: gpu.rt_gpu_denoise_device(px.data_ptr(), px2.data_ptr(), W, H, W, W, 3, sptr), W * H * 6)):
        for _ in range(3):
            gpu_check(call())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            gpu_check(call())
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "GB/s": round(gbs, 1),
                     "frac_of_hbm_peak": round(gbs / peak_gbs, 4), "note": "back-to-back launches: the 25 MB working set stays in the 126 MB L2"}
    return out


def dump_outputs(out_dir: str, frames: dict, seed: int = 2026) -> None:
    """Writes every (H, W, 3) array of `frames` as out_dir/<name>.npy in float32: whole when they fit in DUMP_BYTES
    together, else the same seeded sample of pixels from each, (n, 3), with their row-major indices in
    pixel_index.npy (float64, exact).  Two builds given the same arguments can then be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in frames.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        h, w = next(iter(arrays.values())).shape[:2]
        n = (DUMP_BYTES - 4096) // (total // (h * w) + 8)
        idx = np.sort(np.random.default_rng(seed).choice(h * w, size=n, replace=False))
        arrays = {k: a.reshape(h * w, -1)[idx] for k, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def measured_peaks() -> dict:
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def run_gpu(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import SPLIT_AUTO, SPLIT_CHUNKS, SPLIT_SAMPLES, gpu_check

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gpu = gpu_lib()
    gpu_check(gpu.rt_gpu_init(local))
    dev = torch.device("cuda", local)

    W, H, SPP, B = args.width, args.height, args.spp, args.bounces
    split_req = {"auto": SPLIT_AUTO, "samples": SPLIT_SAMPLES, "chunks": SPLIT_CHUNKS}[args.split]
    slice_spp = args.slice

    driver.use_pinned_host_buffers(not args.pageable)      # scene buffers in pinned memory: H2D is a DMA from them
    t0 = time.perf_counter()
    loaded = load_workload(args)               # Shader/Background procs = the GPU library's own identities
    t_load = time.perf_counter() - t0
    driver.register_callbacks(loaded)
    scene_ref = C.byref(loaded.scene)
    t0 = time.perf_counter()
    gpu_check(gpu.rt_gpu_scene_upload(scene_ref))
    torch.cuda.synchronize()
    t_upload = time.perf_counter() - t0
    scene_bytes = int(gpu.rt_gpu_scene_device_bytes(scene_ref))
    upload_bytes = int(gpu.rt_gpu_scene_upload_bytes(scene_ref))

    # the accumulator and the counters are the library's own buffers (cudaMalloc: exportable over CUDA IPC)
    accum_ptr, ctr_ptr = C.c_void_p(), C.c_void_p()
    gpu_check(gpu.rt_gpu_accum_buffer(W, H, C.byref(accum_ptr)))
    gpu_check(gpu.rt_gpu_counters_buffer(C.byref(ctr_ptr)))
    total = torch.zeros(H * W * 3, dtype=torch.float32, device=dev)        # rank 0: the combined accumulator
    pixels = torch.zeros(H * W * 3, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)      # a real stream (not the legacy default one): stream attributes apply
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)
    launches = {"n": 0}
    mode_used = C.c_int32(SPLIT_SAMPLES)

    # ---- the cross-GPU film.  Default: rank 0's fused reduce+resolve kernel reads the other ranks' accumulators in
    # place over NVLink (CUDA IPC mappings); two 4-byte NCCL all-reduces fence it (all shares finished / all shares read).
    # --reduce nccl: dist.reduce of the 24.9 MB accumulators, then the resolve kernel.
    reduce_how = "single GPU: resolve only"
    part_ptrs = None
    if world > 1:
        reduce_how = "nccl"
        if args.reduce == "p2p":
            handle = C.create_string_buffer(64)
            ok = gpu.rt_gpu_ipc_export(accum_ptr, handle) == 0
            handles = [None] * world
            dist.all_gather_object(handles, handle.raw if ok else None)
            if all(h is not None for h in handles):
                if rank == 0:
                    ptrs = [accum_ptr.value]
                    for r in range(1, world):
                        p = C.c_void_p()
                        if gpu.rt_gpu_ipc_open(handles[r], C.byref(p)) != 0:
                            ptrs = None
                            break
                        ptrs.append(p.value)
                    part_ptrs = (C.c_void_p * world)(*ptrs) if ptrs else None
                opened = [rank != 0 or part_ptrs is not None]
                dist.broadcast_object_list(opened, src=0)
                if opened[0]:
                    reduce_how = "p2p"
                elif rank == 0:
                    sys.stderr.write("bench.py: CUDA IPC mapping failed (%s); falling back to the NCCL reduce\n" %
                                     gpu.rt_gpu_last_error().decode())
    if reduce_how == "nccl":
        accum_t = torch.zeros(H * W * 3, dtype=torch.float32, device=dev)   # NCCL needs a torch tensor: the render writes into it
        accum_ptr = C.c_void_p(accum_t.data_ptr())

    def fence():
        dist.all_reduce(flag)            # stream-ordered: completes on a rank only after every rank reached it

    def step(timed: bool):
        flush.zero_()                                              # L2 flush between steps
        n0 = gpu.rt_gpu_last_launches()
        # one call: the library picks this rank's share of the frame and cuts it into wavefront chunks
        gpu_check(gpu.rt_gpu_render_shard_device(scene_ref, W, H, SPP, B, 0, rank, world, split_req, C.byref(mode_used),
                                                 accum_ptr, ctr_ptr if timed else None, sptr))
        if world == 1:
            one = (C.c_void_p * 1)(accum_ptr.value)
            gpu_check(gpu.rt_gpu_reduce_resolve_device(one, 1, total.data_ptr(), W, H, SPP, pixels.data_ptr(), W, 3, sptr))
        elif reduce_how == "p2p":
            fence()
            if rank == 0:
                gpu_check(gpu.rt_gpu_reduce_resolve_device(part_ptrs, world, total.data_ptr(), W, H, SPP, pixels.data_ptr(), W, 3, sptr))
            fence()
        else:
            dist.reduce(accum_t, dst=0, op=dist.ReduceOp.SUM)      # NCCL over NVLink: 24.9 MB f32
            if rank == 0:
                total.copy_(accum_t)
                gpu_check(gpu.rt_gpu_resolve_device(accum_t.data_ptr(), W, H, SPP, pixels.data_ptr(), W, 3, sptr))
        launches["n"] += gpu.rt_gpu_last_launches() - n0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    driver.set_options(fast_math=args.fast)
    for _ in range(args.warmup):
        step(False)
    barrier()
    launches["n"] = 0
    gpu_check(gpu.rt_gpu_counters_reset())        # the library's counter block is only ever added to
    gpu.rt_gpu_stage_profile_enable(1)
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step(True)
    e1.record(stream)
    barrier()
    clocks = sampler.finish()
    timed_launches = launches["n"]
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    ms_per_step = total_ms / args.steps
    value = W * H * SPP / (ms_per_step * 1e-3) / 1e6

    # dominant kernel: rt_trace_kernel (closest-hit BVH traversal; primary and bounce launches are one template),
    # CUDA-event time of every launch in the timed region on this rank
    stage_ms, stage_n = (C.c_double * 4)(), (C.c_int64 * 4)()
    gpu_check(gpu.rt_gpu_stage_profile_read(C.byref(stage_ms), C.byref(stage_n)))
    gpu.rt_gpu_stage_profile_enable(0)
    stage_names = ["trace", "miss", "shade", "accumulate"]
    kern_ms, n_kern = float(stage_ms[0]), int(stage_n[0])
    raw16 = (C.c_uint64 * 16)()
    gpu_check(gpu.rt_gpu_read_counters_ex(raw16))
    raw = [int(v) for v in raw16]
    ctr = dict(zip(COUNTER_NAMES, raw[:8]))
    root_misses, primary_rays = raw[8], raw[9]
    trace_flops = (FLOP_RAYGEN * primary_rays + FLOP_NODE * ctr["nodes"] + FLOP_LEAF * ctr["leaves"] +
                   FLOP_ACCEPT * ctr["accepts"])
    # the same with a root-union miss counted as the 18 lane-ops it costs here instead of a 200-op node visit
    trace_flops_strict = trace_flops - (FLOP_NODE - 18.0) * root_misses
    flops_per_launch = trace_flops / max(n_kern, 1)
    launch_s = kern_ms / max(n_kern, 1) * 1e-3
    achieved_tflops = flops_per_launch / launch_s / 1e12
    peak_ops = float(gpu.rt_gpu_measure_fp32_issue())
    peaks = measured_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6551.0))
    # per-launch DRAM traffic and executed instructions come from the ncu capture of THIS command committed under
    # profiles/ (tools/ncu_traffic.py writes the JSON from the CSV next to it); absent => null
    traffic, ncu_info = None, None
    prof = os.path.join(ROOT, "profiles", "r02_trace_traffic.json")
    if os.path.exists(prof):
        try:
            ncu_info = json.load(open(prof))
            traffic = ncu_info.get("rt_trace_kernel", {}).get("dram_bytes_per_launch")
        except Exception:
            traffic, ncu_info = None, None
    cache_bytes = (BYTES_NODE * ctr["nodes"] + BYTES_LEAF * ctr["leaves"] + BYTES_ACCEPT * ctr["accepts"]) / max(n_kern, 1)
    all_ms = sum(float(v) for v in stage_ms)
    executed = None
    if ncu_info and ncu_info.get("rt_trace_kernel", {}).get("thread_inst_per_launch"):
        t = ncu_info["rt_trace_kernel"]
        executed = {"thread_inst_per_launch": t["thread_inst_per_launch"], "ncu_launch_ms": t.get("ms_per_launch"),
                    "lane_ops_per_s_T": round(t["thread_inst_per_launch"] / launch_s / 1e12, 3),
                    "frac_of_peak": round(t["thread_inst_per_launch"] / launch_s / peak_ops, 4) if peak_ops else None,
                    "source": ncu_info.get("source"),
                    "note": "ALL executed thread-instructions of the kernel (address arithmetic, selects, queue I/O included), "
                            "from the committed ncu capture of this command, over this run's CUDA-event launch time"}
    roofline = {"kernel": "rt_trace_kernel", "bound": "fp32_issue (not hbm, not tensor: SURVEY 8d)",
                "achieved": round(achieved_tflops, 3), "peak": round(peak_ops / 1e12, 3), "unit": "TFLOP/s",
                "frac": round(achieved_tflops / (peak_ops / 1e12), 4) if peak_ops else None, "traffic": traffic,
                "traffic_source": ncu_info.get("source") if ncu_info else None,
                "peak_source": "measured live: non-fused FMUL+FADD issue rate (csrc/rt_peak.cu); MEASURED_PEAKS.json has no FP32 entry",
                "flop_model": "SURVEY 8d, traversal terms: 40/primary ray + 200/node + 456/leaf + 33/accept, from the kernels' own counters",
                "flops_per_launch": flops_per_launch, "launch_ms": round(kern_ms / max(n_kern, 1), 4), "launches": n_kern,
                "root_union_misses": root_misses,
                "frac_root_miss_as_18_ops": round(trace_flops_strict / max(n_kern, 1) / launch_s / peak_ops, 4) if peak_ops else None,
                "executed": executed,
                "cache_level_bytes_per_launch": cache_bytes,
                "hbm_compulsory_bytes_per_step": scene_bytes + 2 * W * H * 12,
                "hbm_achieved_GBps": round(traffic / launch_s / 1e9, 1) if traffic else None,
                "hbm_peak_GBps": hbm_peak,
                "stage_share_of_kernel_time": {k: round(float(stage_ms[i]) / all_ms, 4) if all_ms else None
                                               for i, k in enumerate(stage_names)},
                "stage_launches": {k: int(stage_n[i]) for i, k in enumerate(stage_names)},
                "whole_step": {"flops": algorithmic_flops(ctr) / args.steps, "kernel_ms": round(all_ms / args.steps, 3),
                               "achieved_tflops": round(algorithmic_flops(ctr) / (all_ms * 1e-3) / 1e12, 3) if all_ms else None},
                "per_sample": {k: round(ctr[k] / max(ctr["samples"], 1), 3) for k in ("rays", "nodes", "leaves", "shades", "misses")}}
    if rank == 0:
        roofline.update(film_kernel_rates(gpu, gpu_check, torch, W, H, SPP, sptr, hbm_peak))

    # the combined accumulator and image of the last timed step, for the parity check below
    accum_host = total.cpu().numpy() if rank == 0 else None
    pixels_host = pixels.cpu().numpy() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # what the caller of the timed path receives: the summed radiance (accum / spp = mean) and the u8 sRGB film
        dump_outputs(args.dump_outputs, {"accum": accum_host.reshape(H, W, 3), "pixels": pixels_host.reshape(H, W, 3)})

    # ---- e2e: through render_thread_proc with HOST buffers (N=1), or its device-level pieces + the cross-GPU film (N>1);
    # every step re-uploads the scene (H2D) and reads the image back (D2H)
    host_pixels = np.zeros((H, W, 3), dtype=np.uint8)
    pinned = torch.empty(H * W * 3, dtype=torch.uint8).pin_memory()
    e2e_steps = max(1, min(args.steps, 3))
    parts = {"upload_ms": [], "reduce_ms": [], "d2h_ms": []}

    def e2e_step():
        t_a = time.perf_counter()
        gpu_check(gpu.rt_gpu_scene_upload(scene_ref))              # H2D: nodes, triangles, textures, environment (asynchronous)
        parts["upload_ms"].append(1e3 * (time.perf_counter() - t_a))
        if world == 1:
            driver.set_options(slice_samples=slice_spp, fast_math=args.fast)
            driver.render(loaded, W, H, SPP, B, n_threads=1, out=host_pixels)   # D2H inside
            bd = (C.c_double * 4)()
            gpu.rt_gpu_last_frame_breakdown(C.byref(bd))
            parts["reduce_ms"].append(bd[1])
            parts["d2h_ms"].append(bd[2])
        else:
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            gpu_check(gpu.rt_gpu_render_shard_device(scene_ref, W, H, SPP, B, 0, rank, world, split_req, C.byref(mode_used),
                                                     accum_ptr, None, sptr))
            r0.record(stream)
            if reduce_how == "p2p":
                fence()
                if rank == 0:
                    gpu_check(gpu.rt_gpu_reduce_resolve_device(part_ptrs, world, None, W, H, SPP, pixels.data_ptr(), W, 3, sptr))
                fence()
            else:
                dist.reduce(accum_t, dst=0, op=dist.ReduceOp.SUM)
                if rank == 0:
                    gpu_check(gpu.rt_gpu_resolve_device(accum_t.data_ptr(), W, H, SPP, pixels.data_ptr(), W, 3, sptr))
            r1.record(stream)
            t_b = time.perf_counter()
            if rank == 0:
                pinned.copy_(pixels, non_blocking=True)
            torch.cuda.synchronize()
            parts["d2h_ms"].append(1e3 * (time.perf_counter() - t_b))      # includes waiting for the render to drain
            parts["reduce_ms"].append(r0.elapsed_time(r1))

    e2e_step()
    barrier()
    for v in parts.values():
        v.clear()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = W * H * SPP / float(e2e_s.item()) / 1e6
    driver.set_options()

    if rank == 0:
        parity = None
        if not args.no_parity:
            parity = parity_against_oracle(args, accum_host, pixels_host)
        cpu, cpu_spp, cpu_dt = (None, None, None)
        if world == 1 and not args.no_cpu:
            cpu, cpu_spp, cpu_dt = cpu_reference_rate(args)
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            driver.save_image(os.path.join(tmp, "frame.png"), host_pixels if world == 1 else pinned.numpy().reshape(H, W, 3))
            t_save = time.perf_counter() - t0
        mode_name = {SPLIT_SAMPLES: "sample-range", SPLIT_CHUNKS: "32x32-chunk round-robin"}[mode_used.value]
        film = {"p2p": "rank 0's fused reduce+resolve kernel reads the peers' accumulators over NVLink (CUDA IPC), two 4-byte NCCL all-reduces as fences",
                "nccl": "NCCL reduce(sum) of the f32 accumulators to rank 0, then the resolve kernel"}.get(reduce_how, reduce_how)
        mean = lambda v: round(sum(v) / len(v), 3) if v else None
        line = {"metric": metric_name(args), "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(workload_config(args, f"{mode_name} split x{world} (the library's policy, rt_gpu_render_shard_device); film: {film}"),
                               l2="flushed between steps (256 MiB memset inside the timed region, ~0.05 ms)",
                               chunk="the library renders as many samples of every pixel per wavefront chunk as its path queues hold (512 Mi paths by default = 256 spp at 1080p)",
                               host_buffers="pinned (rt_gpu_host_alloc)" if not args.pageable else "pageable (staged through a pinned ring)",
                               arithmetic="FAST MODE (opt-in): bounce stages FMA-contracted with hardware transcendentals; primary hits, ray generation, film exact"
                               if args.fast else "exact: every sample bit-identical to the reference arithmetic (no FMA contraction, rt_math.h)"),
                "clocks": clocks, "gpu_launches": timed_launches, "parity": parity,
                "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": upload_bytes,
                        "d2h_bytes_per_step": W * H * 3,
                        "upload_ms": mean(parts["upload_ms"]), "reduce_ms": mean(parts["reduce_ms"]), "d2h_ms": mean(parts["d2h_ms"]),
                        "ms_per_step": round(1e3 * float(e2e_s.item()), 3),
                        "how": "rt_gpu_scene_upload + render_thread_proc(host Image) per step" if world == 1 else
                               "scene upload + per-rank shard render + cross-GPU film + D2H to pinned host on rank 0, per step; "
                               "upload_ms = host time of the asynchronous upload call, d2h_ms includes draining the render"},
                "roofline": roofline, "cpu_baseline": cpu,
                "time_to_image_s": {"load_decode_bvh": round(t_load, 3), "upload": round(t_upload, 3),
                                    "render_e2e": round(float(e2e_s.item()), 3), "png_encode": round(t_save, 3)}}
        print(json.dumps(line), flush=True)
    loaded.close()
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="helmet1080p", choices=sorted(WORKLOADS))
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--bounces", type=int, default=8)
    ap.add_argument("--slice", type=int, default=0, help="e2e leg: samples per progress slice of render_thread_proc (0 = one wavefront chunk)")
    ap.add_argument("--cpu-spp", type=int, default=128, help="--impl reference: spp of each bounded CPU step (~6 s on 16 cores)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the reduced accumulator")
    ap.add_argument("--split", default="auto", choices=["auto", "samples", "chunks"], help="how a frame is split over GPUs")
    ap.add_argument("--reduce", default="p2p", choices=["p2p", "nccl"], help="cross-GPU film: fused P2P reduce+resolve, or NCCL reduce")
    ap.add_argument("--pageable", action="store_true", help="keep host scene buffers pageable (staged) instead of pinned")
    ap.add_argument("--fast", action="store_true",
                    help="opt-in fast mode (RT_GPU_Options.fast_math): FMA-contracted bounce stages with hardware transcendentals; "
                         "NOT the headline — the default is the bit-exact path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU path (--impl ours) only: write the accumulator and the u8 film of the last timed step to "
                         "DIR/accum.npy, DIR/pixels.npy (float32; a seeded pixel sample when they exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's frame: not available with --impl reference")
    for key in ("width", "height", "spp"):
        if getattr(args, key) is None:
            setattr(args, key, WORKLOADS[args.workload][key])
    import __graft_entry__ as entry
    if not (os.path.exists(os.path.join(ROOT, "raytracing_c_b200", "csrc", "libraytracer_gpu.so"))
            and os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so"))):
        entry.build()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
