"""Small fixed workload for ncu: helmet.glb 1920x1080, `--spp` samples in one launch, `--reps` launches.

    python tools/profile_render.py --spp 16 --reps 3
Prints the CUDA-event time per launch (never quote a number taken under a profiler)."""
import argparse
import ctypes as C

import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
from raytracing_c_b200 import driver
from raytracing_c_b200._ffi import gpu_check

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="helmet.glb")
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--spp", type=int, default=64)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--denoise", action="store_true")
ap.add_argument("--stages", action="store_true", help="print CUDA-event time per stage and bounce of the last rep")
ap.add_argument("--eye", type=float, nargs=3, default=None, help="camera position (with --target; default: the model's camera)")
ap.add_argument("--target", type=float, nargs=3, default=(0.0, 0.0, 0.0))
args = ap.parse_args()

gpu = benchkit.init()
torch.cuda.set_device(0)
camera = driver.look_at(args.eye, args.target) if args.eye else None
loaded = benchkit.resident(args.model, camera=camera)
scene = C.byref(loaded.scene)
W, H = args.width, args.height
accum = torch.zeros(W * H * 3, dtype=torch.float32, device="cuda")
pixels = torch.zeros(W * H * 3, dtype=torch.uint8, device="cuda")
pixels2 = torch.zeros(W * H * 3, dtype=torch.uint8, device="cuda")
counters = torch.zeros(8, dtype=torch.int64, device="cuda")
stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
for rep in range(args.reps):
    counters.zero_()
    if args.stages and rep == args.reps - 1:
        gpu.rt_gpu_stage_profile_enable(1)
    times = globals().setdefault("times", [])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gpu_check(gpu.rt_gpu_render_accum_device(scene, W, H, 0, args.spp, 8, 0, 0, accum.data_ptr(), None, None,
                                             counters.data_ptr(), stream))
    e1.record()
    gpu_check(gpu.rt_gpu_resolve_device(accum.data_ptr(), W, H, args.spp, pixels.data_ptr(), W, 3, stream))
    if args.denoise:
        gpu_check(gpu.rt_gpu_denoise_device(pixels.data_ptr(), pixels2.data_ptr(), W, H, W, W, 3, stream))
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    c = counters.cpu().tolist()
    times.append(ms)
    print(f"rep {rep}: render {ms:.3f} ms  {W * H * args.spp / ms / 1e3:.1f} Msamples/s  counters {c}", flush=True)
if len(times) > 2:
    t = sorted(times[1:])
    print(f"render ms over reps 1..{len(times) - 1}: min {t[0]:.3f} median {t[len(t) // 2]:.3f} max {t[-1]:.3f}  "
          f"=> {W * H * args.spp / t[0] / 1e3:.1f} Msamples/s best", flush=True)
if args.stages:
    ms, n = (C.c_double * 64)(), (C.c_int64 * 64)()
    gpu_check(gpu.rt_gpu_stage_profile_read_bounces(C.byref(ms), C.byref(n)))
    for s, name in enumerate(["trace", "miss", "shade", "accumulate"]):
        print(name, " ".join(f"b{b}:{ms[s * 16 + b] * 1e3:.0f}us" for b in range(16) if n[s * 16 + b]), flush=True)
    print(f"sum of kernel times {sum(ms) :.3f} ms", flush=True)
loaded.close()
