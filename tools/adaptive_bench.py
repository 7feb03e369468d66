#!/usr/bin/env python
"""adaptive_bench.py — what masked sample passes (rt_gpu_render_masked_device) cost and what a simple adaptive loop
built on them buys, on helmet.glb at 1920x1080 with 8 bounces.

    python tools/adaptive_bench.py [--reps 5] [--out profiles/r07_adaptive_bench.json]

1. Mask read: a NULL-mask call and rt_gpu_render_accum_device at 64 spp, alternating, `reps` pairs after a warm-up of
   each; CUDA events per call.  Their accumulators must be bitwise identical.
2. Pass cost against mask density: one 32-sample pass at 100 / 50 / 10 / 1 % of the pixels, for two mask shapes —
   random pixels, and whole 8x4 job tiles (a warp's pixels all selected or all skipped at fewer than 32 samples, and
   always at 32: one warp is one pixel's 32 samples) — the median over `reps` calls.
3. A reference adaptive loop (host policy, torch on the device): 32 spp of every pixel with second moments, then
   passes of 32 samples over the pixels whose relative standard error of mean luminance is above a threshold, capped
   at 1024 spp; a pixel that falls below the threshold is not selected again.  The luminance standard deviation is
   bounded by sum_c w_c * sd_c (Rec. 709 weights), which needs only the per-channel second moments.  Reported per
   threshold: time (CUDA events around the whole loop, mask computation included), samples spent, and the RMSE of the
   u8 sRGB image (rt_gpu_resolve_counts_device) against a 1024-spp uniform render with another user_seed (so the
   reference does not share the loop's samples), beside the RMSE of a uniform render with the same total samples; and
   the time and RMSE of uniform renders at 32 .. 512 spp.
The card name and power limit are read in the same run.
"""
from __future__ import annotations

import ctypes as C
import json

import numpy as np
import torch

import benchkit  # first: it puts the repository root and tests/ on sys.path
from raytracing_c_b200 import driver
from raytracing_c_b200._ffi import gpu_check

W, H, BOUNCES = 1920, 1080, 8
PASS, CAP = 32, 1024
DENSITIES = (1.0, 0.5, 0.1, 0.01)
THRESHOLDS = (0.1, 0.05, 0.02)
UNIFORM_SPPS = (32, 64, 128, 256, 512)
LUMA = (0.2126, 0.7152, 0.0722)


def main() -> None:
    args = benchkit.parser(reps=5).parse_args()
    gpu = benchkit.init()
    loaded = benchkit.resident("helmet.glb")
    scene = C.byref(loaded.scene)
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    acc = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
    acc2 = torch.empty_like(acc)
    sq = torch.empty_like(acc)
    result = {"card": benchkit.card(), "model": "helmet.glb", "frame": f"{W}x{H}", "max_bounces": BOUNCES,
              "reps": args.reps}

    def render(begin, end, out, seed=0):
        gpu_check(gpu.rt_gpu_render_accum_device(scene, W, H, begin, end, BOUNCES, seed, 0, out.data_ptr(), None, None,
                                                 None, st))

    def masked(mask, begin, end, out, out_sq=None, accumulate=False, seed=0):
        gpu_check(gpu.rt_gpu_render_masked_device(scene, W, H, mask.data_ptr() if mask is not None else None, begin, end,
                                                  BOUNCES, seed, int(accumulate), out.data_ptr(),
                                                  out_sq.data_ptr() if out_sq is not None else None, None, st))

    # ---- 1. the mask read: NULL mask against the renderer, alternating
    spp = 64
    render(0, spp, acc); masked(None, 0, spp, acc2)                      # warm-up: workspace, modules
    torch.cuda.synchronize()
    t_render, t_null = [], []
    for _ in range(args.reps):
        t_render.append(benchkit.window_ms(lambda: render(0, spp, acc), stream))
        t_null.append(benchkit.window_ms(lambda: masked(None, 0, spp, acc2), stream))
    identical = bool(torch.equal(acc.view(torch.int32), acc2.view(torch.int32)))
    r1 = {"spp": spp, "render_ms": [round(t, 3) for t in t_render], "null_mask_ms": [round(t, 3) for t in t_null],
          "render_median_ms": round(float(np.median(t_render)), 3), "null_mask_median_ms": round(float(np.median(t_null)), 3),
          "null_over_render": round(float(np.median(t_null) / np.median(t_render)), 4), "outputs_bitwise_identical": identical}
    result["mask_read"] = r1
    print(json.dumps({"mask_read": r1}), flush=True)

    # ---- 2. one 32-sample pass against mask density and shape
    gen = torch.Generator(device="cuda").manual_seed(2026)
    tiles_shape = ((H + 3) // 4, (W + 7) // 8)
    r2 = {}
    full_ms = None
    for shape in ("random", "tiles"):
        for d in DENSITIES:
            if shape == "random":
                m = (torch.rand((H, W), generator=gen, device="cuda") < d).to(torch.uint8)
            else:
                t = (torch.rand(tiles_shape, generator=gen, device="cuda") < d).to(torch.uint8)
                m = t.repeat_interleave(4, 0).repeat_interleave(8, 1)[:H, :W].contiguous()
            if d == 1.0:
                m.fill_(1)
            masked(m, 0, PASS, acc)
            torch.cuda.synchronize()
            ts = [benchkit.window_ms(lambda: masked(m, 0, PASS, acc), stream) for _ in range(args.reps)]
            ms = float(np.median(ts))
            if full_ms is None:
                full_ms = ms
            sel = int(m.sum().item())
            key = f"{shape}_{int(d * 100)}pct"
            r2[key] = {"selected_pixels": sel, "ms": round(ms, 3), "over_full_pass": round(ms / full_ms, 4),
                       "Msamples_per_s": round(sel * PASS / (ms * 1e-3) / 1e6, 1)}
            print(json.dumps({key: r2[key]}), flush=True)
    result["pass_cost"] = r2

    # ---- 3. a reference adaptive loop against uniform renders
    ref = torch.empty_like(acc)
    render(0, CAP, ref, seed=1)
    ref_px = driver.resolve_counts(ref, torch.full((H, W), CAP, dtype=torch.int32, device="cuda")).float()
    w_luma = torch.tensor(LUMA, device="cuda")

    def rmse(px):
        return float(torch.sqrt(((px.float() - ref_px) ** 2).mean()).item())

    r3 = {"pass_samples": PASS, "cap_spp": CAP, "reference": f"uniform {CAP} spp, user_seed 1", "thresholds": {}}
    for thr in THRESHOLDS:
        counts = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        passes = []

        def loop():
            masked(None, 0, PASS, acc, sq)
            counts.fill_(PASS)
            active = torch.ones((H, W), dtype=torch.bool, device="cuda")
            n = PASS
            while n < CAP:
                mean = acc / n
                var = torch.clamp(sq / n - mean * mean, min=0) * (n / (n - 1))
                sd_luma = (torch.sqrt(var) * w_luma).sum(-1)
                mean_luma = (mean * w_luma).sum(-1)
                rse = sd_luma / (mean_luma * n ** 0.5)
                active &= rse > thr                        # a converged pixel (or a black one: 0 / 0) is not selected again
                m = active.to(torch.uint8)
                masked(m, n, n + PASS, acc, sq, accumulate=True)
                counts.add_(m.to(torch.int32) * PASS)
                passes.append(m)
                n += PASS
        ms = benchkit.window_ms(loop, stream)
        spent = int(counts.sum().item())
        px = driver.resolve_counts(acc, counts)
        eq_spp = max(1, round(spent / (W * H)))
        render(0, eq_spp, acc2)
        eq_px = driver.resolve_counts(acc2, torch.full((H, W), eq_spp, dtype=torch.int32, device="cuda"))
        eq_ms = benchkit.window_ms(lambda: render(0, eq_spp, acc2), stream)
        hist = torch.bincount(counts.flatten().long() // PASS, minlength=CAP // PASS + 1).cpu().numpy()
        r = {"ms": round(ms, 3), "samples": spent, "mean_spp": round(spent / (W * H), 2),
             "passes": len(passes), "pixels_at_cap": int((counts == CAP).sum().item()),
             "spp_histogram": {str(k * PASS): int(v) for k, v in enumerate(hist) if v},
             "rmse_u8": round(rmse(px), 4),
             "uniform_equal_samples": {"spp": eq_spp, "ms": round(eq_ms, 3), "rmse_u8": round(rmse(eq_px), 4)}}
        r3["thresholds"][str(thr)] = r
        print(json.dumps({f"adaptive_{thr}": r}), flush=True)
    # the uniform curve the loop is compared with: RMSE and time of a uniform render per sample count
    r3["uniform"] = {}
    for spp in UNIFORM_SPPS:
        ms = benchkit.window_ms(lambda: render(0, spp, acc2), stream)
        px = driver.resolve_counts(acc2, torch.full((H, W), spp, dtype=torch.int32, device="cuda"))
        r3["uniform"][str(spp)] = {"ms": round(ms, 3), "rmse_u8": round(rmse(px), 4)}
    print(json.dumps({"uniform": r3["uniform"]}), flush=True)
    result["adaptive_loop"] = r3

    result["parity_ok"] = identical
    benchkit.finish(args, result, ("parity_ok",), loaded)


if __name__ == "__main__":
    main()
