"""Masked sample passes, for the tests: the CPU reference (the oracle renderer with its pixel_mask and sample range, and the
second moments summed from its per-sample radiance) and the device-level GPU call on torch tensors.
TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

import oracle_ffi


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def sequential_sums(per_sample):
    """(sum, sum of squares) over axis -2 of (..., S, 3) float32 radiance, added one sample at a time in sample order in
    float32: each product rounded, then each add — the arithmetic of the renderer's accumulate without contraction."""
    per_sample = np.asarray(per_sample, dtype=np.float32)
    s = np.zeros(per_sample.shape[:-2] + (3,), dtype=np.float32)
    q = np.zeros_like(s)
    for k in range(per_sample.shape[-2]):
        v = per_sample[..., k, :]
        s = s + v
        q = q + v * v
    return s, q


def oracle_masked(loaded, width, height, mask, sample_begin, sample_end, max_bounces, n_threads=None) -> dict:
    """The oracle renderer over samples [sample_begin, sample_end) of the pixels `mask` ((H, W), None = all) selects:
    {"accum", "accum_sq": (H, W, 3) float32, 0 on unselected pixels; "counters"}."""
    n = sample_end - sample_begin
    assert n > 0
    out = oracle_ffi.render(loaded, width, height, sample_end, max_bounces, n_threads=n_threads or os.cpu_count() or 8,
                            sample_begin=sample_begin, sample_end=sample_end, want_per_sample=True,
                            pixel_mask=None if mask is None else (np.asarray(mask) != 0).astype(np.uint8))
    s, q = sequential_sums(out["per_sample"])
    assert np.array_equal(bits(s), bits(out["accum"]))
    return {"accum": out["accum"], "accum_sq": q, "counters": out["counters"], "per_sample": out["per_sample"]}


def device_masked(loaded, width, height, mask, sample_begin, sample_end, max_bounces=8, accum=None, accum_sq=True,
                  accumulate=False, stream=None, user_seed=0) -> dict:
    """rt_gpu_render_masked_device on torch buffers, on `stream` (default: torch's current stream).  `mask` is a numpy
    (H, W) array or None.  `accum` / `accum_sq` (CUDA float32 tensors of W*H*3) are continued from with accumulate; fresh
    ones are filled with 7.0 first, so a value the call does not write shows.  accum_sq=False passes NULL.  Returns
    numpy copies, the eight counters and the kernels launched."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    acc = accum if accum is not None else torch.full((width * height * 3,), 7.0, dtype=torch.float32, device="cuda")
    if accum_sq is True:
        sq = torch.full((width * height * 3,), 7.0, dtype=torch.float32, device="cuda")
    else:
        sq = accum_sq if accum_sq is not False else None
    m = None if mask is None else torch.from_numpy((np.asarray(mask) != 0).astype(np.uint8)).cuda()
    ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
    st = stream or torch.cuda.current_stream()
    driver.register_callbacks(loaded)
    torch.cuda.synchronize()
    gpu = gpu_lib()
    before = gpu.rt_gpu_last_launches()
    gpu_check(gpu.rt_gpu_render_masked_device(C.byref(loaded.scene), width, height, m.data_ptr() if m is not None else None,
                                              sample_begin, sample_end, max_bounces, user_seed, int(accumulate),
                                              acc.data_ptr(), sq.data_ptr() if sq is not None else None, ctr.data_ptr(),
                                              st.cuda_stream))
    launches = gpu.rt_gpu_last_launches() - before
    st.synchronize()
    return {"accum": acc.cpu().numpy().reshape(height, width, 3),
            "accum_sq": sq.cpu().numpy().reshape(height, width, 3) if sq is not None else None,
            "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy()))), "launches": launches}


def device_render(loaded, width, height, sample_begin, sample_end, max_bounces=8, user_seed=0) -> dict:
    """rt_gpu_render_accum_device from zero on a fresh buffer: the accumulator, counters and kernels launched."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    acc = torch.full((width * height * 3,), 7.0, dtype=torch.float32, device="cuda")
    ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
    driver.register_callbacks(loaded)
    torch.cuda.synchronize()
    gpu = gpu_lib()
    before = gpu.rt_gpu_last_launches()
    gpu_check(gpu.rt_gpu_render_accum_device(C.byref(loaded.scene), width, height, sample_begin, sample_end, max_bounces,
                                             user_seed, 0, acc.data_ptr(), None, None, ctr.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream))
    launches = gpu.rt_gpu_last_launches() - before
    torch.cuda.synchronize()
    return {"accum": acc.cpu().numpy().reshape(height, width, 3),
            "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy()))), "launches": launches}


def masks(width, height, seed=0) -> dict:
    """The mask shapes the tests use, as (H, W) uint8 (None = the NULL mask)."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[:height, :width]
    single = np.zeros((height, width), dtype=np.uint8)
    single[height // 3, width // 2] = 1
    return {"random30": (rng.random((height, width)) < 0.3).astype(np.uint8),
            "checker": ((x + y) % 2).astype(np.uint8),
            "single": single,
            "empty": np.zeros((height, width), dtype=np.uint8),
            "ones": np.full((height, width), 255, dtype=np.uint8),
            "null": None}
