"""Masked sample passes (rt_gpu_render_masked_device) and the per-pixel-count film (rt_gpu_resolve_counts_device) on the
GPU.  Every accumulator, second moment and all eight work counters are compared bit for bit: against the oracle renderer
with its pixel_mask (six models and the inside-tower camera, six mask shapes, bounces 0/1/2/8, two sample offsets);
composed passes against uniform renders at each pixel's own sample count; the buffer rules; the NULL mask against the
renderer; chunked runs; fast_math; ordering against uploads and the other workspace users; refusals; one 1080p helmet
pass; the film; the compile-time budget of the new kernels.
"""
import contextlib
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import aov_ffi as A
import masked_ffi as M
import oracle_ffi
from helpers import load
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu

MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing_c_b200", "csrc", "libraytracer_gpu.so")
ZERO_COUNTERS = dict.fromkeys(oracle_ffi.COUNTER_NAMES, 0)


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    gpu_check(gpu_lib().rt_gpu_init(0))
    yield
    driver.set_options()


def upload(loaded):
    driver.register_callbacks(loaded)
    gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))


@pytest.fixture(scope="module", params=MODEL_NAMES + ["tower.obj:inside"])
def scene(request):
    loaded = A.load_default_camera("tower.obj") if request.param.endswith(":inside") else load(request.param)
    upload(loaded)
    yield request.param, loaded
    loaded.close()


@contextlib.contextmanager
def chunk_paths(n):
    """Path-queue chunks of at most n paths (RT_GPU_CHUNK_PATHS, read at every launch)."""
    old = os.environ.get("RT_GPU_CHUNK_PATHS")
    os.environ["RT_GPU_CHUNK_PATHS"] = str(n)
    try:
        yield
    finally:
        if old is None:
            del os.environ["RT_GPU_CHUNK_PATHS"]
        else:
            os.environ["RT_GPU_CHUNK_PATHS"] = old


def assert_same(got, want, where=None, counters=True):
    """accum and accum_sq bit for bit (on the pixels `where` selects, default all), and the counters."""
    sel = (slice(None),) if where is None else (where,)
    for key in ("accum", "accum_sq"):
        if want.get(key) is None:
            continue
        bad = M.bits(got[key][sel]) != M.bits(want[key][sel])
        assert not bad.any(), f"{key} differs on {int(bad.any(axis=-1).sum())} pixels"
    if counters:
        assert got["counters"] == want["counters"]


# (max_bounces, sample_begin)
CASES = [(8, 0), (1, 13), (2, 0), (0, 13), (8, 13)]


def test_bit_exact_against_the_oracle(scene):
    name, loaded = scene
    w, h, n = (128, 96, 8) if name == "helmet.glb" else (64, 48, 12)
    masks = M.masks(w, h)
    for bounces, begin in CASES:
        full = M.oracle_masked(loaded, w, h, None, begin, begin + n, max(bounces, 1)) if bounces else None
        for mname, mask in masks.items():
            got = M.device_masked(loaded, w, h, mask, begin, begin + n, bounces)
            if bounces == 0:
                # cast_ray's loop never runs: nothing traced or counted, the buffers zeroed (as the renderer does)
                assert not got["accum"].any() and not got["accum_sq"].any() and got["counters"] == ZERO_COUNTERS
                continue
            if mname in ("null", "ones"):
                want = full
            elif mname == "empty":
                want = {"accum": np.zeros((h, w, 3), np.float32), "accum_sq": np.zeros((h, w, 3), np.float32),
                        "counters": ZERO_COUNTERS}
            else:
                want = M.oracle_masked(loaded, w, h, mask, begin, begin + n, bounces)
            assert_same(got, want)
            sel = np.ones((h, w), bool) if mask is None else mask != 0
            assert got["counters"]["samples"] == int(sel.sum()) * n, mname


def test_passes_compose_to_uniform_renders_at_each_pixels_count():
    """A NULL-mask base [0, 16), then [16, 24) on mask A, then [24, 40) on a subset of A, chained with accumulate: every
    pixel equals a uniform render and the oracle at its own count (16, 24 or 40)."""
    import torch
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 96, 64
        rng = np.random.default_rng(3)
        a = (rng.random((h, w)) < 0.4).astype(np.uint8)
        b = a * (rng.random((h, w)) < 0.5).astype(np.uint8)
        acc = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        sq = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        parts = [M.device_masked(loaded, w, h, None, 0, 16, 8, accum=acc, accum_sq=sq),
                 M.device_masked(loaded, w, h, a, 16, 24, 8, accum=acc, accum_sq=sq, accumulate=True),
                 M.device_masked(loaded, w, h, b, 24, 40, 8, accum=acc, accum_sq=sq, accumulate=True)]
        got = parts[-1]
        count = np.where(b != 0, 40, np.where(a != 0, 24, 16))
        ref = oracle_ffi.render(loaded, w, h, 40, 8, n_threads=os.cpu_count() or 8, want_per_sample=True)
        for n in (16, 24, 40):
            sel = count == n
            assert sel.any()
            s, q = M.sequential_sums(ref["per_sample"][:, :, :n])
            assert_same(got, {"accum": s, "accum_sq": q}, where=sel, counters=False)
            uniform = M.device_render(loaded, w, h, 0, n, 8)
            assert np.array_equal(M.bits(got["accum"][sel]), M.bits(uniform["accum"][sel]))
        assert sum(p["counters"]["samples"] for p in parts) == int(count.sum())
    finally:
        loaded.close()


def test_buffer_rules_for_unselected_pixels():
    import torch
    loaded = load("spheres.glb")
    try:
        upload(loaded)
        w, h = 64, 48
        mask = M.masks(w, h)["checker"]
        sel = mask != 0
        want = M.oracle_masked(loaded, w, h, mask, 2, 10, 8)
        got = M.device_masked(loaded, w, h, mask, 2, 10, 8)              # buffers prefilled with 7.0, accumulate = 0
        assert_same(got, want)
        assert not got["accum"][~sel].any() and not got["accum_sq"][~sel].any()
        acc = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        sq = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        cont = M.device_masked(loaded, w, h, mask, 2, 10, 8, accum=acc, accum_sq=sq, accumulate=True)
        assert (cont["accum"][~sel] == 7).all() and (cont["accum_sq"][~sel] == 7).all()
        # selected pixels continue from the buffers: 7 + v0 + v1 ... and 7 + v0 * v0 + v1 * v1 ..., in float32
        ps = want["per_sample"][sel]
        s_ref = np.full(ps.shape[:1] + (3,), 7.0, np.float32)
        q_ref = s_ref.copy()
        for k in range(ps.shape[1]):
            s_ref = s_ref + ps[:, k]
            q_ref = q_ref + ps[:, k] * ps[:, k]
        assert np.array_equal(M.bits(cont["accum"][sel]), M.bits(s_ref))
        assert np.array_equal(M.bits(cont["accum_sq"][sel]), M.bits(q_ref))
    finally:
        loaded.close()


def test_null_mask_without_moments_is_the_renderer():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 160, 90
        want = M.device_render(loaded, w, h, 3, 21, 8)
        got = M.device_masked(loaded, w, h, None, 3, 21, 8, accum_sq=False)
        assert np.array_equal(M.bits(got["accum"]), M.bits(want["accum"]))
        assert got["counters"] == want["counters"] and got["launches"] == want["launches"]
        masked = M.device_masked(loaded, w, h, M.masks(w, h)["random30"], 3, 21, 8)
        assert masked["launches"] == want["launches"]
    finally:
        loaded.close()


def test_chunked_runs_equal_one_chunk():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 120, 80
        mask = M.masks(w, h, seed=5)["random30"]
        whole = M.device_masked(loaded, w, h, mask, 1, 30, 8)
        with chunk_paths(w * h * 4):           # rounded up to whole job tiles: chunks of 4 samples of every pixel
            chunked = M.device_masked(loaded, w, h, mask, 1, 30, 8)
        assert_same(chunked, whole)
        assert chunked["launches"] > whole["launches"]
    finally:
        loaded.close()


def test_fast_math_masked_is_the_fast_render_on_selected_pixels():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 96, 64
        mask = M.masks(w, h, seed=7)["random30"]
        sel = mask != 0
        driver.set_options(fast_math=True)
        fast = M.device_render(loaded, w, h, 0, 12, 8)
        got = M.device_masked(loaded, w, h, mask, 0, 12, 8)
        assert np.array_equal(M.bits(got["accum"][sel]), M.bits(fast["accum"][sel]))
        assert not got["accum"][~sel].any()
        null = M.device_masked(loaded, w, h, None, 0, 12, 8, accum_sq=False)
        assert np.array_equal(M.bits(null["accum"]), M.bits(fast["accum"]))
        driver.set_options()
        exact = M.device_masked(loaded, w, h, mask, 0, 12, 8)
        assert_same(exact, M.oracle_masked(loaded, w, h, mask, 0, 12, 8))
    finally:
        driver.set_options()
        loaded.close()


def test_on_a_user_stream_right_after_upload():
    """A fresh scene, uploaded and given a masked pass at once on a torch stream: the call waits for the texels."""
    import torch
    loaded = load("helmet.glb")
    try:
        w, h = 128, 96
        mask = M.masks(w, h)["random30"]
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        upload(loaded)
        with torch.cuda.stream(stream):
            got = M.device_masked(loaded, w, h, mask, 0, 4, 8, stream=stream)
        torch.cuda.synchronize()
        assert_same(got, M.oracle_masked(loaded, w, h, mask, 0, 4, 8))
    finally:
        loaded.close()


def test_interleaved_with_renders_aov_and_cast_rays():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 96, 64
        mask = M.masks(w, h)["checker"]
        want = M.oracle_masked(loaded, w, h, mask, 0, 6, 8)
        rays_o = np.zeros((64, 3), np.float32)
        rays_d = np.tile(np.array([0.0, 0.0, -1.0], np.float32), (64, 1))
        rays_o[:, 2] = 5.0
        first_cast = driver.cast_rays(loaded, rays_o, rays_d, 4)
        first_aov = A.device_aov(loaded, w, h, 0, 4, 8)
        for _ in range(2):
            driver.render(loaded, 64, 48, 4, 8)
            assert_same(M.device_masked(loaded, w, h, mask, 0, 6, 8), want)
            assert np.array_equal(M.bits(driver.cast_rays(loaded, rays_o, rays_d, 4)), M.bits(first_cast))
            assert_same(M.device_masked(loaded, w, h, mask, 0, 6, 8), want)
            got_aov = A.device_aov(loaded, w, h, 0, 4, 8)
            assert np.array_equal(A.bits(got_aov["records"]), A.bits(first_aov["records"]))
    finally:
        loaded.close()


def test_refusals_and_empty_calls():
    import torch
    loaded = load("quad.obj")
    other = load("quad.obj")
    try:
        upload(loaded)
        gpu = gpu_lib()
        w, h = 32, 16
        acc = torch.full((w * h * 3 + 4,), 7.0, dtype=torch.float32, device="cuda")
        sq = torch.full((w * h * 3 + 4,), 7.0, dtype=torch.float32, device="cuda")
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        mask = torch.ones(w * h, dtype=torch.uint8, device="cuda")
        sc = C.byref(loaded.scene)
        st = torch.cuda.current_stream().cuda_stream

        def dev(scene=sc, width=w, height=h, begin=0, end=2, bounces=8, out=acc.data_ptr(), accumulate=0):
            return gpu.rt_gpu_render_masked_device(scene, width, height, mask.data_ptr(), begin, end, bounces, 0, accumulate,
                                                   out, sq.data_ptr(), ctr.data_ptr(), st)
        cases = [
            (lambda: dev(width=0), "empty"),
            (lambda: dev(height=-1), "empty"),
            (lambda: dev(width=1 << 20, height=1 << 12), "too large"),
            (lambda: dev(width=1 << 31), "too large"),
            (lambda: dev(begin=-1), "samples"),
            (lambda: dev(begin=5, end=4), "samples"),
            (lambda: dev(end=1 << 31), "samples"),
            (lambda: dev(bounces=-1), "max_bounces"),
            (lambda: dev(out=None), "accum"),
            (lambda: dev(scene=C.byref(other.scene)), "resident"),
            (lambda: dev(scene=None), "scene"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in gpu.rt_gpu_last_error().decode(), word
        assert gpu.rt_gpu_scene_device_bytes(C.byref(other.scene)) == 0, "a refused call uploads nothing"
        torch.cuda.synchronize()
        assert (acc == 7).all() and (sq == 7).all() and not ctr.any()
        # empty range or no bounces: buffers kept with accumulate, zeroed without; nothing traced or counted
        for kw in (dict(begin=5, end=5), dict(bounces=0)):
            assert dev(accumulate=1, **kw) == 0
            torch.cuda.synchronize()
            assert (acc == 7).all() and (sq == 7).all()
            assert dev(**kw) == 0
            torch.cuda.synchronize()
            for buf in (acc, sq):
                assert not buf[:w * h * 3].any() and (buf[w * h * 3:] == 7).all()
            assert not ctr.any()
            acc.fill_(7.0)
            sq.fill_(7.0)
        # the film's refusals
        px = torch.zeros(w * h * 4, dtype=torch.uint8, device="cuda")
        counts = torch.ones(w * h, dtype=torch.int32, device="cuda")
        assert gpu.rt_gpu_resolve_counts_device(acc.data_ptr(), None, w, h, px.data_ptr(), w, 3, st) != 0
        assert "d_samples" in gpu.rt_gpu_last_error().decode()
        assert gpu.rt_gpu_resolve_counts_device(acc.data_ptr(), counts.data_ptr(), w, h, px.data_ptr(), w, 2, st) != 0
        assert "components" in gpu.rt_gpu_last_error().decode()
        # the library still answers after the refusals
        m = M.masks(w, h)["random30"]
        assert_same(M.device_masked(loaded, w, h, m, 0, 3, 8), M.oracle_masked(loaded, w, h, m, 0, 3, 8))
    finally:
        other.close()
        loaded.close()


def test_whole_helmet_frame_pass():
    """A 20 % pass over a 1920x1080 helmet frame, checked against the oracle on 4096 of its pixels."""
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h, n = 1920, 1080, 8
        rng = np.random.default_rng(11)
        mask = (rng.random((h, w)) < 0.2).astype(np.uint8)
        got = M.device_masked(loaded, w, h, mask, 0, n, 8)
        assert got["counters"]["samples"] == int(mask.sum()) * n
        sel = np.flatnonzero(mask)
        check = np.zeros(h * w, np.uint8)
        check[rng.choice(sel, 4096, replace=False)] = 1
        check = check.reshape(h, w)
        want = M.oracle_masked(loaded, w, h, check, 0, n, 8)
        assert_same(got, want, where=check != 0, counters=False)
        assert not got["accum"][mask == 0].any()
    finally:
        loaded.close()


def test_resolve_counts():
    import torch
    loaded = load("sheen.glb")
    try:
        upload(loaded)
        w, h = 64, 48
        st = torch.cuda.current_stream().cuda_stream
        gpu = gpu_lib()
        got = M.device_masked(loaded, w, h, None, 0, 24, 8)
        acc = torch.from_numpy(got["accum"]).cuda().contiguous()
        # uniform counts: the existing film byte for byte
        want = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
        gpu_check(gpu.rt_gpu_resolve_device(acc.data_ptr(), w, h, 24, want.data_ptr(), w, 3, st))
        uniform = driver.resolve_counts(acc, torch.full((h, w), 24, dtype=torch.int32, device="cuda"))
        torch.cuda.synchronize()
        assert torch.equal(uniform, want)
        # mixed counts: each group is oracle_resolve at its count; counts <= 0 and NaN sums give 0
        counts = np.random.default_rng(2).choice([1, 7, 24, 1000, 0, -3], size=(h, w)).astype(np.int32)
        accum = got["accum"].copy()
        accum[5, 7] = np.nan
        counts[5, 7] = 24
        px = driver.resolve_counts(torch.from_numpy(accum).cuda(), torch.from_numpy(counts).cuda()).cpu().numpy()
        for n in np.unique(counts):
            sel = counts == n
            if n <= 0:
                assert not px[sel].any()
            else:
                assert np.array_equal(px[sel], oracle_ffi.resolve(accum[sel], int(n)))
        assert not px[5, 7].any()
        # RGBA output with a padded stride: the fourth byte and the padding are not written
        rgba = torch.full((h, w + 3, 4), 9, dtype=torch.uint8, device="cuda")
        gpu_check(gpu.rt_gpu_resolve_counts_device(acc.data_ptr(), torch.from_numpy(counts).cuda().data_ptr(), w, h,
                                                   rgba.data_ptr(), w + 3, 4, st))
        torch.cuda.synchronize()
        out = rgba.cpu().numpy()
        assert np.array_equal(out[:, :w, :3], driver.resolve_counts(acc, torch.from_numpy(counts).cuda()).cpu().numpy())
        assert (out[:, :w, 3] == 9).all() and (out[:, w:] == 9).all()
    finally:
        loaded.close()


BUDGET = {   # mangled-name fragment -> (max registers per thread, max bytes of stack), from -Xptxas -v
    "rt_trace_kernelILb1ELi4ELb1E": (64, 24),       # the unmasked primary trace's 64 registers and 24-byte frame
    "rt_accumulate_masked_kernel": (40, 0),
    "rt_resolve_counts_kernel": (32, 0),
}


@pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB), reason="needs the built library and cuobjdump")
def test_new_kernels_keep_their_register_budget():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
    found = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        for key in BUDGET:
            if key in m.group(1):
                found[key] = (int(m.group(2)), int(m.group(3)))
    assert set(found) == set(BUDGET), f"kernels missing from the library: {set(BUDGET) - set(found)}"
    for key, (regs, stack) in found.items():
        assert regs <= BUDGET[key][0], f"{key}: {regs} registers (budget {BUDGET[key][0]})"
        assert stack <= BUDGET[key][1], f"{key}: {stack} bytes of stack (budget {BUDGET[key][1]})"
