"""Sky tiles: job tiles whose camera rays provably miss the root-union box are rendered by rt_sky_kernel instead of the
primary trace, the bounce-0 miss kernel and the accumulate.  Accumulator, u8 film, primary hit ids and all eight work
counters must stay bit for bit the oracle's, and counters_ex[1] (primary rays) the rendered pixel-samples, for cameras
that see part, none or all of the model as sky, image sizes that are not whole tiles, sample offsets, chunked runs,
masked passes across the sky boundary, pixel splits and fast mode.
"""
import ctypes as C
import os

import numpy as np
import pytest

import aov_ffi as A
import masked_ffi as M
import oracle_ffi
from helpers import chunk_paths, load
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu


# helmet.glb's bounds are about [-1, 1]^3 around the origin; its own camera sits at (1, -0.2, 1.73) facing it
CAMERAS = {
    "default": None,
    "away": dict(eye=(2.0, -0.2, 3.4641), target=(4.0, -0.2, 6.9282)),          # sees only sky
    "behind": dict(eye=(1.2, 0.0, 0.0), target=(1.2, 0.0, -5.0)),              # part of the model behind the camera plane
    "border": dict(eye=(0.0, 0.0, 3.0), target=(1.3, 0.0, 0.0)),               # the model cut by the image border
}


def counters_ex():
    raw = (C.c_uint64 * 16)()
    gpu_check(gpu_lib().rt_gpu_read_counters_ex(raw))
    return [int(v) for v in raw[8:]]


def gpu_frame(loaded, w, h, spp, bounces, **options):
    driver.set_options(keep_hit_ids=True, **options)
    pixels = driver.render(loaded, w, h, spp, bounces)
    return dict(pixels=pixels, accum=driver.read_accum(w, h), hit_ids=driver.read_hit_ids(w, h),
                counters=driver.read_counters(), ex=counters_ex())


def check_frame(loaded, w, h, spp, bounces, sample_begin=0, **options):
    opts = dict(sample_begin=sample_begin, sample_end=spp) if sample_begin else {}
    got = gpu_frame(loaded, w, h, spp, bounces, **opts, **options)
    ref = oracle_ffi.render(loaded, w, h, spp, bounces, n_threads=os.cpu_count() or 8, want_hit_ids=True,
                            sample_begin=sample_begin, sample_end=spp if sample_begin else 0)
    assert np.array_equal(got["hit_ids"], ref["hit_ids"])
    assert np.array_equal(M.bits(got["accum"]), M.bits(ref["accum"]))
    if not sample_begin:
        assert np.array_equal(got["pixels"], ref["pixels"])
    assert got["counters"] == ref["counters"]
    assert got["ex"][1] == w * h * (spp - sample_begin), "counters_ex[1] must be the rendered pixel-samples"
    return got, ref


@pytest.fixture(scope="module", params=sorted(CAMERAS))
def helmet(request):
    cam = CAMERAS[request.param]
    loaded = load("helmet.glb", camera=cam)
    driver.register_callbacks(loaded)
    yield request.param, loaded
    loaded.close()


@pytest.mark.parametrize("w,h", [(96, 64), (83, 45), (7, 3), (1, 1)])
@pytest.mark.parametrize("bounces", [1, 8])
def test_frames_bit_exact(helmet, w, h, bounces):
    name, loaded = helmet
    got, ref = check_frame(loaded, w, h, 6, bounces)
    if name == "away":
        assert (ref["hit_ids"] < 0).all() and got["ex"][0] == got["ex"][1], "every ray is a root-union miss"


def test_sample_offsets_and_small_chunks(helmet):
    _, loaded = helmet
    for begin in (0, 5):
        check_frame(loaded, 70, 42, 13, 8, sample_begin=begin)
        with chunk_paths(72 * 44 * 3):          # whole job tiles: chunks of 3 samples of every pixel
            check_frame(loaded, 70, 42, 13, 8, sample_begin=begin)


def test_inside_tower_camera():
    loaded = A.load_default_camera("tower.obj")
    try:
        driver.register_callbacks(loaded)
        check_frame(loaded, 64, 48, 6, 8)
    finally:
        loaded.close()


def test_masked_passes_across_the_sky_boundary():
    import torch
    loaded = load("helmet.glb", camera=CAMERAS["border"])
    try:
        driver.register_callbacks(loaded)
        gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))
        w, h = 96, 64
        for mname in ("random30", "checker", "ones", "null"):
            mask = M.masks(w, h, seed=7)[mname]
            want = M.oracle_masked(loaded, w, h, mask, 3, 15, 8)
            got = M.device_masked(loaded, w, h, mask, 3, 15, 8)
            for key in ("accum", "accum_sq"):
                assert np.array_equal(M.bits(got[key]), M.bits(want[key])), (mname, key)
            assert got["counters"] == want["counters"], mname
        # continuing: unselected pixels keep the buffers' 7.0, selected ones continue from them
        mask = M.masks(w, h, seed=7)["random30"]
        sel = mask != 0
        acc = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        sq = torch.full((w * h * 3,), 7.0, dtype=torch.float32, device="cuda")
        cont = M.device_masked(loaded, w, h, mask, 3, 15, 8, accum=acc, accum_sq=sq, accumulate=True)
        ps = M.oracle_masked(loaded, w, h, mask, 3, 15, 8)["per_sample"][sel]
        s_ref = np.full(ps.shape[:1] + (3,), 7.0, np.float32)
        q_ref = s_ref.copy()
        for k in range(ps.shape[1]):
            s_ref = s_ref + ps[:, k]
            q_ref = q_ref + ps[:, k] * ps[:, k]
        assert (cont["accum"][~sel] == 7).all() and (cont["accum_sq"][~sel] == 7).all()
        assert np.array_equal(M.bits(cont["accum"][sel]), M.bits(s_ref))
        assert np.array_equal(M.bits(cont["accum_sq"][sel]), M.bits(q_ref))
    finally:
        loaded.close()


def test_per_sample_radiance():
    import torch
    loaded = load("helmet.glb", camera=CAMERAS["border"])
    try:
        driver.register_callbacks(loaded)
        gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))
        w, h, n = 80, 48, 40
        ref = oracle_ffi.render(loaded, w, h, n, 8, n_threads=os.cpu_count() or 8, want_per_sample=True)
        acc = torch.zeros(w * h * 3, dtype=torch.float32, device="cuda")
        ps = torch.zeros(w * h * n * 3, dtype=torch.float32, device="cuda")
        gpu_check(gpu_lib().rt_gpu_render_accum_device(C.byref(loaded.scene), w, h, 0, n, 8, 0, 0, acc.data_ptr(),
                                                       ps.data_ptr(), None, None, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert np.array_equal(M.bits(ps.cpu().numpy().reshape(h, w, n, 3)), M.bits(ref["per_sample"]))
        assert np.array_equal(M.bits(acc.cpu().numpy().reshape(h, w, 3)), M.bits(ref["accum"]))
    finally:
        loaded.close()


@pytest.mark.parametrize("world", [2, 3])
def test_pixel_split(world):
    loaded = load("helmet.glb", camera=CAMERAS["border"])
    try:
        driver.register_callbacks(loaded)
        w, h, spp = 200, 150, 6
        full = gpu_frame(loaded, w, h, spp, 8)
        ref = oracle_ffi.render(loaded, w, h, spp, 8, n_threads=os.cpu_count() or 8, want_hit_ids=True)
        assert np.array_equal(M.bits(full["accum"]), M.bits(ref["accum"])) and full["counters"] == ref["counters"]
        total = np.zeros_like(full["accum"])
        ids = np.full((h, w), -(2 ** 31), dtype=np.int64)
        counters, primary = {}, 0
        for r in range(world):
            part = gpu_frame(loaded, w, h, spp, 8, pixel_rank=r, pixel_world=world)
            total += part["accum"]
            ids = np.maximum(ids, part["hit_ids"])
            primary += part["ex"][1]
            for k, v in part["counters"].items():
                counters[k] = counters.get(k, 0) + v
        assert np.array_equal(M.bits(total), M.bits(ref["accum"]))
        assert np.array_equal(ids, ref["hit_ids"])
        assert counters == ref["counters"] and primary == w * h * spp
    finally:
        loaded.close()


@pytest.mark.parametrize("cam", ["default", "away"])
def test_fast_mode_close_to_exact(cam):
    loaded = load("helmet.glb", camera=CAMERAS[cam])
    try:
        driver.register_callbacks(loaded)
        w, h, spp = 320, 180, 64
        exact = gpu_frame(loaded, w, h, spp, 8)
        fast = gpu_frame(loaded, w, h, spp, 8, fast_math=True)
        ref = oracle_ffi.render(loaded, w, h, 1, 8, n_threads=os.cpu_count() or 8, want_hit_ids=True)
        assert np.array_equal(fast["hit_ids"], ref["hit_ids"])
        rel = np.abs(fast["accum"] - exact["accum"]) / np.maximum(np.abs(exact["accum"]), 1e-6)
        a, b = fast["pixels"].astype(np.float64) / 255, exact["pixels"].astype(np.float64) / 255
        rmse = float(np.sqrt(np.mean((a - b) ** 2)))
        assert np.median(rel) < 1e-4 and rmse < 0.005
        assert abs(fast["counters"]["rays"] / exact["counters"]["rays"] - 1) < 0.01
        assert fast["ex"][1] == exact["ex"][1] == w * h * spp
    finally:
        loaded.close()
