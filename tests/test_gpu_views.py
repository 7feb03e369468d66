"""Many views of a resident scene in one call (rt_gpu_render_views_device / rt_gpu_render_views) on the GPU.  Every view's
accumulator is compared bit for bit with the single render it replaces (rt_gpu_render_accum_device with scene->camera
set to that view's camera and its seed), and the counters with the sum of those renders' counters: six models and the
inside-tower camera, camera sets with a duplicate, different fields of view, an all-sky view and a view from inside the
bounds, bounces 0/1/2/8, two sample offsets, NULL and distinct seeds.  Also: two views against the oracle renderer;
chunked calls (sample chunks and view groups) and accumulation; fast_math; the one-view call against a render (bits,
counters, launches); ordering against uploads, renders, AOV, cast_rays and a refit; refusals and empty calls; the host
form and its film.  The primary trace's register budget is in test_build_properties.py.
"""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

import aov_ffi as A
import oracle_ffi
import views_ffi as V
from helpers import MODEL_NAMES, chunk_paths, load, upload
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import Camera, gpu_check

pytestmark = pytest.mark.gpu

ZERO_COUNTERS = dict.fromkeys(oracle_ffi.COUNTER_NAMES, 0)
W, H = 96, 64


@pytest.fixture(scope="module", params=MODEL_NAMES + ["tower.obj:inside"])
def scene(request):
    loaded = A.load_default_camera("tower.obj") if request.param.endswith(":inside") else load(request.param)
    upload(loaded)
    yield request.param, loaded
    loaded.close()


def assert_views(got, want, counters=True):
    assert got["accum"].shape == want["accum"].shape
    for v in range(got["accum"].shape[0]):
        bad = V.bits(got["accum"][v]) != V.bits(want["accum"][v])
        assert not bad.any(), f"view {v} differs on {int(bad.any(axis=-1).sum())} pixels"
    if counters:
        assert got["counters"] == want["counters"]


# (max_bounces, sample_begin, distinct seeds)
CASES = [(8, 0, False), (8, 13, True), (1, 13, False), (2, 0, True), (2, 13, False), (1, 0, True), (0, 13, True)]
SEEDS = [7, 0x9e3779b9, 12345, 1, 0xffffffff, 42]


def test_each_view_is_its_single_render(scene):
    name, loaded = scene
    cams = V.camera_set(loaded)
    n = 6 if name == "helmet.glb" else 9
    for bounces, begin, distinct in CASES:
        seeds = SEEDS[:len(cams)] if distinct else None
        got = V.device_views(loaded, cams, W, H, begin, begin + n, bounces, seeds)
        if bounces == 0:
            # cast_ray's loop never runs: nothing traced or counted, every slice zeroed (as the renderer does)
            assert not got["accum"].any() and got["counters"] == ZERO_COUNTERS
            continue
        want = V.singles(loaded, cams, W, H, begin, begin + n, bounces, seeds)
        assert_views(got, want)
        assert got["counters"]["samples"] == len(cams) * W * H * n


def test_extended_counters_are_the_sums_of_the_single_renders():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        got = V.device_views(loaded, cams, W, H, 3, 11, 8, SEEDS, n_counters=16)
        want = V.singles(loaded, cams, W, H, 3, 11, 8, SEEDS, n_counters=16)
        assert_views(got, want)
        assert got["counters"]["ex1"] == len(cams) * W * H * 8        # primary rays, sky tiles included
        assert got["counters"]["ex0"] > 0
    finally:
        loaded.close()


def test_order_and_number_of_views_do_not_matter():
    loaded = load("spheres.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        seeds = np.array(SEEDS, np.uint32)
        whole = V.device_views(loaded, cams, W, H, 0, 8, 8, seeds)
        order = [4, 0, 5, 2, 1, 3]
        shuffled = V.device_views(loaded, [cams[k] for k in order], W, H, 0, 8, 8, seeds[order])
        for i, k in enumerate(order):
            assert np.array_equal(V.bits(shuffled["accum"][i]), V.bits(whole["accum"][k]))
        assert shuffled["counters"] == whole["counters"]
        for k in (0, 3, 5):
            one = V.device_views(loaded, [cams[k]], W, H, 0, 8, 8, seeds[k:k + 1])
            assert np.array_equal(V.bits(one["accum"][0]), V.bits(whole["accum"][k]))
        # the same camera twice with the same seed: the same bits; with another seed: other noise
        same = V.device_views(loaded, [cams[1], cams[1], cams[1]], W, H, 0, 8, 8, [5, 5, 6])
        assert np.array_equal(V.bits(same["accum"][0]), V.bits(same["accum"][1]))
        assert not np.array_equal(V.bits(same["accum"][0]), V.bits(same["accum"][2]))
    finally:
        loaded.close()


@pytest.mark.parametrize("name", ["helmet.glb", "spheres.glb"])
def test_two_views_against_the_oracle(name):
    loaded = load(name)
    try:
        upload(loaded)
        cams = [V.orbit(loaded, 3, fov=50.0)[0], V.orbit(loaded, 3, radius_scale=1.6, fov=80.0)[2]]
        seeds = [11, 3]
        w, h, begin, end = 48, 32, 2, 7
        got = V.device_views(loaded, cams, w, h, begin, end, 8, seeds)
        own = V.copy_camera(loaded.scene.camera)
        try:
            for v, cam in enumerate(cams):
                loaded.scene.camera = V.copy_camera(cam)
                ref = oracle_ffi.render(loaded, w, h, end, 8, n_threads=os.cpu_count() or 8, user_seed=seeds[v],
                                        sample_begin=begin, sample_end=end)
                assert np.array_equal(V.bits(got["accum"][v]), V.bits(ref["accum"])), f"view {v}"
        finally:
            loaded.scene.camera = own
    finally:
        loaded.close()


def test_chunked_calls_and_accumulation():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        per_view = ((W + 7) // 8) * ((H + 3) // 4) * 32          # paths of one sample of one view
        whole = V.device_views(loaded, cams, W, H, 1, 21, 8, SEEDS)
        for paths in (per_view, 2 * per_view, 4 * per_view + 100, 5 * per_view + 100):
            # fewer paths than one sample of every view: groups of 1, 2, 4 (then 2) and 5 (then 1) views
            with chunk_paths(paths):
                chunked = V.device_views(loaded, cams, W, H, 1, 21, 8, SEEDS)
            assert_views(chunked, whole)
            assert chunked["launches"] > whole["launches"]
        # [1, 9) then [9, 21) with accumulate equals [1, 21)
        import torch
        acc = torch.full((len(cams) * W * H * 3,), 7.0, dtype=torch.float32, device="cuda")
        V.device_views(loaded, cams, W, H, 1, 9, 8, SEEDS, accum=acc)
        with chunk_paths(2 * per_view):
            cont = V.device_views(loaded, cams, W, H, 9, 21, 8, SEEDS, accum=acc, accumulate=True)
        assert_views(cont, whole, counters=False)
    finally:
        loaded.close()


def test_fast_math_views_are_the_fast_single_renders():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        driver.set_options(fast_math=True)
        got = V.device_views(loaded, cams, W, H, 0, 8, 8, SEEDS)
        want = V.singles(loaded, cams, W, H, 0, 8, 8, SEEDS)
        assert_views(got, want)
        driver.set_options()
        exact = V.device_views(loaded, cams, W, H, 0, 8, 8, SEEDS)
        assert_views(exact, V.singles(loaded, cams, W, H, 0, 8, 8, SEEDS))
    finally:
        driver.set_options()
        loaded.close()


@pytest.mark.parametrize("name", ["helmet.glb", "tower.obj:inside"])
def test_one_view_is_the_render(name):
    loaded = A.load_default_camera("tower.obj") if name.endswith(":inside") else load(name)
    try:
        upload(loaded)
        cam = V.copy_camera(loaded.scene.camera)
        for paths in (None, ((W + 7) // 8) * ((H + 3) // 4) * 32 * 3):
            with (chunk_paths(paths) if paths else contextlib.nullcontext()):
                want = V.device_single(loaded, None, W, H, 2, 19, 8, 77)
                got = V.device_views(loaded, [cam], W, H, 2, 19, 8, [77])
            assert np.array_equal(V.bits(got["accum"][0]), V.bits(want["accum"]))
            assert got["counters"] == want["counters"]
            assert got["launches"] == want["launches"]
    finally:
        loaded.close()


def test_scene_camera_is_untouched_and_used_after():
    loaded = load("sheen.glb")
    try:
        upload(loaded)
        before = V.camera_bytes(loaded.scene.camera)
        first = V.device_single(loaded, None, W, H, 0, 6, 8)
        cams = V.orbit(loaded, 4)
        V.device_views(loaded, cams, W, H, 0, 6, 8)
        assert V.camera_bytes(loaded.scene.camera) == before
        after = V.device_single(loaded, None, W, H, 0, 6, 8)
        assert np.array_equal(V.bits(after["accum"]), V.bits(first["accum"]))
        assert after["counters"] == first["counters"]
    finally:
        loaded.close()


def test_on_a_user_stream_right_after_upload():
    """A fresh scene, uploaded and given a views call at once on a torch stream: the call waits for the texels."""
    import torch
    loaded = load("helmet.glb")
    try:
        cams = V.orbit(loaded, 3)
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        upload(loaded)
        with torch.cuda.stream(stream):
            got = V.device_views(loaded, cams, 128, 96, 0, 4, 8, stream=stream)
        torch.cuda.synchronize()
        assert_views(got, V.singles(loaded, cams, 128, 96, 0, 4, 8))
    finally:
        loaded.close()


def test_interleaved_with_renders_aov_cast_rays_and_a_refit():
    import refit_ffi
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        want = V.singles(loaded, cams, W, H, 0, 6, 8)
        rays_o = np.zeros((64, 3), np.float32)
        rays_d = np.tile(np.array([0.0, 0.0, -1.0], np.float32), (64, 1))
        rays_o[:, 2] = 5.0
        first_cast = driver.cast_rays(loaded, rays_o, rays_d, 4)
        first_aov = A.device_aov(loaded, W, H, 0, 4, 8)
        for _ in range(2):
            driver.render(loaded, 64, 48, 4, 8)
            assert_views(V.device_views(loaded, cams, W, H, 0, 6, 8), want)
            assert np.array_equal(V.bits(driver.cast_rays(loaded, rays_o, rays_d, 4)), V.bits(first_cast))
            assert_views(V.device_views(loaded, cams, W, H, 0, 6, 8), want)
            assert np.array_equal(A.bits(A.device_aov(loaded, W, H, 0, 4, 8)["records"]), A.bits(first_aov["records"]))
        # a refit moves the geometry: the next views call sees it, and each view is the single render after the refit
        pos = driver.scene_positions(loaded)
        moved, _ = refit_ffi.rigid(pos, None, refit_ffi.rotation(0.3, 0.1), (0.05, -0.02, 0.0))
        driver.refit(loaded, moved)
        got = V.device_views(loaded, cams, W, H, 0, 6, 8)
        assert_views(got, V.singles(loaded, cams, W, H, 0, 6, 8))
        assert not np.array_equal(V.bits(got["accum"][0]), V.bits(want["accum"][0]))
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
        cams = V.orbit(loaded, 2)
        carr = (Camera * 2)(*cams)
        acc = torch.full((2 * w * h * 3 + 4,), 7.0, dtype=torch.float32, device="cuda")
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        sc = C.byref(loaded.scene)
        st = torch.cuda.current_stream().cuda_stream

        def dev(scene=sc, n=2, cameras=carr, width=w, height=h, begin=0, end=2, bounces=8, out=acc.data_ptr(), accumulate=0):
            return gpu.rt_gpu_render_views_device(scene, n, cameras, None, width, height, begin, end, bounces, accumulate,
                                                  out, ctr.data_ptr(), st)
        px = np.zeros((2, h, w, 3), np.uint8)

        def host(n=2, cameras=carr, out=None, pixels=px.ctypes.data):
            return gpu.rt_gpu_render_views(sc, n, cameras, None, w, h, 0, 2, 8, out, pixels)
        cases = [
            (lambda: dev(width=0), "empty"),
            (lambda: dev(height=-1), "empty"),
            (lambda: dev(width=1 << 20, height=1 << 12), "too large"),
            (lambda: dev(begin=-1), "samples"),
            (lambda: dev(begin=5, end=4), "samples"),
            (lambda: dev(end=1 << 31), "samples"),
            (lambda: dev(bounces=-1), "max_bounces"),
            (lambda: dev(out=None), "accum"),
            (lambda: dev(n=-1), "n_views"),
            (lambda: dev(cameras=None), "cameras"),
            (lambda: dev(scene=C.byref(other.scene)), "resident"),
            (lambda: dev(scene=None), "scene"),
            (lambda: host(pixels=None), "accum and pixels"),
            (lambda: host(n=-3), "n_views"),
            (lambda: host(cameras=None), "cameras"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in gpu.rt_gpu_last_error().decode(), word
        assert gpu.rt_gpu_scene_device_bytes(C.byref(other.scene)) == 0, "a refused call uploads nothing"
        torch.cuda.synchronize()
        assert (acc == 7).all() and not ctr.any() and not px.any()
        # n_views = 0 is a no-op, NULL cameras included
        assert dev(n=0) == 0 and dev(n=0, cameras=None) == 0 and host(n=0, cameras=None) == 0
        torch.cuda.synchronize()
        assert (acc == 7).all() and not ctr.any()
        # empty range or no bounces: every slice kept with accumulate, zeroed without; nothing traced or counted
        for kw in (dict(begin=5, end=5), dict(bounces=0)):
            assert dev(accumulate=1, **kw) == 0
            torch.cuda.synchronize()
            assert (acc == 7).all()
            assert dev(**kw) == 0
            torch.cuda.synchronize()
            assert not acc[:2 * w * h * 3].any() and (acc[2 * w * h * 3:] == 7).all()
            assert not ctr.any()
            acc.fill_(7.0)
        # the library still answers after the refusals
        assert_views(V.device_views(loaded, cams, w, h, 0, 3, 8), V.singles(loaded, cams, w, h, 0, 3, 8))
    finally:
        other.close()
        loaded.close()


def test_host_form_and_its_film():
    import torch
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        cams = V.camera_set(loaded)
        seeds = np.array(SEEDS, np.uint32)
        pixels, accum = driver.render_views_images(loaded, cams, W, H, 9, 8, sample_begin=3, user_seeds=seeds,
                                                   want_accum=True)
        dev = V.device_views(loaded, cams, W, H, 3, 12, 8, seeds)
        assert np.array_equal(V.bits(accum), V.bits(dev["accum"]))
        st = torch.cuda.current_stream().cuda_stream
        for v in range(len(cams)):
            a = torch.from_numpy(dev["accum"][v]).cuda().contiguous()
            film = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda")
            gpu_check(gpu_lib().rt_gpu_resolve_device(a.data_ptr(), W, H, 9, film.data_ptr(), W, 3, st))
            torch.cuda.synchronize()
            assert np.array_equal(pixels[v], film.cpu().numpy()), f"view {v}"
        # accum alone, pixels alone; an empty range gives black images and zero sums
        only_accum = np.zeros_like(accum)
        gpu_check(gpu_lib().rt_gpu_render_views(C.byref(loaded.scene), len(cams), (Camera * len(cams))(*cams),
                                                seeds.ctypes.data, W, H, 3, 12, 8, only_accum.ctypes.data, None))
        assert np.array_equal(V.bits(only_accum), V.bits(accum))
        assert np.array_equal(driver.render_views_images(loaded, cams, W, H, 9, 8, sample_begin=3, user_seeds=seeds), pixels)
        empty, empty_acc = driver.render_views_images(loaded, cams, W, H, 0, 8, want_accum=True)
        assert not empty.any() and not empty_acc.any()
        # the torch wrapper
        t = torch.full((len(cams), H, W, 3), 7.0, dtype=torch.float32, device="cuda")
        driver.render_views(loaded, cams, t, 3, 12, user_seeds=seeds)
        torch.cuda.synchronize()
        assert np.array_equal(V.bits(t.cpu().numpy()), V.bits(accum))
        with pytest.raises(ValueError):
            driver.render_views(loaded, cams, t[:2], 3, 12)
    finally:
        loaded.close()
