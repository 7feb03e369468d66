"""Radiance for caller rays on the GPU (rt_gpu_cast_rays*, csrc/rt_render.cu) against its CPU reference (oracle_cast_rays):
every per-sample value, every sum and the eight work counters bit-exact on the six shipped models, for every ray family,
bounce count, seed, sample offset and key mode; the renderer's own per-sample radiance reproduced from its camera rays;
split calls, subsets and chunked batches equal to the single call; the host form equal to the device form; ordering
against uploads, renders and queries; refusals before launch.  The kernels' register budgets are in
test_build_properties.py.
"""
import ctypes as C

import numpy as np
import pytest

import cast_rays_ffi as R
import query_ffi as Q
from helpers import MODEL_NAMES, chunk_paths, load, upload
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    upload(loaded)
    yield loaded
    loaded.close()


def all_families(loaded, seed, n_each=256, grid=(32, 24)):
    """camera grid, interior (normalised and not), axis-aligned / zero components, surface-offset rays"""
    rays, _ = Q.mixed_rays(loaded, seed=seed, n_each=n_each, grid=grid)
    return rays


def assert_equal(got, want, per_sample=True):
    if per_sample:
        bad = R.bits(got["per_sample"]) != R.bits(want["per_sample"])
        assert not bad.any(), f"per-sample radiance differs on {int(bad.any(axis=-1).sum())} paths"
    assert np.array_equal(R.bits(got["radiance"]), R.bits(want["radiance"])), "sums differ"
    assert got["counters"] == want["counters"]


# (max_bounces, user_seed, sample_begin, keys given)
CASES = [(8, 0, 0, False), (8, 0x9E37, 13, True), (0, 0, 13, True), (1, 0x9E37, 0, False), (2, 0, 13, True),
         (2, 0x9E37, 0, False), (1, 0, 13, True)]


def test_bit_exact_against_the_oracle(scene):
    rays = all_families(scene, seed=70)
    keys = np.random.default_rng(71).integers(0, 2**32, size=len(rays), dtype=np.uint32)
    for max_bounces, user_seed, sample_begin, with_keys in CASES:
        k = keys if with_keys else None
        want = R.oracle_cast_rays(scene, rays, 4, max_bounces, sample_begin, user_seed, k)
        got = R.device_cast_rays(scene, rays, 4, max_bounces, sample_begin, user_seed, k)
        assert_equal(got, want)
        assert got["counters"]["samples"] == 4 * len(rays)
    assert want["counters"]["shades"] > 0 and want["counters"]["misses"] > 0


@pytest.mark.parametrize("name", ["helmet.glb", "spheres.glb"])
def test_camera_rays_reproduce_the_renderers_samples(name):
    import torch
    loaded = load(name)
    try:
        w, h, n_s, seed = 256, 192, 14, 5
        upload(loaded)
        accum = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
        per = torch.zeros(h * w * n_s * 3, dtype=torch.float32, device="cuda")
        gpu_check(gpu_lib().rt_gpu_render_accum_device(C.byref(loaded.scene), w, h, 0, n_s, 8, seed, 0, accum.data_ptr(),
                                                       per.data_ptr(), None, None, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        rendered = per.cpu().numpy().reshape(h * w, n_s, 3)
        pixels = np.arange(w * h, dtype=np.uint32)
        for s in (0, 5, 13):
            got = R.device_cast_rays(loaded, R.camera_rays(loaded, w, h, s), 1, 8, s, seed, pixels)
            assert np.array_equal(R.bits(got["per_sample"][:, 0]), R.bits(rendered[:, s])), s
            assert np.array_equal(R.bits(got["radiance"]), R.bits(rendered[:, s])), s
    finally:
        loaded.close()


def test_split_calls_and_subsets_equal_one_call():
    import torch
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        rays = all_families(loaded, seed=72, n_each=1024)
        keys = np.arange(len(rays), dtype=np.uint32) * 3 + 1
        full = R.device_cast_rays(loaded, rays, 10, 8, 3, 9, keys)
        rad = torch.full((len(rays), 3), 7.0, dtype=torch.float32, device="cuda")
        a = R.device_cast_rays(loaded, rays, 4, 8, 3, 9, keys, radiance=rad)
        b = R.device_cast_rays(loaded, rays, 6, 8, 7, 9, keys, radiance=rad, accumulate=True)
        assert np.array_equal(R.bits(b["radiance"]), R.bits(full["radiance"]))
        assert np.array_equal(R.bits(np.concatenate([a["per_sample"], b["per_sample"]], axis=1)), R.bits(full["per_sample"]))
        assert {k: a["counters"][k] + b["counters"][k] for k in a["counters"]} == full["counters"]
        idx = np.sort(np.random.default_rng(73).choice(len(rays), size=300, replace=False))
        sub = R.device_cast_rays(loaded, rays[idx], 10, 8, 3, 9, keys[idx])
        assert np.array_equal(R.bits(sub["per_sample"]), R.bits(full["per_sample"][idx]))
        assert np.array_equal(R.bits(sub["radiance"]), R.bits(full["radiance"][idx]))
    finally:
        loaded.close()


def test_chunked_batches():
    """Batches larger than one chunk of path queues: split over rays (70001 rays x 3 samples in chunks of 33333 rays) and
    over samples (3000 rays x 100 samples in chunks of 33 samples).  The chunked results equal the unchunked call on every
    ray, and the oracle on a seeded subset that includes both sides of every chunk boundary."""
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        rng = np.random.default_rng(74)
        for n, samples, boundaries in ((70001, 3, [0, 33332, 33333, 66665, 66666, 70000]), (3000, 100, [0, 2999])):
            rays = Q.interior_rays(loaded.scene, rng, n)
            whole = R.device_cast_rays(loaded, rays, samples, 8, 1, 4)
            with chunk_paths(100000):
                got = R.device_cast_rays(loaded, rays, samples, 8, 1, 4)
            assert_equal(got, whole)
            idx = np.unique(np.concatenate([boundaries, rng.choice(n, size=40, replace=False)]))
            want = R.oracle_cast_rays(loaded, rays[idx], samples, 8, 1, 4, idx.astype(np.uint32))
            assert np.array_equal(R.bits(got["per_sample"][idx]), R.bits(want["per_sample"]))
            assert np.array_equal(R.bits(got["radiance"][idx]), R.bits(want["radiance"]))
    finally:
        loaded.close()


def test_host_form_equals_device_form():
    loaded = load("sheen.glb")
    try:
        upload(loaded)
        rays = all_families(loaded, seed=75)
        keys = np.random.default_rng(76).integers(0, 2**32, size=len(rays), dtype=np.uint32)
        dev = R.device_cast_rays(loaded, rays, 5, 8, 2, 6, keys)
        rad, per = driver.cast_rays(loaded, rays[:, :3], rays[:, 3:], 5, 8, sample_begin=2, user_seed=6, keys=keys,
                                    per_sample=True)
        assert np.array_equal(R.bits(rad), R.bits(dev["radiance"]))
        assert np.array_equal(R.bits(per), R.bits(dev["per_sample"]))
        plain = driver.cast_rays(loaded, rays[:, :3], rays[:, 3:], 5, 8, sample_begin=2, user_seed=6)
        assert gpu_lib().rt_gpu_last_launches() == 1 + 3 * 8 + 1       # one chunk: raygen, 8 x (trace, miss, shade), sum
        assert np.array_equal(R.bits(plain), R.bits(R.device_cast_rays(loaded, rays, 5, 8, 2, 6)["radiance"]))
    finally:
        loaded.close()


def test_on_a_user_stream_right_after_upload():
    """A fresh scene, uploaded and cast at once on a torch stream: the call waits for the texels."""
    import torch
    loaded = load("helmet.glb")
    try:
        rays = all_families(loaded, seed=77, n_each=1024)
        r = torch.from_numpy(rays).cuda()
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        upload(loaded)
        with torch.cuda.stream(stream):
            got = R.device_cast_rays(loaded, r, 2, 8, 0, 8, stream=stream)
        torch.cuda.synchronize()
        assert_equal(got, R.device_cast_rays(loaded, rays, 2, 8, 0, 8))
        assert_equal(got, R.oracle_cast_rays(loaded, rays, 2, 8, 0, 8))
    finally:
        loaded.close()


def test_interleaving_leaves_results_unchanged():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h, spp = 160, 90, 4
        rays = all_families(loaded, seed=78, n_each=2048)
        driver.render(loaded, w, h, spp, 8)
        first = driver.read_accum(w, h).copy()
        before = R.device_cast_rays(loaded, rays, 3, 8, 0, 1)
        driver.render(loaded, w, h, spp, 8)
        assert np.array_equal(R.bits(driver.read_accum(w, h)), R.bits(first))
        driver.closest_hit(loaded, rays[:, :3], rays[:, 3:], surface=True)
        assert_equal(R.device_cast_rays(loaded, rays, 3, 8, 0, 1), before)
    finally:
        loaded.close()


def test_fast_math_option_does_not_apply():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        rays = all_families(loaded, seed=79)
        want = R.oracle_cast_rays(loaded, rays, 3, 8, 0, 2)
        driver.set_options(fast_math=True)
        assert_equal(R.device_cast_rays(loaded, rays, 3, 8, 0, 2), want)
    finally:
        driver.set_options()
        loaded.close()


def test_refusals_and_empty_calls():
    import torch
    loaded = load("quad.obj")
    other = load("quad.obj")
    try:
        upload(loaded)
        gpu = gpu_lib()
        rays = Q.interior_rays(loaded.scene, np.random.default_rng(80), 64)
        r = torch.from_numpy(rays).cuda()
        rad = torch.full((64, 3), 7.0, dtype=torch.float32, device="cuda")
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        sc = C.byref(loaded.scene)
        st = torch.cuda.current_stream().cuda_stream

        def dev(scene=sc, rays_p=r.data_ptr(), n=64, begin=0, samples=2, bounces=8, out=rad.data_ptr()):
            return gpu.rt_gpu_cast_rays_device(scene, rays_p, None, n, begin, samples, bounces, 0, 0, out, None,
                                               ctr.data_ptr(), st)
        cases = [
            (lambda: dev(n=-1), "n_rays"),
            (lambda: dev(n=1 << 31), "n_rays"),
            (lambda: dev(samples=-1), "samples"),
            (lambda: dev(begin=-1), "samples"),
            (lambda: dev(begin=(1 << 31) - 2, samples=2), "samples"),
            (lambda: dev(bounces=-1), "max_bounces"),
            (lambda: dev(rays_p=None), "rays"),
            (lambda: dev(out=None), "radiance"),
            (lambda: dev(scene=C.byref(other.scene)), "resident"),
            (lambda: dev(scene=None), "scene"),
            (lambda: gpu.rt_gpu_cast_rays(sc, None, None, 3, 0, 1, 8, 0, 0, None, None), "rays"),
            (lambda: gpu.rt_gpu_cast_rays(sc, rays.ctypes.data, None, -3, 0, 1, 8, 0, 0, None, None), "n_rays"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in gpu.rt_gpu_last_error().decode(), word
        assert gpu.rt_gpu_scene_device_bytes(C.byref(other.scene)) == 0, "a refused call uploads nothing"
        # n_rays = 0 touches nothing, even with null pointers
        assert dev(n=0) == 0 and dev(n=0, rays_p=None, out=None) == 0
        assert gpu.rt_gpu_cast_rays(sc, None, None, 0, 0, 4, 8, 0, 0, None, None) == 0
        torch.cuda.synchronize()
        assert (rad == 7).all() and not ctr.any()
        # an empty sample range: sums zeroed, or kept with accumulate; nothing traced
        assert gpu.rt_gpu_cast_rays_device(sc, r.data_ptr(), None, 64, 5, 0, 8, 0, 1, rad.data_ptr(), None, ctr.data_ptr(), st) == 0
        torch.cuda.synchronize()
        assert (rad == 7).all()
        assert dev(samples=0) == 0
        torch.cuda.synchronize()
        assert (rad == 0).all() and not ctr.any()
        # the library still answers after the refusals
        assert_equal(R.device_cast_rays(loaded, rays, 2, 8, 0, 0), R.oracle_cast_rays(loaded, rays, 2, 8, 0, 0))
    finally:
        other.close()
        loaded.close()
