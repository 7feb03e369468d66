"""The CPU reference of rt_gpu_cast_rays (oracle_cast_rays, tests/csrc/cast_rays_oracle.c), which the GPU call is
checked against, pinned:
  - every path equals the oracle's single cast_ray with the generator seeded by hand, and, where a reference checkout is
    available, the reference's own cast_ray seeded the same way;
  - the renderer's camera rays (tests/csrc/camera_rays.c) cast with key = pixel give the oracle renderer's per-sample
    radiance of that sample;
  - a permuted batch with permuted keys gives permuted results.
"""
import numpy as np
import pytest

import cast_rays_ffi as R
import oracle_ffi
import query_ffi as Q
from helpers import load

MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    yield loaded
    loaded.close()


def small_batch(loaded, seed, n_each=12):
    rng = np.random.default_rng(seed)
    sc = loaded.scene
    return np.concatenate([Q.camera_rays(sc, 6, 4), Q.interior_rays(sc, rng, n_each), Q.axis_rays(sc, rng, n_each)])


def test_batch_equals_single_cast_ray(scene):
    rays = small_batch(scene, seed=1)
    keys = np.random.default_rng(2).integers(0, 2**32, size=len(rays), dtype=np.uint32)
    for max_bounces, sample_begin, user_seed, k in ((8, 0, 0, None), (2, 13, 77, keys), (0, 5, 0, keys)):
        got = R.oracle_cast_rays(scene, rays, 3, max_bounces, sample_begin, user_seed, k, n_threads=4)
        for i, ray in enumerate(rays):
            key = int(k[i]) if k is not None else i
            total = np.zeros(3, dtype=np.float32)
            for s in range(3):
                want = R.oracle_cast_ray_seeded(scene, ray, key, sample_begin + s, max_bounces, user_seed)
                assert np.array_equal(R.bits(got["per_sample"][i, s]), R.bits(want)), (i, s)
                total = total + want
            assert np.array_equal(R.bits(got["radiance"][i]), R.bits(total)), i
        assert got["counters"]["samples"] == 3 * len(rays)
        if max_bounces == 0:
            assert not got["radiance"].any() and got["counters"]["rays"] == 0
        else:
            assert got["counters"]["rays"] >= 3 * len(rays)


@pytest.mark.skipif(not Q.ref_available(),
                    reason="needs the reference's own sources (set RT_REFERENCE_DIR to a reference checkout)")
def test_batch_equals_reference_cast_ray(scene):
    rays = small_batch(scene, seed=3, n_each=6)
    got = R.oracle_cast_rays(scene, rays, 2, 8, 9, 5, None, n_threads=2)
    for i, ray in enumerate(rays):
        for s in range(2):
            want = R.ref_cast_ray_seeded(scene, ray, i, 9 + s, 8, 5)
            assert np.array_equal(R.bits(got["per_sample"][i, s]), R.bits(want)), (i, s)


@pytest.mark.parametrize("name", ["spheres.glb", "helmet.glb"])
def test_camera_rays_reproduce_the_renderer(name):
    loaded = load(name)
    try:
        w, h = 24, 16
        pixels = np.arange(w * h, dtype=np.uint32)
        for s in (0, 5, 11):
            rays = R.camera_rays(loaded, w, h, s)
            got = R.oracle_cast_rays(loaded, rays, 1, 8, s, 3, pixels)
            want = oracle_ffi.render(loaded, w, h, s + 1, 8, n_threads=2, user_seed=3, sample_begin=s, sample_end=s + 1,
                                     want_per_sample=True)
            assert np.array_equal(R.bits(got["per_sample"].reshape(h, w, 3)), R.bits(want["per_sample"][:, :, 0])), s
            assert got["counters"] == want["counters"], s
    finally:
        loaded.close()


def test_permuted_keys_permute_the_results():
    loaded = load("helmet.glb")
    try:
        rays = small_batch(loaded, seed=4, n_each=40)
        keys = np.arange(len(rays), dtype=np.uint32) * 7 + 3
        base = R.oracle_cast_rays(loaded, rays, 4, 8, 2, 11, keys)
        perm = np.random.default_rng(5).permutation(len(rays))
        got = R.oracle_cast_rays(loaded, rays[perm], 4, 8, 2, 11, keys[perm])
        assert np.array_equal(R.bits(got["per_sample"]), R.bits(base["per_sample"][perm]))
        assert np.array_equal(R.bits(got["radiance"]), R.bits(base["radiance"][perm]))
        # NULL keys are the indices
        plain = R.oracle_cast_rays(loaded, rays, 4, 8, 2, 11, None)
        idx = R.oracle_cast_rays(loaded, rays, 4, 8, 2, 11, np.arange(len(rays), dtype=np.uint32))
        assert np.array_equal(R.bits(plain["per_sample"]), R.bits(idx["per_sample"]))
        assert not np.array_equal(R.bits(plain["per_sample"]), R.bits(base["per_sample"]))
    finally:
        loaded.close()
