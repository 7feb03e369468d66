"""lightmap_bake (raytracer.h:56, reference raytracer.c:722-784) on the GPU against the CPU oracle's restatement, which
is itself pinned to the reference's own lightmap_bake (tests/test_golden_reference_vectors.py).  Both sides seed per
(texel, sample) (include/rt_seed.h); the f32 value of every texel before the u8 store, the owning triangle and the
u8 lightmap must be identical."""
import numpy as np
import pytest

import oracle_ffi
from helpers import load
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import Vec3, gpu_check

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    gpu_check(gpu_lib().rt_gpu_init(0))
    yield
    driver.set_options()


@pytest.mark.parametrize("name,w,h,samples,seed", [("spheres.glb", 96, 80, 5, 0), ("tower.obj", 128, 64, 3, 9), ("sheen.glb", 64, 64, 4, 1)])
def test_lightmap_values_owner_and_bytes_equal_the_oracle(name, w, h, samples, seed):
    loaded = load(name, emission=Vec3(30.0, 20.0, 10.0))
    try:
        driver.set_options(user_seed=seed)
        before = np.full((h, w, 3), 77, dtype=np.uint8)
        got = driver.lightmap_bake(loaded, w, h, samples, out=before.copy(), want_values=True)
        ref = oracle_ffi.lightmap_bake(loaded, w, h, samples, user_seed=seed)
        assert (ref["owner"] >= 0).sum() > 300, "the model's UVs must cover part of the lightmap"
        assert np.array_equal(got["owner"], ref["owner"])
        assert np.array_equal(got["values"], ref["values"]), "texel values are expected bit-identical"
        written = ref["owner"] >= 0
        assert np.array_equal(got["pixels"][written], ref["pixels"][written])
        assert (got["pixels"][~written] == 77).all(), "untouched texels keep their bytes"
        assert ref["values"].max() > 0.3
    finally:
        driver.set_options()
        loaded.close()


def test_lightmap_through_the_reference_entry_point_and_in_chunks(monkeypatch):
    """lightmap_bake(Image*, Scene*, samples) as raytracer.h declares it; the sample loop cut into several wavefront
    chunks gives the same bytes."""
    loaded = load("tower.obj", emission=Vec3(30.0, 20.0, 10.0))
    try:
        w, h, samples = 80, 60, 6
        whole = driver.lightmap_bake(loaded, w, h, samples)
        ref = oracle_ffi.lightmap_bake(loaded, w, h, samples)
        assert np.array_equal(whole, ref["pixels"]) and whole.max() > 10
        n_jobs = int((ref["owner"] >= 0).sum())
        monkeypatch.setenv("RT_GPU_CHUNK_PATHS", str(n_jobs * 2))        # 2 samples per chunk
        assert np.array_equal(driver.lightmap_bake(loaded, w, h, samples), whole)
        # owner and jobs, 3 chunks x (raygen, 8 x trace / miss / shade, accumulate), store
        assert gpu_lib().rt_gpu_last_launches() == 2 + 3 * (1 + 8 * 3 + 1) + 1
    finally:
        loaded.close()


def test_lightmap_rejects_bad_images():
    loaded = load("quad.obj")
    try:
        with pytest.raises(RuntimeError, match="components"):
            driver.lightmap_bake(loaded, 8, 8, 1, out=np.zeros((8, 8, 1), dtype=np.uint8))
        with pytest.raises(RuntimeError, match="samples"):
            driver.lightmap_bake(loaded, 8, 8, 0)
    finally:
        loaded.close()
