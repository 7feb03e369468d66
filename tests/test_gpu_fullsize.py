"""Parity at the sizes BASELINE.json states (north star: "per-pixel agreement to the reference" at the stated
configs): the sm_100a path through the C ABI against the CPU oracle on the SAME frames —

  config 1  spheres.glb  1024x1024 x 16 spp                    whole image
  config 5  tower.obj    3840x2160 x 16 spp                    whole image
  config 3  helmet.glb   1920x1080 x 64 spp (one wavefront chunk of the headline)   whole image
            helmet.glb   1920x1080 x 1024 spp (the headline)   4096 random pixels + 4 full scanlines

Per-(pixel,sample) seeds make every pixel independent of the others, so a subset of the 1024-spp frame is
checked exactly as the whole frame would be (oracle `pixel_mask`); the oracle does ~50-100 Msamples/s on the GPU
box's host cores, so each case is seconds.  Bar: f32 radiance sums bit-identical (the north star asks 1e-3
relative), u8 film byte-identical, primary-hit slots identical.
"""
import numpy as np
import pytest

import oracle_ffi
from helpers import load
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver

pytestmark = pytest.mark.gpu


def check_frame(name, w, h, spp, mask=None, threads=None):
    import os
    threads = threads or len(os.sched_getaffinity(0))
    loaded = load(name)
    try:
        driver.set_options(keep_hit_ids=True)
        pixels = driver.render(loaded, w, h, spp, 8)
        accum, ids = driver.read_accum(w, h), driver.read_hit_ids(w, h)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=threads, want_hit_ids=True, pixel_mask=mask)
        sel = np.ones((h, w), dtype=bool) if mask is None else mask.astype(bool)
        assert sel.sum() > 0 and (ref["hit_ids"][sel] >= 0).sum() > 100, "the camera must see the model"
        assert np.array_equal(ids[sel], ref["hit_ids"][sel]), "primary-hit slots differ"
        a, b = accum[sel], ref["accum"][sel]
        assert not np.isnan(b).any()
        rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-6)
        assert rel.max() <= 1e-3, f"north-star tolerance violated: max rel {rel.max()}"
        assert np.array_equal(a, b), f"radiance sums expected bit-identical; max rel {rel.max()}"
        assert np.array_equal(pixels[sel], ref["pixels"][sel]), "u8 film differs"
        return int(sel.sum())
    finally:
        driver.set_options()
        loaded.close()


def test_config1_spheres_1024x1024_16spp_whole_image():
    assert check_frame("spheres.glb", 1024, 1024, 16) == 1024 * 1024


def test_config5_tower_4k_16spp_whole_image():
    assert check_frame("tower.obj", 3840, 2160, 16) == 3840 * 2160


def test_config3_helmet_1080p_64spp_whole_image():
    assert check_frame("helmet.glb", 1920, 1080, 64) == 1920 * 1080


def headline_mask(w=1920, h=1080, n_random=4096, seed=2026):
    """4096 random pixels + 4 full scanlines (one through sky only, three through the helmet)."""
    rng = np.random.default_rng(seed)
    mask = np.zeros((h, w), dtype=np.uint8)
    flat = rng.choice(w * h, size=n_random, replace=False)
    mask.reshape(-1)[flat] = 1
    for y in (h // 8, h // 3, h // 2, (2 * h) // 3):
        mask[y, :] = 1
    return mask


def test_config3_helmet_1080p_1024spp_headline_subset():
    mask = headline_mask()
    assert check_frame("helmet.glb", 1920, 1080, 1024, mask=mask) >= 4096 + 4 * 1920 - 64
