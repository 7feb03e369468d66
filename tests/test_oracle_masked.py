"""The CPU reference of rt_gpu_render_masked_device, which the GPU tests compare against: the oracle renderer with a
pixel_mask, and the second moments summed from its per-sample radiance.
  - on the selected pixels a masked oracle run gives the unmasked run's per-sample radiance and sums bit for bit, the
    unselected pixels stay 0, and the counters of a mask and of its complement add up to the unmasked counters;
  - a sequential numpy float32 sum over the oracle's per_sample equals its accum bit for bit, which is what licenses
    computing the reference second moments the same way.
"""
import numpy as np
import pytest

import masked_ffi as M
import oracle_ffi
from helpers import load

MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    yield loaded
    loaded.close()


@pytest.mark.parametrize("begin,end,bounces", [(0, 8, 8), (5, 13, 2)])
def test_masked_oracle_is_the_unmasked_oracle_on_selected_pixels(scene, begin, end, bounces):
    w, h = 40, 28
    mask = M.masks(w, h)["random30"]
    full = oracle_ffi.render(scene, w, h, end, bounces, n_threads=4, sample_begin=begin, sample_end=end,
                             want_per_sample=True)
    part = oracle_ffi.render(scene, w, h, end, bounces, n_threads=4, sample_begin=begin, sample_end=end,
                             want_per_sample=True, pixel_mask=mask)
    rest = oracle_ffi.render(scene, w, h, end, bounces, n_threads=4, sample_begin=begin, sample_end=end,
                             pixel_mask=1 - mask)
    sel = mask != 0
    assert np.array_equal(M.bits(part["per_sample"][sel]), M.bits(full["per_sample"][sel]))
    assert np.array_equal(M.bits(part["accum"][sel]), M.bits(full["accum"][sel]))
    assert not part["accum"][~sel].any() and not part["per_sample"][~sel].any()
    assert part["counters"]["samples"] == int(sel.sum()) * (end - begin)
    assert {k: part["counters"][k] + rest["counters"][k] for k in full["counters"]} == full["counters"]


def test_sequential_float32_sum_of_per_sample_is_the_accumulator(scene):
    w, h = 32, 24
    out = oracle_ffi.render(scene, w, h, 24, 8, n_threads=4, sample_begin=3, sample_end=24, want_per_sample=True)
    s, q = M.sequential_sums(out["per_sample"])
    assert np.array_equal(M.bits(s), M.bits(out["accum"]))
    # the second moment is the same loop over v * v: non-negative, and at least sum^2 / n (Cauchy-Schwarz, up to rounding)
    fin = np.isfinite(q) & np.isfinite(s)
    assert fin.mean() > 0.99
    n = out["per_sample"].shape[2]
    assert (q[fin] >= 0).all() and (q[fin] * n >= s[fin] * s[fin] * (1 - 1e-4)).all()
