"""The opt-in fast mode (RT_GPU_Options.fast_math, csrc/rt_render_fast.cu): bounce stages FMA-contracted with hardware
transcendentals.  Contract: primary-hit triangle ids stay bit-exact, the picture stays the picture (statistically), and
the default path is untouched."""
import numpy as np
import pytest

import oracle_ffi
from helpers import load
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver

pytestmark = pytest.mark.gpu


def render(loaded, w, h, spp, **opt):
    driver.set_options(keep_hit_ids=True, **opt)
    px = driver.render(loaded, w, h, spp, 8)
    return dict(pixels=px, accum=driver.read_accum(w, h), hit_ids=driver.read_hit_ids(w, h), counters=driver.read_counters())


@pytest.mark.parametrize("name", ["helmet.glb", "spheres.glb"])
def test_fast_mode_keeps_primary_hits_exact_and_the_picture_close(name):
    loaded = load(name)
    try:
        w, h, spp = 320, 180, 256
        exact = render(loaded, w, h, spp)
        fast = render(loaded, w, h, spp, fast_math=True)
        again = render(loaded, w, h, spp)
        ref = oracle_ffi.render(loaded, w, h, 1, n_threads=8, want_hit_ids=True)
        assert np.array_equal(fast["hit_ids"], ref["hit_ids"]), "primary-hit ids must stay bit-exact in fast mode"
        assert np.array_equal(again["accum"], exact["accum"]), "the default path must not be affected by an earlier fast render"
        assert not np.array_equal(fast["accum"], exact["accum"]), "fast mode is expected to differ in the last bits"
        rel = np.abs(fast["accum"] - exact["accum"]) / np.maximum(np.abs(exact["accum"]), 1e-6)
        a, b = fast["pixels"].astype(np.float64) / 255, exact["pixels"].astype(np.float64) / 255
        rmse = float(np.sqrt(np.mean((a - b) ** 2)))
        rays = fast["counters"]["rays"] / exact["counters"]["rays"]
        print(f"\n{name}: fast vs exact at {spp} spp: median rel {np.median(rel):.2e}, 99th pct {np.percentile(rel, 99):.2e}, "
              f"within 1e-3: {(rel <= 1e-3).mean():.4f}, sRGB RMSE {rmse:.5f}, rays ratio {rays:.5f}")
        assert np.median(rel) < 1e-4 and rmse < 0.005 and abs(rays - 1) < 0.01
        lum = np.array([0.2126, 0.7152, 0.0722])
        ratio = float((fast["accum"].astype(np.float64) @ lum).mean() / (exact["accum"].astype(np.float64) @ lum).mean())
        assert abs(ratio - 1.0) < 0.002, f"mean luminance ratio {ratio}"
    finally:
        loaded.close()
