"""Cross-check: the oracle against the reference's own sources.

The live comparison needs oracle/_ref/libref.so, built by `make -C oracle ref` from a reference checkout named by
RT_REFERENCE_DIR.  Where it is absent, every test compares the oracle with what the reference produced when
tools/make_golden.py last ran it (tests/golden/reference_vectors.*), and skips, saying how to record it, where that
output was never stored.  REFERENCE seed mode (one sequential RNG stream from 0, single thread, _mm256_rsqrt_ps primary
rays — raytracer.c:596-720 exactly as written) depends on the CPU's rsqrt approximation: its stored images are used
only where this CPU's _mm256_rsqrt_ps matches the recording CPU's on the stored inputs.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_ffi
import ref_ffi
from helpers import MODELS, CAMERAS, golden, load, scene_buffers, scene_digest
from raytracing_c_b200 import _ffi, driver

ARRAYS, META = golden()
LIVE = ref_ffi.available()

# sizeof in the reference's headers (ref_sizeof_*), as its own build reported them
REFERENCE_SIZES = {"triangle": 112, "triangle_aos": 112, "bvh_node": 192, "scene": 208, "context": 80}


def stored(key):
    if key not in ARRAYS.files:
        pytest.skip(f"no live reference (set RT_REFERENCE_DIR to a reference checkout) and no stored output '{key}' "
                    "(tools/make_golden.py records it from that checkout)")
    return ARRAYS[key]


def load_oracle(name, **override):
    return load(name, builder=oracle_ffi.lib().oracle_scene_init, **override)


def load_pair(name, **override):
    r = ref_ffi.lib()
    cam = driver.look_at(**CAMERAS[name]) if name in CAMERAS else None
    a = driver.load_scene(f"{MODELS}/{name}", shader_proc=r.ref_shader_proc(), background_proc=r.ref_background_proc(),
                          builder=ref_ffi.scene_builder(), camera=cam)
    for i in range(a.model.n_materials):
        for k, v in override.items():
            setattr(a.model.materials[i], k, v)
    return a, load_oracle(name, **override)


def test_struct_sizes_match_reference_headers():
    if LIVE:
        r = ref_ffi.lib()
        assert {k: getattr(r, f"ref_sizeof_{k}")() for k in REFERENCE_SIZES} == REFERENCE_SIZES
    ours = {"triangle": C.sizeof(_ffi.Triangle), "triangle_aos": _ffi.TRIANGLE_AOS_BYTES, "bvh_node": _ffi.BVH_NODE_BYTES,
            "scene": C.sizeof(_ffi.Scene), "context": C.sizeof(_ffi.RenderingContext)}
    assert ours == REFERENCE_SIZES


@pytest.mark.parametrize("name", ["spheres.glb", "sheen.glb", "tower.obj", "helmet.glb"])
def test_scene_init_bytes(name):
    """Live: the reference's scene_init and the oracle's give the same bytes.  Without the reference this is the
    stored-digest check test_golden_reference_vectors.py::test_bvh_layout_matches_reference_scene_init also makes."""
    if not LIVE:
        loaded = load_oracle(name)
        try:
            assert scene_digest(loaded.scene) == META["bvh"][name]["sha256"]
        finally:
            loaded.close()
        return
    a, b = load_pair(name)
    try:
        assert scene_buffers(a.scene) == scene_buffers(b.scene)
    finally:
        a.close(); b.close()


@pytest.mark.parametrize("name,w,h,spp,override", [
    ("spheres.glb", 96, 64, 4, {}),
    ("helmet.glb", 64, 48, 3, {}),
    ("sheen.glb", 48, 48, 4, {"sheen": 1.0, "sheen_tint": 1.0}),
    ("tower.obj", 48, 32, 2, {}),
])
def test_reference_mode_image_is_identical(name, w, h, spp, override):
    """render_thread_proc as shipped (T=1) vs the oracle in reference seed mode: same u8 image."""
    if LIVE:
        a, b = load_pair(name, **override)
        try:
            want = ref_ffi.render_reference_mode(a, w, h, spp)
        finally:
            a.close()
    else:
        want = stored(f"reference_mode/{name}_{w}x{h}x{spp}")
        if not np.array_equal(oracle_ffi.rsqrt_ps(ARRAYS["rsqrt_in"]), ARRAYS["rsqrt_out"]):
            pytest.skip("this CPU's _mm256_rsqrt_ps differs from the one the stored reference images were recorded on")
        b = load_oracle(name, **override)
    try:
        got = oracle_ffi.render(b, w, h, spp, 8, n_threads=1, seed_mode=oracle_ffi.SEED_REFERENCE, approx_rsqrt=True)["pixels"]
        assert want.any()
        assert np.array_equal(got, want)
    finally:
        b.close()


def test_per_sample_mode_and_denoiser():
    """cast_ray per (pixel, sample) with user seed 99, and denoise_image on the oracle's u8 frame of that render."""
    if LIVE:
        a, b = load_pair("spheres.glb")
        try:
            want = ref_ffi.cast_rays_per_sample(a, 20, 12, 3, user_seed=99)
        finally:
            a.close()
    else:
        want = stored("per_sample/spheres.glb_20x12x3_seed99")
        frame_in, frame_out = stored("denoise_frame_in"), stored("denoise_frame_out")
        b = load_oracle("spheres.glb")
    try:
        got = oracle_ffi.render(b, 20, 12, 3, 8, n_threads=2, user_seed=99, want_per_sample=True)
        assert np.array_equal(got["per_sample"], want)
        if LIVE:
            assert np.array_equal(ref_ffi.denoise(got["pixels"]), oracle_ffi.denoise(got["pixels"]))
        else:
            assert np.array_equal(got["pixels"], frame_in)
            assert np.array_equal(oracle_ffi.denoise(frame_in), frame_out)
    finally:
        b.close()
