"""The oracle against golden vectors produced by the reference's OWN code.

tests/golden/reference_vectors.npz was generated (tools/make_golden.py) by oracle/_ref/libref.so —
raytracer.c, scene.c, denoiser.c and driver.c compiled unmodified over the Codin stand-in.  These
tests need neither the reference checkout nor a GPU; they are what pins the oracle on every machine.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_ffi
from helpers import golden, load, scene_digest
from raytracing_c_b200._ffi import Vec2, Vec3

ARRAYS, META = golden()


@pytest.mark.parametrize("model", sorted(META["bvh"]))
def test_bvh_layout_matches_reference_scene_init(model):
    """BVH node bytes + SoA + AoS records of the oracle builder AND the product host builder
    (scene_init in librt_host.so) equal the reference scene.c:416 byte for byte."""
    want = META["bvh"][model]
    for builder in (oracle_ffi.lib().oracle_scene_init, None):
        loaded = load(model, builder=builder)
        try:
            assert int(loaded.scene.bvh.depth) == want["depth"]
            assert int(loaded.scene.bvh.nodes.len) == want["nodes"]
            assert int(loaded.scene.triangles.len) == want["slots"]
            assert scene_digest(loaded.scene) == want["sha256"]
        finally:
            loaded.close()


@pytest.mark.parametrize("case", sorted(META["radiance_cases"]))
def test_radiance_per_sample_matches_reference_cast_ray(case):
    cfg = META["radiance_cases"][case]
    loaded = load(cfg["model"], camera=cfg["camera"], **cfg["override"])
    try:
        got = oracle_ffi.render(loaded, cfg["width"], cfg["height"], cfg["spp"], cfg["bounces"], n_threads=2,
                                want_per_sample=True)["per_sample"]
        want = ARRAYS["radiance/" + case]
        assert want.shape == got.shape and (want > 0).any()
        assert np.array_equal(got, want)
    finally:
        loaded.close()


def test_denoiser_matches_reference():
    assert np.array_equal(oracle_ffi.denoise(ARRAYS["denoise_in"], n_threads=3), ARRAYS["denoise_out"])


def test_hash12_matches_reference():
    got = np.array([oracle_ffi.lib().oracle_hash12(float(a), float(b)) for a, b in ARRAYS["hash12_xy"]], dtype=np.float32)
    assert np.array_equal(got, ARRAYS["hash12_out"])


def test_texture_and_environment_match_reference():
    loaded = load("sheen.glb")
    try:
        o = oracle_ffi.lib()
        got = np.array([(c.x, c.y, c.z) for c in (o.oracle_sample_texture_bilinear(C.byref(loaded.background), Vec2(*p))
                                                  for p in ARRAYS["bilinear_uv"])], dtype=np.float32)
        assert np.array_equal(got, ARRAYS["bilinear_out"])
        got = np.array([(c.x, c.y, c.z) for c in (o.oracle_sample_background(C.addressof(loaded.background), Vec3(*p))
                                                  for p in ARRAYS["background_dir"])], dtype=np.float32)
        assert np.array_equal(got, ARRAYS["background_out"])
    finally:
        loaded.close()


@pytest.mark.parametrize("case", sorted(META["lightmap_cases"]))
def test_lightmap_bake_matches_reference(case):
    """oracle_lightmap_bake in the reference's sequential seed mode against the reference's own lightmap_bake
    (raytracer.c:722-784): same u8 lightmap, overlapping triangles and out-of-range texels included."""
    cfg = META["lightmap_cases"][case]
    loaded = load(cfg["model"], emission=Vec3(*cfg["emission"]))
    try:
        got = oracle_ffi.lightmap_bake(loaded, cfg["width"], cfg["height"], cfg["samples"], seed_mode=oracle_ffi.SEED_REFERENCE,
                                       dir_state=cfg["dir_state"], shader_state=cfg["shader_state"])
        want = ARRAYS["lightmap/" + case]
        assert (want > 0).sum() > 100 and got["stores"] > (got["owner"] >= 0).sum()      # texels are overwritten: order matters
        assert np.array_equal(got["pixels"], want)
    finally:
        loaded.close()


def test_lightmap_per_sample_seeding_is_order_free():
    """The per-(texel, sample) seeding rule the GPU shares: a texel's value depends only on the LAST triangle that
    covers it, so baking is independent of how the work is scheduled."""
    loaded = load("spheres.glb", emission=Vec3(30.0, 20.0, 10.0))
    try:
        a = oracle_ffi.lightmap_bake(loaded, 40, 40, 2)
        b = oracle_ffi.lightmap_bake(loaded, 40, 40, 2, dir_state=555, shader_state=777)     # stream states are ignored
        assert np.array_equal(a["values"], b["values"]) and np.array_equal(a["pixels"], b["pixels"])
        assert (a["owner"] >= 0).sum() > 500 and a["values"].max() > 1.0
    finally:
        loaded.close()
