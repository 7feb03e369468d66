"""GPU parity tests: the sm_100a path, called through the C ABI, against the CPU oracle.

Bar (BASELINE.json north_star): BVH layout and primary-hit slots bit-exact; per-pixel radiance
with identical per-(pixel,sample) RNG streams within 1e-3 relative — here it is asserted EXACT
(0 ulp) because both sides share rt_math.h and run without FMA contraction; the u8 film and the
denoiser output byte-exact.  Sizes are chosen so the oracle finishes in seconds.
"""
import os

import numpy as np
import pytest

import oracle_ffi
from helpers import MODELS, load
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu


def gpu_render(loaded, w, h, spp, bounces=8, n_threads=1, **options):
    driver.set_options(keep_hit_ids=True, **options)
    pixels = driver.render(loaded, w, h, spp, bounces, n_threads=n_threads)
    return dict(pixels=pixels, accum=driver.read_accum(w, h), hit_ids=driver.read_hit_ids(w, h),
                counters=driver.read_counters())


@pytest.mark.parametrize("name", ["quad.obj", "fov_test.obj"])
def test_primary_hit_ids_bit_exact_1024(name):
    """BASELINE config 2: 1024x1024, 1 spp, slot ids (raytracer.c:162) identical to the oracle."""
    loaded = load(name)
    try:
        got = gpu_render(loaded, 1024, 1024, 1)
        ref = oracle_ffi.render(loaded, 1024, 1024, 1, n_threads=8, want_hit_ids=True)
        assert (ref["hit_ids"] >= 0).sum() > 1000, "camera must see the model"
        assert np.array_equal(got["hit_ids"], ref["hit_ids"])
        assert np.array_equal(got["accum"], ref["accum"])
        assert np.array_equal(got["pixels"], ref["pixels"])
    finally:
        loaded.close()


@pytest.mark.parametrize("name,w,h,spp", [
    ("spheres.glb", 256, 256, 16),      # config 1 at reduced resolution
    ("helmet.glb", 240, 136, 8),        # config 3 aspect, textured PBR + normal map + emission
    ("tower.obj", 192, 108, 8),         # config 5 aspect
    ("sheen.glb", 128, 128, 8),
])
def test_radiance_exact_vs_oracle(name, w, h, spp):
    loaded = load(name)
    try:
        got = gpu_render(loaded, w, h, spp)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=8, want_hit_ids=True)
        assert np.array_equal(got["hit_ids"], ref["hit_ids"])
        assert not np.isnan(ref["accum"]).any()
        rel = np.abs(got["accum"] - ref["accum"]) / np.maximum(np.abs(ref["accum"]), 1e-6)
        assert rel.max() <= 1e-3, f"north-star tolerance violated: {rel.max()}"
        assert np.array_equal(got["accum"], ref["accum"]), "radiance is expected to be bit-identical"
        assert np.array_equal(got["pixels"], ref["pixels"])
        assert got["counters"] == ref["counters"], "work counters (rays, node/leaf visits, shades) differ"
    finally:
        loaded.close()


def _write_triangle_soup(path, n_triangles, seed):
    """An OBJ of small random triangles in a 4 x 4 x 4 cube (no normals, no material file)."""
    rng = np.random.default_rng(seed)
    centre = rng.uniform(-2.0, 2.0, size=(n_triangles, 1, 3))
    verts = (centre + rng.uniform(-0.06, 0.06, size=(n_triangles, 3, 3))).reshape(-1, 3)
    with open(path, "w") as f:
        f.write("".join(f"v {x:.6f} {y:.6f} {z:.6f}\n" for x, y, z in verts))
        f.write("".join(f"f {3 * i + 1} {3 * i + 2} {3 * i + 3}\n" for i in range(n_triangles)))


@pytest.mark.parametrize("n_triangles,expect_root_children", [(30000, 8), (9000, 3)])
def test_generated_scene_full_and_sparse_root(tmp_path, n_triangles, expect_root_children):
    """The trace kernel skips the box tests of the root's padding children (rt_trace.cuh, walk_node_step<ROOT>).  The shipped
    models fill at most four of the root's eight children; 30 000 triangles fill all eight (depth 4 holds 32 768), 9 000
    fill three.  Radiance, primary-hit slots and the node / leaf visit counters must equal the oracle's on both."""
    path = str(tmp_path / f"soup_{n_triangles}.obj")
    _write_triangle_soup(path, n_triangles, seed=n_triangles)
    cam = driver.look_at(eye=(0.3, 0.4, 6.0), target=(0.0, 0.0, 0.0))
    loaded = driver.load_scene(path, shader_proc=oracle_ffi.shader_proc(), background_proc=oracle_ffi.background_proc(), camera=cam)
    try:
        n_int = loaded.scene.bvh.last_row_offset
        import ctypes as C
        root = np.ctypeslib.as_array(C.cast(loaded.scene.bvh.nodes.data, C.POINTER(C.c_float)), shape=(n_int, 6, 8))[0]
        assert int((root[:3] != root[3:]).any(axis=0).sum()) == expect_root_children
        w, h, spp = 160, 120, 4
        got = gpu_render(loaded, w, h, spp)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=8, want_hit_ids=True)
        assert (ref["hit_ids"] >= 0).sum() > 1000, "camera must see the triangles"
        assert np.array_equal(got["hit_ids"], ref["hit_ids"])
        assert np.array_equal(got["accum"], ref["accum"])
        assert got["counters"] == ref["counters"]
    finally:
        loaded.close()


@pytest.mark.parametrize("sheen_tint", [0.0, 1.0])
def test_sheen_injected_and_denoised(sheen_tint):
    """BASELINE config 4: sheen.glb carries no KHR_materials_sheen, so sheen is injected."""
    loaded = load("sheen.glb", sheen=1.0, sheen_tint=sheen_tint)
    plain = load("sheen.glb")
    try:
        w = h = 160
        got = gpu_render(loaded, w, h, 8)
        ref = oracle_ffi.render(loaded, w, h, 8, n_threads=8)
        base = oracle_ffi.render(plain, w, h, 8, n_threads=8)
        assert not np.array_equal(ref["accum"], base["accum"]), "the sheen lobe must change the image"
        assert np.array_equal(got["accum"], ref["accum"])
        assert np.array_equal(got["pixels"], ref["pixels"])
        assert np.array_equal(driver.denoise(got["pixels"]), oracle_ffi.denoise(ref["pixels"]))
    finally:
        loaded.close()
        plain.close()


def test_anisotropic_material():
    loaded = load("spheres.glb", anisotropic_strength=0.7)
    try:
        got = gpu_render(loaded, 128, 128, 4)
        ref = oracle_ffi.render(loaded, 128, 128, 4, n_threads=8)
        assert np.array_equal(got["accum"], ref["accum"])
    finally:
        loaded.close()


def test_random_image_shapes_sample_counts_and_chunks(monkeypatch):
    """Random widths, heights, sample counts, bounce limits and wavefront-chunk sizes (odd ones included): the path id ->
    (pixel, sample) and tile -> (x, y) decode divides by multiply-high with per-launch magic numbers (rt_fastdiv.h), the
    samples of a chunk and the tiles of a row are the divisors.  Radiance, primary-hit slots and counters equal the oracle's."""
    rng = np.random.default_rng(20261018)
    loaded = load("spheres.glb")
    try:
        for _ in range(12):
            w, h = int(rng.integers(1, 200)), int(rng.integers(1, 140))
            spp, bounces = int(rng.integers(1, 24)), int(rng.integers(1, 9))
            per_sample = ((w + 7) // 8) * ((h + 3) // 4) * 32
            monkeypatch.setenv("RT_GPU_CHUNK_PATHS", str(per_sample * int(rng.integers(1, spp + 1))))
            got = gpu_render(loaded, w, h, spp, bounces)
            ref = oracle_ffi.render(loaded, w, h, spp, bounces, n_threads=8, want_hit_ids=True)
            assert np.array_equal(got["hit_ids"], ref["hit_ids"]), (w, h, spp, bounces)
            assert np.array_equal(got["accum"], ref["accum"]), (w, h, spp, bounces)
            assert got["counters"] == ref["counters"], (w, h, spp, bounces)
    finally:
        loaded.close()


@pytest.mark.parametrize("shape", [(1, 1), (7, 5), (33, 31), (64, 64), (257, 130)])
def test_denoiser_byte_exact_random(shape):
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w)
    img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    # smooth regions + salt noise so both blend branches are exercised
    img[: h // 2] = (img[: h // 2] // 32) * 32
    assert np.array_equal(driver.denoise(img), oracle_ffi.denoise(img))


def test_denoiser_constant_and_ties():
    img = np.full((40, 50, 3), 128, dtype=np.uint8)
    img[10, 10] = (255, 255, 255)
    img[20:30, 20:30] = (0, 0, 0)
    assert np.array_equal(driver.denoise(img), oracle_ffi.denoise(img))


def test_ragged_sizes_and_threads():
    """Width/height not multiples of the 8x4 job tile or the 32x32 chunk; several host threads
    enter render_thread_proc with one context (driver.c:801-803)."""
    loaded = load("fov_test.obj")
    try:
        for (w, h) in [(1, 1), (13, 7), (100, 37)]:
            got = gpu_render(loaded, w, h, 3, n_threads=4)
            ref = oracle_ffi.render(loaded, w, h, 3, n_threads=3)
            assert np.array_equal(got["accum"], ref["accum"])
            assert np.array_equal(got["pixels"], ref["pixels"])
    finally:
        loaded.close()


def test_sample_slices_accumulate_in_order():
    """Slicing the sample range over several launches keeps the f32 sum sequential, hence identical."""
    loaded = load("spheres.glb")
    try:
        a = gpu_render(loaded, 96, 96, 24, slice_samples=24)
        b = gpu_render(loaded, 96, 96, 24, slice_samples=5)
        assert np.array_equal(a["accum"], b["accum"])
        ref = oracle_ffi.render(loaded, 96, 96, 24, n_threads=8)
        assert np.array_equal(a["accum"], ref["accum"])
    finally:
        loaded.close()


def test_sample_range_split_matches_sum():
    """The multi-GPU split: ranks render disjoint sample ranges; the sum of the partial accumulators
    equals the full render up to f32 addition order."""
    loaded = load("spheres.glb")
    try:
        w = h = 96
        full = gpu_render(loaded, w, h, 16)["accum"]
        lo = gpu_render(loaded, w, h, 16, sample_begin=0, sample_end=8)["accum"]
        hi = gpu_render(loaded, w, h, 16, sample_begin=8, sample_end=16)["accum"]
        ref_hi = oracle_ffi.render(loaded, w, h, 16, n_threads=8, sample_begin=8, sample_end=16)["accum"]
        assert np.array_equal(hi, ref_hi)
        np.testing.assert_allclose(lo + hi, full, rtol=1e-5, atol=1e-6)
    finally:
        loaded.close()


def test_max_bounces_and_seed():
    loaded = load("spheres.glb")
    try:
        for bounces, seed in [(1, 0), (2, 7), (8, 12345)]:
            got = gpu_render(loaded, 80, 60, 4, bounces=bounces, user_seed=seed)
            ref = oracle_ffi.render(loaded, 80, 60, 4, max_bounces=bounces, n_threads=8, user_seed=seed)
            assert np.array_equal(got["accum"], ref["accum"])
    finally:
        loaded.close()


def test_converged_image_rmse_with_independent_seeds():
    """North star: converged images within a stated RMSE.  Stated here (SURVEY §8d): at 1024 spp with
    INDEPENDENT seeds on the two sides, sRGB u8/255 RMSE <= 0.01 and mean luminance within 0.5 %."""
    loaded = load("spheres.glb")
    try:
        w, h, spp = 160, 90, 1024
        got = gpu_render(loaded, w, h, spp, user_seed=1)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=8, user_seed=2)
        a, b = got["pixels"].astype(np.float64) / 255.0, ref["pixels"].astype(np.float64) / 255.0
        rmse = float(np.sqrt(np.mean((a - b) ** 2)))
        assert rmse <= 0.01, f"converged-image RMSE {rmse}"
        lum = np.array([0.2126, 0.7152, 0.0722])
        ratio = float((got["accum"].astype(np.float64) @ lum).mean() / (ref["accum"].astype(np.float64) @ lum).mean())
        assert abs(ratio - 1.0) <= 0.005, f"mean luminance ratio {ratio}"
    finally:
        loaded.close()


def test_wavefront_chunking_is_invisible(monkeypatch):
    """The path queues hold a bounded number of paths (RT_GPU_CHUNK_PATHS); however one render call is
    cut into chunks (1, 3 or all 7 samples per chunk here) the f32 accumulator, hit ids and counters
    are identical — and equal to the oracle's."""
    loaded = load("helmet.glb")
    try:
        w, h, spp = 120, 68, 7
        per_sample = ((w + 7) // 8) * ((h + 3) // 4) * 32
        base = gpu_render(loaded, w, h, spp, slice_samples=spp)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=8, want_hit_ids=True)
        assert np.array_equal(base["accum"], ref["accum"])
        for per_chunk in (1, 3):
            monkeypatch.setenv("RT_GPU_CHUNK_PATHS", str(per_sample * per_chunk))
            other = gpu_render(loaded, w, h, spp, slice_samples=spp)
            assert gpu_lib().rt_gpu_last_launches() >= 10 * -(-spp // per_chunk)      # >= 10 kernels per chunk (trace, miss, shade per early bounce, one tail kernel, accumulate)
            assert np.array_equal(base["accum"], other["accum"])
            assert np.array_equal(base["hit_ids"], other["hit_ids"])
            assert base["counters"] == other["counters"]
    finally:
        loaded.close()


def test_full_size_properties_helmet_1080p():
    """BASELINE config 3 at its full resolution (the oracle is too slow there): size-independent properties.
    (i) queue order is decided by atomics, the result is not: two runs are bit-identical;
    (ii) every path ends exactly once: samples == W*H*spp == escaped + terminated;
    (iii) rendering the two halves of the sample range and adding them equals the full render up to f32
         addition order (the multi-GPU split), and splitting one render call into chunks changes nothing."""
    loaded = load("helmet.glb")
    try:
        w, h, spp = 1920, 1080, 16
        a = gpu_render(loaded, w, h, spp)
        b = gpu_render(loaded, w, h, spp)
        assert np.array_equal(a["accum"], b["accum"]) and np.array_equal(a["hit_ids"], b["hit_ids"])
        c = a["counters"]
        assert c["samples"] == w * h * spp and c["rays"] == c["samples"] + c["shades"] + c["passthrough"] - (c["samples"] - c["misses"])
        lo = gpu_render(loaded, w, h, spp, sample_begin=0, sample_end=8)["accum"]
        hi = gpu_render(loaded, w, h, spp, sample_begin=8, sample_end=16)["accum"]
        np.testing.assert_allclose(lo + hi, a["accum"], rtol=2e-5, atol=1e-6)
        chunked = gpu_render(loaded, w, h, spp, slice_samples=5)
        assert np.array_equal(chunked["accum"], a["accum"]) and chunked["counters"] == c
        assert not np.isnan(a["accum"]).any() and a["accum"].min() >= 0
    finally:
        loaded.close()


def test_unregistered_shader_is_an_error():
    loaded = driver.load_scene(os.path.join(MODELS, "quad.obj"), shader_proc=0xDEAD0, background_proc=oracle_ffi.background_proc())
    try:
        import ctypes
        gpu_lib().rt_gpu_register_background(oracle_ffi.background_proc())
        rc = gpu_lib().rt_gpu_scene_upload(ctypes.byref(loaded.scene))
        assert rc != 0
        assert b"not registered" in gpu_lib().rt_gpu_last_error()
    finally:
        loaded.close()


def test_gpu_radiance_equals_reference_golden_vectors():
    """The sm_100a path against vectors produced by the reference's OWN cast_ray (tests/golden/,
    generated by tools/make_golden.py from oracle/_ref/libref.so) — no oracle in between."""
    import ctypes
    import torch
    from helpers import golden, load as load_case
    arrays, meta = golden()
    gpu = gpu_lib()
    for case, cfg in meta["radiance_cases"].items():
        loaded = load_case(cfg["model"], camera=cfg["camera"], **cfg["override"])
        try:
            driver.register_callbacks(loaded)
            w, h, spp = cfg["width"], cfg["height"], cfg["spp"]
            accum = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
            per_sample = torch.zeros(h * w * spp * 3, dtype=torch.float32, device="cuda")
            gpu_check(gpu.rt_gpu_render_accum_device(ctypes.byref(loaded.scene), w, h, 0, spp, cfg["bounces"], 0, 0,
                                                     accum.data_ptr(), per_sample.data_ptr(), None, None, None))
            torch.cuda.synchronize()
            got = per_sample.cpu().numpy().reshape(h, w, spp, 3)
            assert np.array_equal(got, arrays["radiance/" + case]), case
        finally:
            loaded.close()


def test_gpu_denoiser_equals_reference_golden_vector():
    from helpers import golden
    arrays, _ = golden()
    assert np.array_equal(driver.denoise(arrays["denoise_in"]), arrays["denoise_out"])


def test_device_level_resolve_and_denoise_with_stride():
    """rt_gpu_resolve_device / rt_gpu_denoise_device on caller-owned device memory, RGBA with a padded stride."""
    import torch
    gpu = gpu_lib()
    rng = np.random.default_rng(4)
    w, h, stride, comps, spp = 37, 21, 40, 4, 5
    accum = (rng.uniform(0, 2, (h, w, 3)) ** 2 * spp).astype(np.float32)
    d_accum = torch.from_numpy(accum).cuda()
    d_px = torch.zeros(h * stride * comps, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros_like(d_px)
    gpu_check(gpu.rt_gpu_resolve_device(d_accum.data_ptr(), w, h, spp, d_px.data_ptr(), stride, comps, None))
    gpu_check(gpu.rt_gpu_denoise_device(d_px.data_ptr(), d_out.data_ptr(), w, h, stride, stride, comps, None))
    torch.cuda.synchronize()
    px = d_px.cpu().numpy().reshape(h, stride, comps)[:, :w, :3]
    want = oracle_ffi.resolve(accum, spp)
    assert np.array_equal(px, want)
    out = d_out.cpu().numpy().reshape(h, stride, comps)[:, :w, :3]
    assert np.array_equal(out, oracle_ffi.denoise(np.ascontiguousarray(want)))
