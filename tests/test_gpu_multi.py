"""The multi-GPU machinery of the library (csrc/rt_multi.cu, rt_cabi.cu) on hardware.

One-device tests exercise every piece that does not need a second GPU: the chunk split and the sample split as
`world` shards rendered one after the other, the fused reduce+resolve kernel over the shards' accumulators, empty
shares, the per-call status.  With >= 2 visible GPUs the same frame is rendered by rt_gpu_init_devices(2) through
render_thread_proc (split, peer-mapped reduce+resolve, denoise) and compared with the single-GPU frame and the
oracle; the C host binary is run with --gpus and its PNG compared byte for byte."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_ffi
from helpers import MODELS, ROOT, load
from raytracing_c_b200 import driver, gpu_lib, sharding
from raytracing_c_b200._ffi import SPLIT_CHUNKS, SPLIT_SAMPLES, REDUCE_NCCL, gpu_check

pytestmark = pytest.mark.gpu
RT_DRIVER = os.path.join(ROOT, "raytracing_c_b200", "host", "rt_driver")


@pytest.fixture(autouse=True)
def _one_gpu():
    gpu_check(gpu_lib().rt_gpu_init(0))
    driver.set_options()
    yield
    driver.set_options()
    gpu_check(gpu_lib().rt_gpu_init(0))


def visible_gpus():
    return int(gpu_lib().rt_gpu_visible_devices())


def render_full(loaded, w, h, spp, **opt):
    driver.set_options(keep_hit_ids=True, **opt)
    px = driver.render(loaded, w, h, spp, 8)
    return dict(pixels=px, accum=driver.read_accum(w, h), hit_ids=driver.read_hit_ids(w, h), counters=driver.read_counters())


def test_chunk_split_at_1080p_with_job_tiles_outside_the_image():
    """1080 rows = 33 chunk rows + 24 pixel rows: the last chunk row holds job tiles that lie entirely outside the
    image; a warp that draws such a tile must go on with the rest of its reserved range."""
    loaded = load("helmet.glb")
    try:
        w, h, spp = 1920, 1080, 8
        full = render_full(loaded, w, h, spp)
        total = np.zeros_like(full["accum"])
        for r in range(2):
            total += render_full(loaded, w, h, spp, pixel_rank=r, pixel_world=2)["accum"]
        assert np.array_equal(total, full["accum"])
    finally:
        loaded.close()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_chunk_split_shards_sum_bit_identically(world):
    """The chunk split gives every pixel to exactly one shard, all its samples in order: the sum over shards
    adds zeros and equals the unsplit frame BIT FOR BIT; work counters add up."""
    loaded = load("helmet.glb")
    try:
        w, h, spp = 200, 150, 6                 # 7 x 5 chunks, ragged right and bottom edges
        full = render_full(loaded, w, h, spp)
        total = np.zeros_like(full["accum"])
        ids = np.full((h, w), -(2 ** 31), dtype=np.int64)
        counters = {}
        for r in range(world):
            part = render_full(loaded, w, h, spp, pixel_rank=r, pixel_world=world)
            owned = sharding.owned_chunks(r, world, w, h)
            assert (part["accum"].reshape(-1, 3).any(axis=1)).sum() <= owned * 32 * 32
            total += part["accum"]
            ids = np.maximum(ids, part["hit_ids"])
            for k, v in part["counters"].items():
                counters[k] = counters.get(k, 0) + v
        assert np.array_equal(total, full["accum"])
        assert np.array_equal(ids, full["hit_ids"])
        assert counters == full["counters"]
    finally:
        loaded.close()


def test_library_shard_policy_and_empty_shares():
    """world > number of 8-sample batches: AUTO deals chunks, and a forced sample split hands empty ranges to
    the surplus ranks — whose accumulators must be zero, not stale (ADVICE r1)."""
    gpu = gpu_lib()
    assert sharding.split_mode(16, 8) == SPLIT_CHUNKS and sharding.split_mode(1024, 8) == SPLIT_SAMPLES
    assert sharding.split_mode(1, 4) == SPLIT_CHUNKS and sharding.split_mode(24, 2) == SPLIT_CHUNKS
    spans = [sharding.sample_range(r, 8, 16) for r in range(8)]
    assert sum(b - a for a, b in spans) == 16 and sum(1 for a, b in spans if a == b) == 6
    import torch
    loaded = load("spheres.glb")
    try:
        driver.register_callbacks(loaded)
        w, h, spp = 96, 64, 16
        full = render_full(loaded, w, h, spp)["accum"]
        scene = C.byref(loaded.scene)
        for mode in (SPLIT_SAMPLES, SPLIT_CHUNKS):
            total = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
            for r in range(8):
                part = torch.full((h * w * 3,), 7.0, dtype=torch.float32, device="cuda")     # stale content must vanish
                used = C.c_int32()
                gpu_check(gpu.rt_gpu_render_shard_device(scene, w, h, spp, 8, 0, r, 8, mode, C.byref(used),
                                                         part.data_ptr(), None, None))
                assert used.value == mode
                torch.cuda.synchronize()
                if mode == SPLIT_SAMPLES and spans[r][0] == spans[r][1]:
                    assert float(part.abs().max()) == 0.0
                total += part
            got = total.cpu().numpy().reshape(h, w, 3)
            if mode == SPLIT_CHUNKS:
                assert np.array_equal(got, full)
            else:
                np.testing.assert_allclose(got, full, rtol=2e-6, atol=1e-6)
        # the same through the entry point's options: an explicitly empty range
        empty = render_full(loaded, w, h, spp, sample_begin=8, sample_end=8, sample_range_set=True)
        assert not empty["accum"].any()
    finally:
        loaded.close()


def test_fused_reduce_resolve_matches_sum_then_resolve():
    """rt_reduce_resolve_kernel: parts summed in rank order, then the film — equal to numpy's sequential f32 sum
    followed by the oracle's resolve, for 1..5 parts, ragged pixel counts, RGBA with a padded stride."""
    import torch
    gpu = gpu_lib()
    rng = np.random.default_rng(11)
    for (w, h, n_parts, comps, stride) in [(37, 21, 1, 3, 37), (64, 33, 2, 3, 64), (125, 7, 5, 4, 130), (3, 1, 3, 3, 3)]:
        spp = 9
        parts = [(rng.uniform(0, 1.5, (h, w, 3)) ** 2 * spp / n_parts).astype(np.float32) for _ in range(n_parts)]
        want = parts[0].copy()
        for p in parts[1:]:
            want = want + p
        d_parts = [torch.from_numpy(p).cuda() for p in parts]
        ptrs = (C.c_void_p * n_parts)(*[p.data_ptr() for p in d_parts])
        d_sum = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
        d_px = torch.zeros(h * stride * comps, dtype=torch.uint8, device="cuda")
        gpu_check(gpu.rt_gpu_reduce_resolve_device(ptrs, n_parts, d_sum.data_ptr(), w, h, spp, d_px.data_ptr(), stride, comps, None))
        torch.cuda.synchronize()
        assert np.array_equal(d_sum.cpu().numpy().reshape(h, w, 3), want)
        px = d_px.cpu().numpy().reshape(h, stride, comps)[:, :w, :3]
        assert np.array_equal(px, oracle_ffi.resolve(want, spp))


def test_failed_render_is_reported_not_swallowed():
    """raytracer.h's entry points return void; a failure must surface through rt_gpu_last_status (ADVICE r1)."""
    loaded = load("quad.obj")
    try:
        bad = np.zeros((8, 8, 1), dtype=np.uint8)            # 1 component: the film needs >= 3
        with pytest.raises(RuntimeError, match="components"):
            driver.render(loaded, 8, 8, 1, 8, out=bad)
        assert gpu_lib().rt_gpu_last_status() != 0
        ok = driver.render(loaded, 8, 8, 1, 8)               # and the next call clears it
        assert gpu_lib().rt_gpu_last_status() == 0 and ok.shape == (8, 8, 3)
        with pytest.raises(RuntimeError, match="samples"):
            driver.render(loaded, 8, 8, 0, 8)
    finally:
        loaded.close()


def test_pinned_host_buffers_and_rebuilt_scene_are_detected():
    """Scene buffers in pinned memory are DMA-read in place (no staging) and give the same frame; a Scene
    rebuilt at the same address (new buffers) is re-uploaded without an explicit call (ADVICE r1)."""
    from raytracing_c_b200._ffi import host_lib
    w, h, spp = 120, 68, 4
    plain = load("helmet.glb")
    try:
        a = render_full(plain, w, h, spp)["accum"]
    finally:
        plain.close()
    driver.use_pinned_host_buffers(True)
    try:
        pinned = load("helmet.glb")
    finally:
        driver.use_pinned_host_buffers(False)
    try:
        b = render_full(pinned, w, h, spp)["accum"]
        assert np.array_equal(a, b)
        # rebuild the BVH of the same Scene struct in place: new node/triangle buffers, same Scene pointer
        host = host_lib()
        host.scene_destroy(C.byref(pinned.scene))
        host.scene_init(C.byref(pinned.scene), pinned.model.triangles)
        c = render_full(pinned, w, h, spp)["accum"]
        assert np.array_equal(a, c)
    finally:
        pinned.close()


def test_two_renders_on_different_streams_do_not_corrupt_each_other():
    """Every render of a device shares its workspace and the scene's camera-relative copies: calls on different
    streams must be serialised by the library (ADVICE r1), whatever the caller's streams do."""
    import torch
    gpu = gpu_lib()
    loaded = load("spheres.glb")
    try:
        driver.register_callbacks(loaded)
        w, h, spp = 256, 256, 8
        want = render_full(loaded, w, h, spp)["accum"]
        scene = C.byref(loaded.scene)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        a = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
        b = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        for _ in range(3):
            gpu_check(gpu.rt_gpu_render_accum_device(scene, w, h, 0, spp, 8, 0, 0, a.data_ptr(), None, None, None, C.c_void_p(s1.cuda_stream)))
            gpu_check(gpu.rt_gpu_render_accum_device(scene, w, h, 0, spp, 8, 0, 0, b.data_ptr(), None, None, None, C.c_void_p(s2.cuda_stream)))
        torch.cuda.synchronize()
        assert np.array_equal(a.cpu().numpy().reshape(h, w, 3), want)
        assert np.array_equal(b.cpu().numpy().reshape(h, w, 3), want)
    finally:
        loaded.close()


def run_driver(args, cwd):
    out = subprocess.run([RT_DRIVER] + args, cwd=cwd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout


def test_c_host_binary_matches_the_library_frame(tmp_path):
    """The C host (host/driver.c, the reference's flags) linked against libraytracer_gpu.so: its PNG equals the
    PNG of driver.render's pixels byte for byte, --dump-accum / --dump-hit-ids equal the parity hooks, -D denoises."""
    w, h, spp = 160, 96, 8
    model = os.path.join(MODELS, "helmet.glb")
    png, acc, ids = str(tmp_path / "c.png"), str(tmp_path / "c.accum"), str(tmp_path / "c.ids")
    text = run_driver(["-W", str(w), "-H", str(h), "-S", str(spp), "-B", "8", "-T", "3", "-V", model, "-O", png,
                       "--dump-accum", acc, "--dump-hit-ids", ids], tmp_path)
    assert "samples/second" in text and "BVH-Nodes: 585" in text
    loaded = load("helmet.glb")
    try:
        mine = render_full(loaded, w, h, spp)
        ref_png = str(tmp_path / "py.png")
        driver.save_image(ref_png, mine["pixels"])
        assert open(png, "rb").read() == open(ref_png, "rb").read()
        assert np.array_equal(np.fromfile(acc, dtype=np.float32).reshape(h, w, 3), mine["accum"])
        assert np.array_equal(np.fromfile(ids, dtype=np.int32).reshape(h, w), mine["hit_ids"])
        den_png = str(tmp_path / "c_den.png")
        run_driver(["-W", str(w), "-H", str(h), "-S", str(spp), "-D", model, "-O", den_png], tmp_path)
        ref_den = str(tmp_path / "py_den.png")
        driver.save_image(ref_den, driver.denoise(mine["pixels"]))
        assert open(den_png, "rb").read() == open(ref_den, "rb").read()
    finally:
        loaded.close()
    # a failing render must exit non-zero
    bad = subprocess.run([RT_DRIVER, "-S", "0", model, "-O", str(tmp_path / "x.png")], cwd=tmp_path, capture_output=True, text=True)
    assert bad.returncode != 0 and "samples" in bad.stderr


@pytest.mark.skipif("visible_gpus() < 2")
@pytest.mark.parametrize("split,reduce", [(SPLIT_CHUNKS, 0), (SPLIT_SAMPLES, 0), (SPLIT_SAMPLES, REDUCE_NCCL)])
def test_multi_device_frame_equals_single_device_and_oracle(split, reduce):
    """G2: one process, N devices.  The frame render_thread_proc returns with N GPUs (split, peer-mapped fused
    reduce+resolve or NCCL reduce, then denoise on device 0) against the single-GPU frame and the oracle."""
    n = min(visible_gpus(), 8)
    loaded = load("helmet.glb")
    try:
        w, h, spp = 320, 180, 16 * n
        one = render_full(loaded, w, h, spp)
        ref = oracle_ffi.render(loaded, w, h, spp, n_threads=len(os.sched_getaffinity(0)), want_hit_ids=True)
        assert np.array_equal(one["accum"], ref["accum"])
        driver.init_devices(n)
        many = render_full(loaded, w, h, spp, split_mode=split, reduce_mode=reduce)
        assert gpu_lib().rt_gpu_device_count() == n
        assert many["counters"] == one["counters"]
        assert np.array_equal(many["hit_ids"], ref["hit_ids"])
        if split == SPLIT_CHUNKS:
            assert np.array_equal(many["accum"], ref["accum"])
            assert np.array_equal(many["pixels"], ref["pixels"])
        else:
            rel = np.abs(many["accum"] - ref["accum"]) / np.maximum(np.abs(ref["accum"]), 1e-6)
            assert rel.max() <= 1e-3 and rel.max() < 1e-5
            assert np.abs(many["pixels"].astype(int) - ref["pixels"].astype(int)).max() <= 1
        den = driver.denoise(many["pixels"])
        assert np.array_equal(den, oracle_ffi.denoise(many["pixels"]))
    finally:
        loaded.close()


@pytest.mark.skipif("visible_gpus() < 2")
def test_c_host_binary_with_gpus_flag(tmp_path):
    n = min(visible_gpus(), 8)
    w, h, spp = 256, 144, 8 * n
    model = os.path.join(MODELS, "helmet.glb")
    one, many = str(tmp_path / "one.png"), str(tmp_path / "many.png")
    run_driver(["-W", str(w), "-H", str(h), "-S", str(spp), model, "-O", one], tmp_path)
    text = run_driver(["-W", str(w), "-H", str(h), "-S", str(spp), "-V", "--gpus", str(n), "--split", "chunks", model, "-O", many], tmp_path)
    assert f"GPUs: {n}" in text
    assert open(one, "rb").read() == open(many, "rb").read()
