"""Refit of a resident scene on the GPU (rt_gpu_scene_refit*, csrc/rt_refit.cu) against the CPU restatement
(tests/csrc/refit_oracle.c) and the oracles of every entry point: node bytes and host write-back byte for byte; renders
(accumulator, hit ids, counters), queries, AOVs and a lightmap bake on the refit scene equal to the oracles on the refit
host scene, for an identity refit, rigid motions and a deformation; sky tiles that follow the moved root box; chained
refits; padding inputs; stream ordering; refusals; several devices."""
import ctypes as C
import os

import numpy as np
import pytest

import aov_ffi as A
import oracle_ffi
import query_ffi as Q
import refit_ffi as R
from helpers import load, scene_buffers, upload
from helpers import gpu_session  # noqa: F401
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu
THREADS = os.cpu_count() or 8


def host_nodes(loaded):
    return C.string_at(loaded.scene.bvh.nodes.data, loaded.scene.bvh.nodes.len * 192)


def counters_ex():
    raw = (C.c_uint64 * 16)()
    gpu_check(gpu_lib().rt_gpu_read_counters_ex(raw))
    return [int(v) for v in raw]


def gpu_frame(loaded, w, h, spp, bounces=8):
    driver.set_options(keep_hit_ids=True)
    try:
        pixels = driver.render(loaded, w, h, spp, bounces)
        return dict(pixels=pixels, accum=driver.read_accum(w, h), hit_ids=driver.read_hit_ids(w, h),
                    counters=driver.read_counters(), ex=counters_ex())
    finally:
        driver.set_options()


def assert_same_frame(got, want):
    assert np.array_equal(got["hit_ids"], want["hit_ids"])
    assert np.array_equal(A.bits(got["accum"]), A.bits(want["accum"]))
    assert got["counters"] == want["counters"]
    if "ex" in want:
        assert got["ex"] == want["ex"]


def check_against_oracles(loaded, w=96, h=64, spp=4, queries=True, aov=True):
    """Render, queries and AOVs of the resident (refit) scene equal the oracles run on its host Scene."""
    got = gpu_frame(loaded, w, h, spp)
    ref = oracle_ffi.render(loaded, w, h, spp, 8, n_threads=THREADS, want_hit_ids=True)
    assert_same_frame(got, ref)
    assert np.array_equal(got["pixels"], ref["pixels"])
    if queries:
        rays, _ = Q.mixed_rays(loaded, seed=5, n_each=512, grid=(32, 24))
        want = Q.oracle_query(loaded, rays, surface=True)
        hit = driver.closest_hit(loaded, rays[:, :3], rays[:, 3:], surface=True)
        assert np.array_equal(hit["slot"], want["slot"])
        assert np.array_equal(Q.bits(hit["t"]), Q.bits(want["t"]))
        assert np.array_equal(driver.occluded(loaded, rays[:, :3], rays[:, 3:]),
                              Q.oracle_query(loaded, rays, any_hit=True)["occluded"])
    if aov:
        want = A.oracle_aov(loaded, 48, 32, 0, 2)
        dev = A.device_aov(loaded, 48, 32, 0, 2)
        assert np.array_equal(A.bits(dev["records"]), A.bits(want["records"]))
        assert dev["counters"] == want["counters"]
    return got


def positions_tensor(pos):
    import torch
    return torch.from_numpy(np.ascontiguousarray(pos, dtype=np.float32)).cuda()


def test_identity_refit_host_and_device_forms():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        nodes, soa, aos = scene_buffers(loaded.scene)
        before = gpu_frame(loaded, 96, 64, 4)
        driver.refit(loaded)
        assert scene_buffers(loaded.scene) == (nodes, soa, aos)
        assert driver.read_nodes(loaded) == nodes
        assert_same_frame(gpu_frame(loaded, 96, 64, 4), before)
        driver.refit_device(loaded, positions_tensor(driver.scene_positions(loaded)),
                            positions_tensor(driver.scene_normals(loaded)))
        assert driver.read_nodes(loaded) == nodes
        assert_same_frame(gpu_frame(loaded, 96, 64, 4), before)
    finally:
        loaded.close()


MOTIONS = {"helmet.glb": ((0.35, -0.2), (0.05, -0.03, 0.02)), "spheres.glb": ((0.6, 0.3), (0.2, 0.1, -0.1)),
           "tower.obj": ((0.15, 0.05), (0.5, -0.3, 0.4))}


@pytest.mark.parametrize("name", sorted(MOTIONS))
def test_rigid_motion(name):
    (ay, ax), shift = MOTIONS[name]
    loaded, twin = load(name), load(name)
    try:
        upload(loaded)
        pos, nrm = R.rigid(driver.scene_positions(loaded), driver.scene_normals(loaded), R.rotation(ay, ax), shift)
        driver.refit(loaded, pos, nrm)
        R.oracle_refit(twin, pos, nrm)
        assert scene_buffers(loaded.scene) == scene_buffers(twin.scene)
        assert driver.read_nodes(loaded) == host_nodes(twin)
        check_against_oracles(loaded)
    finally:
        loaded.close()
        twin.close()


@pytest.mark.parametrize("name", ["helmet.glb", "spheres.glb", "tower.obj"])
def test_deformation(name):
    loaded, twin = load(name), load(name)
    try:
        upload(loaded)
        pos = R.deform(driver.scene_positions(loaded))
        driver.refit_device(loaded, positions_tensor(pos))
        R.oracle_refit(twin, pos)
        assert driver.read_nodes(loaded) == host_nodes(twin)
        driver.refit(loaded, pos)          # the device form left the host buffers alone; the host form with the same
                                           # positions changes nothing on the device and brings the host scene along
        assert driver.read_nodes(loaded) == host_nodes(twin)
        assert scene_buffers(loaded.scene) == scene_buffers(twin.scene)
        check_against_oracles(loaded)
        if name == "spheres.glb":
            got = driver.lightmap_bake(loaded, 96, 80, 3, want_values=True)
            ref = oracle_ffi.lightmap_bake(loaded, 96, 80, 3)
            assert (ref["owner"] >= 0).sum() > 300
            assert np.array_equal(got["owner"], ref["owner"])
            assert np.array_equal(A.bits(got["values"]), A.bits(ref["values"]))
    finally:
        loaded.close()
        twin.close()


def test_sky_tiles_follow_the_refit():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        before = gpu_frame(loaded, 96, 64, 4)
        pos, _ = R.rigid(driver.scene_positions(loaded), None, np.eye(3), (0.9, 0.0, 0.0))
        driver.refit(loaded, pos)
        got = check_against_oracles(loaded, queries=False, aov=False)
        newly_hit = (before["hit_ids"] < 0) & (got["hit_ids"] >= 0)
        assert newly_hit.sum() > 100, "the move must put geometry where there was sky"
    finally:
        loaded.close()


def test_chained_refits_equal_the_last_one():
    a, b = load("helmet.glb"), load("helmet.glb")
    try:
        upload(a)
        upload(b)
        p0 = driver.scene_positions(a)
        pa, _ = R.rigid(p0, None, R.rotation(0.4, 0.1), (0.1, 0.0, 0.0))
        pb = R.deform(p0, 0.03, 5.0)
        driver.refit_device(a, positions_tensor(pa))
        driver.refit_device(a, positions_tensor(pb))
        driver.refit_device(b, positions_tensor(pb))
        assert driver.read_nodes(a) == driver.read_nodes(b)
        assert_same_frame(gpu_frame(a, 96, 64, 4), gpu_frame(b, 96, 64, 4))
    finally:
        a.close()
        b.close()


def test_padding_inputs_are_ignored():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        pos = R.deform(driver.scene_positions(loaded))
        driver.refit_device(loaded, positions_tensor(pos))
        clean = driver.read_nodes(loaded)
        n = loaded.scene.triangles.len
        padding = np.ones(n, dtype=bool)
        padding[loaded.slot_of] = False
        assert padding.sum() > 1000
        garbage = pos.copy()
        garbage[:, :, padding] = np.random.default_rng(3).uniform(-1e6, 1e6, size=(3, 3, int(padding.sum())))
        driver.refit_device(loaded, positions_tensor(garbage), positions_tensor(np.full((n, 3, 3), 5.0)))
        assert driver.read_nodes(loaded) == clean
    finally:
        loaded.close()


def test_ordering_without_host_synchronisation():
    import torch
    loaded, twin = load("spheres.glb"), load("spheres.glb")
    try:
        upload(loaded)
        w, h, spp = 64, 48, 3
        pos = R.deform(driver.scene_positions(loaded), 0.08, 2.0)
        R.oracle_refit(twin, pos)
        rays, _ = Q.mixed_rays(twin, seed=2, n_each=256, grid=(16, 12))
        d_pos, d_rays = positions_tensor(pos), torch.from_numpy(np.ascontiguousarray(rays)).cuda()
        s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        accum = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        hits = torch.zeros((len(rays), 4), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        driver.refit_device(loaded, d_pos, stream=s1)
        driver.render_masked(loaded, accum, 0, spp, stream=s2)
        gpu_check(gpu_lib().rt_gpu_closest_hit_device(C.byref(loaded.scene), d_rays.data_ptr(), None, len(rays),
                                                      hits.data_ptr(), None, None, s3.cuda_stream))
        torch.cuda.synchronize()
        ref = oracle_ffi.render(twin, w, h, spp, 8, n_threads=THREADS)
        assert np.array_equal(A.bits(accum.cpu().numpy()), A.bits(ref["accum"]))
        want = Q.oracle_query(twin, rays)
        got = hits.cpu().numpy()
        assert np.array_equal(got[:, 3].view(np.int32), want["slot"])
        assert np.array_equal(Q.bits(got[:, 0].copy()), Q.bits(want["t"]))
    finally:
        loaded.close()
        twin.close()


def test_refusals_leave_the_scene_unchanged():
    import torch
    gpu = gpu_lib()
    loaded, other = load("spheres.glb"), load("quad.obj")
    try:
        upload(loaded)
        nodes = driver.read_nodes(loaded)
        before = gpu_frame(loaded, 64, 48, 3)
        pos = driver.scene_positions(loaded)
        # not resident
        driver.register_callbacks(other)
        assert gpu.rt_gpu_scene_refit_device(C.byref(other.scene), positions_tensor(driver.scene_positions(other)).data_ptr(),
                                             None, None) != 0
        assert b"not resident" in gpu.rt_gpu_last_error()
        assert gpu.rt_gpu_scene_refit(C.byref(other.scene), 0) != 0
        # NULL positions
        assert gpu.rt_gpu_scene_refit_device(C.byref(loaded.scene), None, None, None) != 0
        assert b"null positions" in gpu.rt_gpu_last_error()
        # non-finite coordinates in an occupied slot, device and host forms
        slot = int(loaded.slot_of[len(loaded.slot_of) // 2])
        for bad in (np.nan, np.inf, -np.inf):
            p = R.deform(pos)
            p[1, 2, slot] = bad
            with pytest.raises(RuntimeError, match="non-finite"):
                driver.refit_device(loaded, positions_tensor(p))
            assert driver.read_nodes(loaded) == nodes
            with pytest.raises(RuntimeError, match="non-finite"):
                driver.refit(loaded, p)
            assert driver.read_nodes(loaded) == nodes
        torch.cuda.synchronize()
        assert_same_frame(gpu_frame(loaded, 64, 48, 3), before)
    finally:
        loaded.close()
        other.close()


def visible_gpus():
    return int(gpu_lib().rt_gpu_visible_devices())


@pytest.mark.skipif("visible_gpus() < 2")
def test_two_devices_in_one_process():
    loaded, twin = load("helmet.glb"), load("helmet.glb")
    try:
        driver.init_devices(2)
        upload(loaded)
        pos, nrm = R.rigid(driver.scene_positions(loaded), driver.scene_normals(loaded), R.rotation(0.3, 0.1), (0.1, 0, 0))
        driver.refit(loaded, pos, nrm)
        R.oracle_refit(twin, pos, nrm)
        assert driver.read_nodes(loaded) == host_nodes(twin)
        for split in (1, 2):            # samples, then 32x32 chunks: both devices trace the refit geometry
            driver.set_options(keep_hit_ids=True, split_mode=split)
            driver.render(loaded, 96, 64, 16, 8)
            got = dict(accum=driver.read_accum(96, 64), hit_ids=driver.read_hit_ids(96, 64))
            ref = oracle_ffi.render(twin, 96, 64, 16, 8, n_threads=THREADS, want_hit_ids=True)
            assert np.array_equal(got["hit_ids"], ref["hit_ids"])
            assert np.allclose(got["accum"], ref["accum"], rtol=1e-5, atol=1e-5)
    finally:
        driver.set_options()
        loaded.close()
        twin.close()
        gpu_check(gpu_lib().rt_gpu_init(0))
