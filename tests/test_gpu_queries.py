"""Ray queries on the GPU (rt_gpu_closest_hit* / rt_gpu_occluded*, csrc/rt_query.cu) against their CPU reference
(tests/csrc/query_oracle.c): t, u, v, slot, the surface record and the four work counters bit-exact, for every ray family and
t_max edge, on the six shipped models; occlusion equal to the oracle's early-exit walk and to (closest slot >= 0).
"""
import ctypes as C
import os

import numpy as np
import pytest

import query_ffi as Q
from helpers import MODELS, load
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu

MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    gpu_check(gpu_lib().rt_gpu_init(0))
    yield
    driver.set_options()


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    yield loaded
    loaded.close()


def torch_rays(rays, t_max):
    import torch
    r = torch.from_numpy(np.ascontiguousarray(rays, dtype=np.float32)).cuda()
    t = torch.from_numpy(np.ascontiguousarray(t_max, dtype=np.float32)).cuda() if t_max is not None else None
    return r, t


def device_query(loaded, rays, t_max=None, any_hit=False, surface=False, stream=None):
    """The device-level calls on torch tensors, on `stream` (default: torch's current stream); returns numpy results and
    the four counters."""
    import torch
    r, t = rays if isinstance(rays, tuple) else torch_rays(rays, t_max)
    n = r.shape[0]
    ctr = torch.zeros(4, dtype=torch.int64, device="cuda")
    st = stream or torch.cuda.current_stream()
    gpu = gpu_lib()
    driver.register_callbacks(loaded)
    tp = t.data_ptr() if t is not None else None
    if any_hit:
        occ = torch.full((max(n, 1),), 7, dtype=torch.uint8, device="cuda")
        gpu_check(gpu.rt_gpu_occluded_device(C.byref(loaded.scene), r.data_ptr(), tp, n, occ.data_ptr(), ctr.data_ptr(),
                                             st.cuda_stream))
        st.synchronize()
        out = {"occluded": occ[:n].cpu().numpy()}
    else:
        hits = torch.full((max(n, 1), 4), 7.0, dtype=torch.float32, device="cuda")
        surf = torch.full((max(n, 1), 11), 7.0, dtype=torch.float32, device="cuda") if surface else None
        gpu_check(gpu.rt_gpu_closest_hit_device(C.byref(loaded.scene), r.data_ptr(), tp, n, hits.data_ptr(),
                                                surf.data_ptr() if surf is not None else None, ctr.data_ptr(), st.cuda_stream))
        st.synchronize()
        h = hits[:n].cpu().numpy()
        out = {"t": h[:, 0].copy(), "u": h[:, 1].copy(), "v": h[:, 2].copy(), "slot": h[:, 3].copy().view(np.int32)}
        if surf is not None:
            out["surface"] = surf[:n].cpu().numpy()
    out["counters"] = dict(zip(Q.QUERY_COUNTERS, map(int, ctr.cpu().numpy())))
    return out


def assert_closest_equal(got, want, surface=True):
    for k in ("t", "u", "v"):
        assert np.array_equal(Q.bits(got[k]), Q.bits(want[k])), f"{k} differs on {int((Q.bits(got[k]) != Q.bits(want[k])).sum())} rays"
    assert np.array_equal(got["slot"], want["slot"])
    if surface:
        for k, s in Q.SURFACE_FIELDS.items():
            assert np.array_equal(Q.bits(got["surface"][:, s]), Q.bits(want["surface"][:, s])), k
    assert got["counters"] == want["counters"]


def test_closest_hit_and_occlusion_bit_exact(scene):
    rng = np.random.default_rng(21)
    rays, closest = Q.mixed_rays(scene, seed=20, n_each=4096)
    assert np.isfinite(closest).sum() > 100
    for t_max in (None, Q.t_max_mix(closest, rng)):
        want = Q.oracle_query(scene, rays, t_max, surface=True)
        got = device_query(scene, rays, t_max, surface=True)
        assert_closest_equal(got, want)
        want_any = Q.oracle_query(scene, rays, t_max, any_hit=True)
        got_any = device_query(scene, rays, t_max, any_hit=True)
        assert np.array_equal(got_any["occluded"].astype(bool), want_any["occluded"])
        assert set(np.unique(got_any["occluded"]).tolist()) <= {0, 1}
        assert got_any["counters"] == want_any["counters"]
        assert np.array_equal(got_any["occluded"].astype(bool), got["slot"] >= 0)
        for k in ("nodes", "leaves", "accepts"):
            assert got_any["counters"][k] <= got["counters"][k]
    # every t_max edge kind of the mix, checked on its own
    kind = np.arange(len(rays)) % 8
    assert np.array_equal(got["slot"][kind == 0] >= 0, np.isfinite(closest[kind == 0]))
    assert np.array_equal(got["slot"][kind == 7] >= 0, np.isfinite(closest[kind == 7]))
    assert (got["slot"][(kind >= 1) & (kind <= 6)] == -1).all(), \
        "a fraction of the closest t, the closest t itself, EPSILON, 0, negative and NaN all miss"


def test_fast_math_option_does_not_apply_to_queries():
    loaded = load("helmet.glb")
    try:
        rays, closest = Q.mixed_rays(loaded, seed=30, n_each=4096)
        want = Q.oracle_query(loaded, rays, surface=True)
        driver.set_options(fast_math=True)
        got = device_query(loaded, rays, surface=True)
        assert_closest_equal(got, want)
    finally:
        driver.set_options()
        loaded.close()


def test_large_ragged_batch():
    """2^25 + 13 rays (ragged last warp, many waves of the persistent grid): the identity on every ray, the oracle on a
    seeded subset."""
    import torch
    loaded = load("helmet.glb")
    try:
        n = (1 << 25) + 13
        lo, hi = Q.root_box(loaded.scene)
        g = torch.Generator(device="cuda").manual_seed(1234)
        o = torch.tensor(lo, device="cuda") + torch.rand(n, 3, device="cuda", generator=g) * torch.tensor(hi - lo, device="cuda")
        d = torch.randn(n, 3, device="cuda", generator=g)
        d = d / d.norm(dim=1, keepdim=True)
        rays = torch.cat([o, d], dim=1).contiguous()
        t_max = torch.where(torch.rand(n, device="cuda", generator=g) < 0.5, torch.full((n,), float("inf"), device="cuda"),
                            torch.rand(n, device="cuda", generator=g) * float((hi - lo).max())).contiguous()
        near = device_query(loaded, (rays, t_max))
        occ = device_query(loaded, (rays, t_max), any_hit=True)
        assert near["counters"]["rays"] == occ["counters"]["rays"] == n
        assert np.array_equal(occ["occluded"].astype(bool), near["slot"] >= 0)
        assert 0.05 < (near["slot"] >= 0).mean() < 0.95
        for k in ("nodes", "leaves", "accepts"):
            assert occ["counters"][k] <= near["counters"][k]
        idx = np.sort(np.random.default_rng(3).choice(n, size=65536, replace=False))
        idx[-1] = n - 1                                                     # the last ray of the ragged warp
        sub_r, sub_t = rays.cpu().numpy()[idx], t_max.cpu().numpy()[idx]
        want = Q.oracle_query(loaded, sub_r, sub_t)
        for k in ("t", "u", "v"):
            assert np.array_equal(Q.bits(near[k][idx]), Q.bits(want[k])), k
        assert np.array_equal(near["slot"][idx], want["slot"])
        assert np.array_equal(occ["occluded"][idx].astype(bool), want["occluded"])
    finally:
        loaded.close()


def test_empty_single_and_host_level_agree():
    loaded = load("spheres.glb")
    try:
        gpu = gpu_lib()
        assert gpu.rt_gpu_closest_hit(C.byref(loaded.scene), None, None, 0, None, None) == 0
        assert gpu.rt_gpu_occluded(C.byref(loaded.scene), None, None, 0, None) == 0
        assert gpu.rt_gpu_closest_hit_device(C.byref(loaded.scene), None, None, 0, None, None, None, None) == 0
        assert gpu.rt_gpu_occluded_device(C.byref(loaded.scene), None, None, 0, None, None, None) == 0
        rays, closest = Q.mixed_rays(loaded, seed=40, n_each=2048)
        hit = np.nonzero(np.isfinite(closest))[0][0]
        for sel in (slice(hit, hit + 1), slice(0, 1)):
            want = Q.oracle_query(loaded, rays[sel], surface=True)
            assert_closest_equal(device_query(loaded, rays[sel], surface=True), want)
        t_max = Q.t_max_mix(closest, np.random.default_rng(41))
        dev = device_query(loaded, rays, t_max, surface=True)
        host = driver.closest_hit(loaded, rays[:, :3], rays[:, 3:], t_max, surface=True)
        for k in ("t", "u", "v", "slot"):
            assert np.array_equal(Q.bits(host[k]) if k != "slot" else host[k], Q.bits(dev[k]) if k != "slot" else dev[k]), k
        for k, s in Q.SURFACE_FIELDS.items():
            assert np.array_equal(Q.bits(host[k]), Q.bits(dev["surface"][:, s])), k
        occ_host = driver.occluded(loaded, rays[:, :3], rays[:, 3:], t_max)
        assert occ_host.dtype == bool and np.array_equal(occ_host, device_query(loaded, rays, t_max, any_hit=True)["occluded"].astype(bool))
        assert np.array_equal(occ_host, host["slot"] >= 0)
        # no t_max array and a scalar one
        assert np.array_equal(driver.closest_hit(loaded, rays[:, :3], rays[:, 3:])["slot"], Q.oracle_query(loaded, rays)["slot"])
        assert np.array_equal(driver.occluded(loaded, rays[:, :3], rays[:, 3:], 0.5),
                              Q.oracle_query(loaded, rays, np.full(len(rays), 0.5, np.float32), any_hit=True)["occluded"])
        assert gpu.rt_gpu_last_launches() == 1
    finally:
        loaded.close()


def test_query_on_a_user_stream_right_after_upload():
    """A fresh scene, uploaded and queried at once on a torch stream: the query waits for the geometry only."""
    import torch
    loaded = driver.load_scene(os.path.join(MODELS, "helmet.glb"))
    try:
        rays, _ = Q.mixed_rays(loaded, seed=50, n_each=4096)
        r, _ = torch_rays(rays, None)
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        driver.register_callbacks(loaded)
        gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))
        with torch.cuda.stream(stream):
            got = device_query(loaded, (r, None), surface=True, stream=stream)
        assert_closest_equal(got, Q.oracle_query(loaded, rays, surface=True))
    finally:
        loaded.close()


def test_validation_errors_before_launch():
    import torch
    loaded = load("quad.obj")
    try:
        gpu = gpu_lib()
        r, _ = torch_rays(Q.interior_rays(loaded.scene, np.random.default_rng(1), 64), None)
        hits = torch.zeros(64 * 4 + 4, dtype=torch.float32, device="cuda")
        occ = torch.zeros(64, dtype=torch.uint8, device="cuda")
        sc = C.byref(loaded.scene)
        cases = [
            (lambda: gpu.rt_gpu_closest_hit_device(sc, r.data_ptr(), None, -1, hits.data_ptr(), None, None, None), "n_rays"),
            (lambda: gpu.rt_gpu_closest_hit_device(sc, r.data_ptr(), None, 1 << 31, hits.data_ptr(), None, None, None), "n_rays"),
            (lambda: gpu.rt_gpu_closest_hit_device(sc, r.data_ptr(), None, 64, hits.data_ptr() + 4, None, None, None), "aligned"),
            (lambda: gpu.rt_gpu_closest_hit_device(sc, None, None, 64, hits.data_ptr(), None, None, None), "rays"),
            (lambda: gpu.rt_gpu_closest_hit_device(sc, r.data_ptr(), None, 64, None, None, None, None), "output"),
            (lambda: gpu.rt_gpu_occluded_device(sc, r.data_ptr(), None, 64, None, None, None), "output"),
            (lambda: gpu.rt_gpu_occluded_device(sc, None, None, 64, occ.data_ptr(), None, None), "rays"),
            (lambda: gpu.rt_gpu_occluded(sc, None, None, 64, None), "rays"),
            (lambda: gpu.rt_gpu_closest_hit(sc, None, None, -5, None, None), "n_rays"),
            (lambda: gpu.rt_gpu_closest_hit(None, None, None, 3, None, None), "scene"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in gpu.rt_gpu_last_error().decode()
        torch.cuda.synchronize()
        # the library still answers after the refusals
        rays = r.cpu().numpy()
        assert np.array_equal(driver.closest_hit(loaded, rays[:, :3], rays[:, 3:])["slot"], Q.oracle_query(loaded, rays)["slot"])
    finally:
        loaded.close()


def test_queries_do_not_disturb_renders():
    loaded = load("helmet.glb")
    try:
        w, h, spp = 160, 90, 4
        driver.set_options(keep_hit_ids=True)
        driver.render(loaded, w, h, spp, 8)
        first = driver.read_accum(w, h).copy()
        rays, _ = Q.mixed_rays(loaded, seed=60, n_each=8192)
        driver.closest_hit(loaded, rays[:, :3], rays[:, 3:], surface=True)
        driver.occluded(loaded, rays[:, :3], rays[:, 3:])
        device_query(loaded, rays, surface=True)
        driver.render(loaded, w, h, spp, 8)
        assert np.array_equal(Q.bits(driver.read_accum(w, h)), Q.bits(first))
    finally:
        driver.set_options()
        loaded.close()
