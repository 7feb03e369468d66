"""The CPU reference of the ray queries (tests/csrc/query_oracle.c), which the GPU queries are checked against, pinned:
  - at t_max = inf they are the renderer's own walk (oracle_trace_ray);
  - the closest t equals a brute-force scan over every triangle slot (the slot too where that t is unique, i.e. where
    the walk's order cannot decide a tie);
  - the early-exit walk says occluded exactly where the closest-hit walk with the same t_max finds a hit, and counts
    no more rays, nodes, leaves or accepts;
  - where a reference checkout is available, every field equals the reference's own ray_scene_hit started at t_max.
"""
import ctypes as C

import numpy as np
import pytest

import query_ffi as Q
from helpers import MODEL_NAMES, load


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    yield loaded
    loaded.close()


def brute_force(scene, rays, t_max):
    """raytracer.c:115-159 over every slot in numpy float32 (no contraction): min t over the accepted triangles with
    0 < t < t_max, and the slots that reach it."""
    tr = scene.scene.triangles
    n = tr.len
    arr = lambda p: np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(n,)).copy()
    p0 = np.stack([arr(tr.x[0]), arr(tr.y[0]), arr(tr.z[0])], axis=1)
    p1 = np.stack([arr(tr.x[1]), arr(tr.y[1]), arr(tr.z[1])], axis=1)
    p2 = np.stack([arr(tr.x[2]), arr(tr.y[2]), arr(tr.z[2])], axis=1)
    e1, e2 = p1 - p0, p2 - p0
    dot = lambda a, b: a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]
    cross = lambda a, b: np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                                   a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)
    best_t, best_slots = [], []
    with np.errstate(all="ignore"):
        for ray, tm in zip(rays, t_max):
            o, d = ray[None, :3], np.broadcast_to(ray[None, 3:], e2.shape)
            pv = cross(d, e2)
            inv_det = np.float32(1) / dot(e1, pv)
            tv = o - p0
            qv = cross(tv, e1)
            u = inv_det * dot(tv, pv)
            v = inv_det * dot(d, qv)
            t = inv_det * dot(e2, qv)
            out = (u < -Q.EPS) | (u > 1 + Q.EPS) | (v < -Q.EPS) | (u + v > 1 + Q.EPS) | (t < Q.EPS)
            dist = np.where(out, np.float32(np.inf), t)
            ok = (dist > 0) & (dist < tm)
            if ok.any():
                m = dist[ok].min()
                best_t.append(m)
                best_slots.append(set(np.nonzero(ok & (dist == m))[0].tolist()))
            else:
                best_t.append(np.float32(np.inf))
                best_slots.append(set())
    return np.array(best_t, dtype=np.float32), best_slots


def test_query_at_inf_is_the_renderers_walk(scene):
    rays, _ = Q.mixed_rays(scene, seed=11, n_each=300, grid=(24, 16))
    got = Q.oracle_query(scene, rays)
    for i, ray in enumerate(rays):
        slot, t = Q.oracle_trace_ray(scene, ray)
        assert got["slot"][i] == slot and Q.bits(got["t"][i:i + 1]) == Q.bits(np.array([t], dtype=np.float32)), i


def test_closest_t_equals_brute_force(scene):
    rng = np.random.default_rng(5)
    rays, closest = Q.mixed_rays(scene, seed=12, n_each=120, grid=(16, 12))
    t_max = Q.t_max_mix(closest, rng)
    got = Q.oracle_query(scene, rays, t_max)
    want_t, want_slots = brute_force(scene, rays, t_max)
    assert np.array_equal(Q.bits(got["t"]), Q.bits(want_t))
    for i, slots in enumerate(want_slots):
        if len(slots) == 1:
            assert got["slot"][i] in slots, i
        elif not slots:
            assert got["slot"][i] == -1
    assert (got["slot"] >= 0).sum() >= 10, "the rays must hit something"


def test_occlusion_is_the_closest_hit_prefix(scene):
    rng = np.random.default_rng(6)
    rays, closest = Q.mixed_rays(scene, seed=13, n_each=1000)
    for t_max in (None, Q.t_max_mix(closest, rng), np.float32(rng.random(len(rays)) * 5)):
        near = Q.oracle_query(scene, rays, t_max)
        anyh = Q.oracle_query(scene, rays, t_max, any_hit=True)
        assert np.array_equal(anyh["occluded"], near["slot"] >= 0)
        assert np.array_equal(near["occluded"], near["slot"] >= 0)
        assert anyh["counters"]["rays"] == near["counters"]["rays"] == len(rays)
        for k in ("nodes", "leaves", "accepts"):
            assert anyh["counters"][k] <= near["counters"][k], k
    assert anyh["occluded"].any() and not anyh["occluded"].all()


def test_t_max_edges_miss(scene):
    rays, closest = Q.mixed_rays(scene, seed=14, n_each=200, grid=(16, 12))
    for t in (0.0, float(Q.EPS), -1.0, np.nan):
        got = Q.oracle_query(scene, rays, np.full(len(rays), t, dtype=np.float32), surface=True)
        assert (got["slot"] == -1).all() and np.isinf(got["t"]).all() and (got["u"] == 0).all() and (got["v"] == 0).all()
        assert not got["surface"].any()
    hit = np.isfinite(closest)
    got = Q.oracle_query(scene, rays[hit], closest[hit])
    assert (got["slot"] == -1).all(), "t_max equal to the closest t is exclusive"


def test_surface_record_matches_the_triangle(scene):
    rays, _ = Q.mixed_rays(scene, seed=15, n_each=200, grid=(16, 12))
    got = Q.oracle_query(scene, rays, surface=True)
    hit = got["slot"] >= 0
    s = got["surface"]
    p = rays[:, :3] + rays[:, 3:] * np.where(hit, got["t"], 0)[:, None]
    assert np.array_equal(Q.bits(s[hit, 0:3]), Q.bits(p[hit].astype(np.float32)))
    assert not s[~hit].any()


@pytest.mark.skipif(not Q.ref_available(),
                    reason="needs the reference's own sources (set RT_REFERENCE_DIR to a reference checkout)")
def test_oracle_query_equals_reference_ray_scene_hit(scene):
    rng = np.random.default_rng(7)
    rays, closest = Q.mixed_rays(scene, seed=16, n_each=150, grid=(16, 12))
    t_max = Q.t_max_mix(closest, rng)
    got = Q.oracle_query(scene, rays, t_max, surface=True)
    for i, ray in enumerate(rays):
        h = Q.ref_query(scene, ray, t_max[i])
        if got["slot"][i] < 0:
            # the reference leaves hit.distance at t_max on a miss
            assert Q.bits(np.float32([h.distance])) == Q.bits(t_max[i:i + 1]), i
            continue
        want = np.array([h.point.x, h.point.y, h.point.z, h.normal.x, h.normal.y, h.normal.z,
                         h.normal_geo.x, h.normal_geo.y, h.normal_geo.z, h.tex_coords.x, h.tex_coords.y], dtype=np.float32)
        assert Q.bits(np.float32([h.distance])) == Q.bits(got["t"][i:i + 1]), i
        assert np.array_equal(Q.bits(want), Q.bits(got["surface"][i])), i
