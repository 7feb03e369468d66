"""The CPU reference of rt_gpu_render_aov (oracle_render_aov, tests/csrc/aov_oracle.c), which the GPU call is checked
against, pinned to the oracle renderer and the query oracle:
  - with one walk, a fully covered pixel's emission sum is the oracle renderer's radiance sum bit for bit (the path
    ends at its first shade with radiance = emission), and the work counters are the renderer's;
  - a covered sample's position is the closest-hit point of its camera ray;
  - shading normals of covered samples have unit length;
  - inside tower.obj (the loader's own camera), camera rays step through back faces and some pixels are covered only
    after such a step.
"""
import numpy as np
import pytest

import aov_ffi as A
import cast_rays_ffi as R
import oracle_ffi
import query_ffi as Q
from helpers import MODEL_NAMES, load


@pytest.fixture(scope="module", params=MODEL_NAMES)
def scene(request):
    loaded = load(request.param)
    yield loaded
    loaded.close()


def test_one_walk_emission_is_the_renderers_radiance(scene):
    w, h, begin, end = 48, 32, 3, 11
    got = A.oracle_aov(scene, w, h, begin, end, max_bounces=1)
    f = A.fields(got["records"])
    want = oracle_ffi.render(scene, w, h, end, 1, n_threads=4, user_seed=0, sample_begin=begin, sample_end=end)
    full = f["coverage"] == end - begin
    assert full.any()
    assert np.array_equal(R.bits(f["emission"][full]), R.bits(want["accum"][full]))
    assert float(f["coverage"].sum()) == want["counters"]["shades"]
    assert got["counters"] == want["counters"]


def test_position_is_the_closest_hit_point(scene):
    w, h, s = 40, 30, 5
    rays = R.camera_rays(scene, w, h, s)
    hit = Q.oracle_query(scene, rays, surface=True)
    f = A.fields(A.oracle_aov(scene, w, h, s, s + 1, max_bounces=1)["records"])
    covered = f["coverage"].reshape(-1) == 1
    assert covered.any()
    assert (hit["slot"][covered] >= 0).all()
    assert np.array_equal(R.bits(f["position"].reshape(-1, 3)[covered]), R.bits(hit["surface"][covered, 0:3]))
    assert not f["position"].reshape(-1, 3)[~covered].any()


def test_normals_have_unit_length(scene):
    w, h = 32, 24
    for s in (0, 7):
        f = A.fields(A.oracle_aov(scene, w, h, s, s + 1, max_bounces=8)["records"])
        n = f["normal"][f["coverage"] == 1].astype(np.float64)
        assert len(n)
        assert np.abs(np.linalg.norm(n, axis=-1) - 1).max() < 1e-6


def test_back_face_chains_inside_tower():
    loaded = A.load_default_camera("tower.obj")
    try:
        w, h, n = 48, 32, 4
        one = A.oracle_aov(loaded, w, h, 0, n, max_bounces=1)
        many = A.oracle_aov(loaded, w, h, 0, n, max_bounces=8)
        assert one["counters"]["passthrough"] > 0 and many["counters"]["passthrough"] > one["counters"]["passthrough"]
        c1, c8 = A.fields(one["records"])["coverage"], A.fields(many["records"])["coverage"]
        stepped = (c1 == 0) & (c8 > 0)
        assert stepped.any(), "no pixel is covered only after a back-face step"
        assert (c8 >= c1).all()
        assert many["counters"]["shades"] == float(c8.sum()) and many["counters"]["samples"] == w * h * n
    finally:
        loaded.close()
