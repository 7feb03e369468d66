"""The slot map of rt_scene_init_slots and the CPU restatement of the refit, pinned to scene_init (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

import refit_ffi as R
from helpers import MODEL_NAMES, load, scene_buffers, scene_digest
from raytracing_c_b200 import driver
from raytracing_c_b200._ffi import Scene, host_lib


@pytest.fixture(scope="module", params=MODEL_NAMES)
def loaded(request):
    sc = load(request.param)
    yield sc
    sc.close()


def test_slot_map_build_equals_scene_init(loaded):
    plain = Scene()
    host_lib().scene_init(C.byref(plain), loaded.model.triangles)
    try:
        assert scene_digest(plain) == scene_digest(loaded.scene)
    finally:
        host_lib().scene_destroy(C.byref(plain))

    n, slots = loaded.n_triangles, loaded.scene.triangles.len
    slot_of = loaded.slot_of
    assert slot_of.shape == (n,) and len(np.unique(slot_of)) == n
    assert slot_of.min() >= 0 and slot_of.max() < slots
    aos = np.ctypeslib.as_array((C.c_uint64 * (slots * 14)).from_address(loaded.scene.triangles.aos)).reshape(slots, 14)
    occupied = (aos[:, 12] != 0) | (aos[:, 13] != 0)          # the Shader pair
    assert occupied.sum() == n and occupied[slot_of].all()
    src = np.ctypeslib.as_array((C.c_float * (n * 28)).from_address(C.addressof(loaded.model.triangles.data.contents)))
    src_pos = src.reshape(n, 28)[:, :9].reshape(n, 3, 3)               # [triangle][vertex][axis]
    pos = driver.scene_positions(loaded).transpose(2, 1, 0)           # [slot][vertex][axis]
    assert np.array_equal(pos[slot_of].view(np.uint32), src_pos.view(np.uint32))


def test_identity_refit_reproduces_scene_init(loaded):
    nodes, soa, aos96 = scene_buffers(loaded.scene)
    R.oracle_refit(loaded, driver.scene_positions(loaded))
    assert scene_buffers(loaded.scene) == (nodes, soa, aos96)
    R.oracle_refit(loaded, driver.scene_positions(loaded), driver.scene_normals(loaded))
    assert scene_buffers(loaded.scene) == (nodes, soa, aos96)


def test_refit_there_and_back(loaded):
    """A deformation and the refit back to the original positions restore every byte."""
    before = scene_buffers(loaded.scene)
    pos = driver.scene_positions(loaded)
    R.oracle_refit(loaded, R.deform(pos))
    moved = scene_buffers(loaded.scene)
    assert moved[0] != before[0] and moved[1] != before[1]
    R.oracle_refit(loaded, pos)
    assert scene_buffers(loaded.scene) == before
