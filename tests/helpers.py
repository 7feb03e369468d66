"""Shared helpers for the test-suite (paths, scene loading with oracle callbacks, layout digests, the GPU session)."""
import contextlib
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_ffi
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing_c_b200", "csrc", "libraytracer_gpu.so")
CSRC = os.path.join(ROOT, "tests", "csrc")
MODELS = os.path.join(ROOT, "assets", "models")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]

# Camera overrides recorded in DESIGN.md (SURVEY §8d configs 2 and 5): the default camera sits
# inside quad.obj's plane and inside tower.obj's footprint.
CAMERAS = {
    "quad.obj": dict(eye=(3.0, 0.0, 0.0), target=(0.0, 0.0, 0.0)),
    "tower.obj": dict(eye=(0.0, 12.5, 40.0), target=(0.0, 12.5, 0.0)),
}


def load(name, builder=None, camera=None, **material_override):
    cam = driver.look_at(**camera) if camera else (driver.look_at(**CAMERAS[name]) if name in CAMERAS else None)
    loaded = driver.load_scene(os.path.join(MODELS, name), shader_proc=oracle_ffi.shader_proc(),
                               background_proc=oracle_ffi.background_proc(), camera=cam, builder=builder)
    for i in range(loaded.model.n_materials):
        for key, value in material_override.items():
            setattr(loaded.model.materials[i], key, value)
    return loaded


def scene_buffers(scene):
    """(node bytes, SoA bytes, AoS bytes without the Shader pointers)"""
    n_nodes, n_slots = scene.bvh.nodes.len, scene.triangles.len
    nodes = C.string_at(scene.bvh.nodes.data, n_nodes * 192)
    soa = C.string_at(scene.triangles.x[0], n_slots * 36)
    aos = np.frombuffer(C.string_at(scene.triangles.aos, n_slots * 112), dtype=np.uint8).reshape(n_slots, 112)
    return nodes, soa, np.ascontiguousarray(aos[:, :96]).tobytes()


def scene_digest(scene) -> str:
    h = hashlib.sha256()
    for part in scene_buffers(scene):
        h.update(part)
    return h.hexdigest()


def golden():
    arrays = np.load(os.path.join(GOLDEN_DIR, "reference_vectors.npz"))
    meta = json.load(open(os.path.join(GOLDEN_DIR, "reference_vectors.json")))
    return arrays, meta


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module", autouse=True)
def gpu_session():
    """Device 0 for a GPU test module (import it into the module), default options restored afterwards."""
    gpu_check(gpu_lib().rt_gpu_init(0))
    yield
    driver.set_options()


def upload(loaded):
    driver.register_callbacks(loaded)
    gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))


@contextlib.contextmanager
def chunk_paths(n):
    """Path-queue chunks of at most n paths (RT_GPU_CHUNK_PATHS, read at every launch)."""
    old = os.environ.get("RT_GPU_CHUNK_PATHS")
    os.environ["RT_GPU_CHUNK_PATHS"] = str(n)
    try:
        yield
    finally:
        if old is None:
            del os.environ["RT_GPU_CHUNK_PATHS"]
        else:
            os.environ["RT_GPU_CHUNK_PATHS"] = old
