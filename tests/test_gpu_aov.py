"""First-surface AOVs on the GPU (rt_gpu_render_aov*, csrc/rt_render.cu) against their CPU reference (oracle_render_aov):
every field of every record and the eight work counters bit-exact on the six shipped models and inside tower.obj, for
walk counts 0/1/2/8 and two sample offsets, and on one whole 1080p helmet frame; agreement with the renderer's own
accumulator and counters; split ranges, chunked runs and the host form equal to one device call; ordering against
uploads and renders; fast_math; refusals before launch; the compile-time budget of the two new kernels.
"""
import contextlib
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import aov_ffi as A
from helpers import load
from raytracing_c_b200 import driver, gpu_lib
from raytracing_c_b200._ffi import gpu_check

pytestmark = pytest.mark.gpu

MODEL_NAMES = ["fov_test.obj", "quad.obj", "tower.obj", "spheres.glb", "sheen.glb", "helmet.glb"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing_c_b200", "csrc", "libraytracer_gpu.so")


@pytest.fixture(scope="module", autouse=True)
def _gpu():
    gpu_check(gpu_lib().rt_gpu_init(0))
    yield
    driver.set_options()


def upload(loaded):
    driver.register_callbacks(loaded)
    gpu_check(gpu_lib().rt_gpu_scene_upload(C.byref(loaded.scene)))


@pytest.fixture(scope="module", params=MODEL_NAMES + ["tower.obj:inside"])
def scene(request):
    loaded = A.load_default_camera("tower.obj") if request.param.endswith(":inside") else load(request.param)
    upload(loaded)
    yield request.param, loaded
    loaded.close()


def assert_equal(got, want):
    bad = A.bits(got["records"]) != A.bits(want["records"])
    assert not bad.any(), f"records differ on {int(bad.any(axis=-1).sum())} pixels, fields {np.nonzero(bad.any(axis=(0, 1)))[0]}"
    assert got["counters"] == want["counters"]


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


# (max_bounces, sample_begin)
CASES = [(8, 0), (1, 13), (2, 0), (0, 13), (8, 13), (2, 13)]


def test_bit_exact_against_the_oracle(scene):
    name, loaded = scene
    w, h, n = (256, 192, 8) if name == "helmet.glb" else (64, 48, 16)
    for max_bounces, begin in CASES:
        want = A.oracle_aov(loaded, w, h, begin, begin + n, max_bounces)
        got = A.device_aov(loaded, w, h, begin, begin + n, max_bounces)
        assert_equal(got, want)
        if max_bounces == 0:
            assert not got["records"].any() and not any(got["counters"].values())
        else:
            assert got["counters"]["samples"] == w * h * n and got["counters"]["shades"] > 0
    if name == "tower.obj:inside":
        assert want["counters"]["passthrough"] > 0


def test_whole_helmet_frame():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 1920, 1080
        want = A.oracle_aov(loaded, w, h, 0, 16, 8, n_threads=max(8, os.cpu_count() or 8))
        assert_equal(A.device_aov(loaded, w, h, 0, 16, 8), want)
    finally:
        loaded.close()


@pytest.mark.parametrize("name", ["helmet.glb", "sheen.glb", "tower.obj"])
def test_one_walk_agrees_with_the_renderer(name):
    """max_bounces = 1: a path ends at its first shade with radiance = emission, so on every fully covered pixel the
    emission sum is the renderer's accumulator, and the total coverage is its SHADES counter."""
    import torch
    loaded = load(name)
    try:
        upload(loaded)
        w, h, begin, end = 160, 90, 2, 14
        accum = torch.zeros(h * w * 3, dtype=torch.float32, device="cuda")
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        gpu_check(gpu_lib().rt_gpu_render_accum_device(C.byref(loaded.scene), w, h, begin, end, 1, 0, 0, accum.data_ptr(),
                                                       None, None, ctr.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        rendered = accum.cpu().numpy().reshape(h, w, 3)
        got = A.device_aov(loaded, w, h, begin, end, 1)
        f = A.fields(got["records"])
        full = f["coverage"] == end - begin
        assert full.any()
        assert np.array_equal(A.bits(f["emission"][full]), A.bits(rendered[full]))
        counters = dict(zip(got["counters"], map(int, ctr.cpu().numpy())))
        assert float(f["coverage"].sum()) == counters["shades"]
        assert got["counters"] == counters
    finally:
        loaded.close()


def test_split_ranges_chunks_and_host_form_equal_one_call():
    import torch
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h = 200, 120
        whole = A.device_aov(loaded, w, h, 3, 40, 8)
        buf = torch.full((w * h * A.FLOATS,), 7.0, dtype=torch.float32, device="cuda")
        a = A.device_aov(loaded, w, h, 3, 20, 8, aov=buf)
        b = A.device_aov(loaded, w, h, 20, 40, 8, aov=buf, accumulate=True)
        assert np.array_equal(A.bits(b["records"]), A.bits(whole["records"]))
        assert {k: a["counters"][k] + b["counters"][k] for k in a["counters"]} == whole["counters"]
        with chunk_paths(w * h * 5):               # chunks of 5 samples of every pixel (the last one 2)
            assert_equal(A.device_aov(loaded, w, h, 3, 40, 8), whole)
        host = driver.render_aov(loaded, w, h, 37, 8, sample_begin=3)
        assert gpu_lib().rt_gpu_last_launches() == 1 + 1 + 7 + 8 + 1   # camera copies, primary, 7 traces, 8 surface, sum
        for k, v in A.fields(whole["records"]).items():
            assert np.array_equal(A.bits(host[k]), A.bits(v)), k
    finally:
        loaded.close()


def test_on_a_user_stream_right_after_upload():
    """A fresh scene, uploaded and asked for AOVs at once on a torch stream: the call waits for the texels."""
    import torch
    loaded = load("helmet.glb")
    try:
        w, h = 128, 96
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        upload(loaded)
        with torch.cuda.stream(stream):
            got = A.device_aov(loaded, w, h, 0, 4, 8, stream=stream)
        torch.cuda.synchronize()
        assert_equal(got, A.oracle_aov(loaded, w, h, 0, 4, 8))
    finally:
        loaded.close()


def test_render_aov_render_gives_the_same_accumulator():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        w, h, spp = 160, 90, 4
        driver.render(loaded, w, h, spp, 8)
        first = driver.read_accum(w, h).copy()
        before = A.device_aov(loaded, w, h, 0, 4, 8)
        driver.render(loaded, w, h, spp, 8)
        assert np.array_equal(A.bits(driver.read_accum(w, h)), A.bits(first))
        assert_equal(A.device_aov(loaded, w, h, 0, 4, 8), before)
    finally:
        loaded.close()


def test_camera_change_between_calls():
    """The call reads the camera the Scene holds at the call, as a render does."""
    loaded = load("spheres.glb")
    try:
        upload(loaded)
        w, h = 64, 48
        first = A.device_aov(loaded, w, h, 0, 4, 8)
        loaded.scene.camera = driver.look_at(eye=(0.5, 0.3, 6.0), target=(0.0, 0.0, 0.0))
        moved = A.device_aov(loaded, w, h, 0, 4, 8)
        assert_equal(moved, A.oracle_aov(loaded, w, h, 0, 4, 8))
        assert not np.array_equal(A.bits(moved["records"]), A.bits(first["records"]))
    finally:
        loaded.close()


def test_fast_math_option_does_not_apply():
    loaded = load("helmet.glb")
    try:
        upload(loaded)
        want = A.oracle_aov(loaded, 96, 64, 0, 6, 8)
        driver.set_options(fast_math=True)
        assert_equal(A.device_aov(loaded, 96, 64, 0, 6, 8), want)
    finally:
        driver.set_options()
        loaded.close()


def test_refusals_and_empty_calls():
    import torch
    loaded = load("quad.obj")
    other = load("quad.obj")
    try:
        upload(loaded)
        gpu = gpu_lib()
        w, h = 32, 16
        buf = torch.full((w * h * A.FLOATS + 4,), 7.0, dtype=torch.float32, device="cuda")
        ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
        sc = C.byref(loaded.scene)
        st = torch.cuda.current_stream().cuda_stream

        def dev(scene=sc, width=w, height=h, begin=0, end=2, bounces=8, out=buf.data_ptr(), accumulate=0):
            return gpu.rt_gpu_render_aov_device(scene, width, height, begin, end, bounces, accumulate, out, ctr.data_ptr(), st)
        host = np.zeros((h, w, A.FLOATS), dtype=np.float32)
        cases = [
            (lambda: dev(width=0), "empty"),
            (lambda: dev(height=-1), "empty"),
            (lambda: dev(width=1 << 20, height=1 << 12), "too large"),
            (lambda: dev(width=1 << 31), "too large"),
            (lambda: dev(begin=-1), "samples"),
            (lambda: dev(begin=5, end=4), "samples"),
            (lambda: dev(end=1 << 31), "samples"),
            (lambda: dev(bounces=-1), "max_bounces"),
            (lambda: dev(out=None), "aov"),
            (lambda: dev(out=buf.data_ptr() + 4), "aligned"),
            (lambda: dev(scene=C.byref(other.scene)), "resident"),
            (lambda: dev(scene=None), "scene"),
            (lambda: gpu.rt_gpu_render_aov(sc, w, h, 0, 1, 8, None), "aov"),
            (lambda: gpu.rt_gpu_render_aov(sc, w, h, 2, 1, 8, host.ctypes.data), "samples"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in gpu.rt_gpu_last_error().decode(), word
        assert gpu.rt_gpu_scene_device_bytes(C.byref(other.scene)) == 0, "a refused call uploads nothing"
        torch.cuda.synchronize()
        assert (buf == 7).all() and not ctr.any()
        # empty range or no walks: records kept with accumulate, zeroed without; nothing traced or counted
        for kw in (dict(begin=5, end=5), dict(bounces=0)):
            assert dev(accumulate=1, **kw) == 0
            torch.cuda.synchronize()
            assert (buf == 7).all()
            assert dev(**kw) == 0
            torch.cuda.synchronize()
            assert not buf[:w * h * A.FLOATS].any() and (buf[w * h * A.FLOATS:] == 7).all() and not ctr.any()
            buf.fill_(7.0)
        # the library still answers after the refusals
        assert_equal(A.device_aov(loaded, w, h, 0, 3, 8), A.oracle_aov(loaded, w, h, 0, 3, 8))
    finally:
        other.close()
        loaded.close()


BUDGET = {   # mangled-name fragment -> (max registers per thread, max bytes of stack), from -Xptxas -v
    "rt_aov_surface_kernel": (32, 0),
    "rt_aov_accumulate_kernel": (64, 16),
}


@pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB), reason="needs the built library and cuobjdump")
def test_new_kernels_keep_their_register_budget():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
    found = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        for key in BUDGET:
            if key in m.group(1):
                found[key] = (int(m.group(2)), int(m.group(3)))
    assert set(found) == set(BUDGET), f"kernels missing from the library: {set(BUDGET) - set(found)}"
    for key, (regs, stack) in found.items():
        assert regs <= BUDGET[key][0], f"{key}: {regs} registers (budget {BUDGET[key][0]})"
        assert stack <= BUDGET[key][1], f"{key}: {stack} bytes of stack (budget {BUDGET[key][1]})"
