"""First-surface AOVs, for the tests: the CPU reference (oracle_render_aov, tests/csrc/aov_oracle.c) and the device-level
GPU call on torch tensors.  TEST INFRASTRUCTURE ONLY.

The C file is compiled on first use into a private temporary directory (the tree is never written).  Records are
(H, W, 16) float32 arrays in RT_GPU_AOV order; `fields` splits them into the named sums.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

import oracle_ffi
from helpers import CSRC, MODELS, ROOT, bits  # noqa: F401  (bits is re-exported)
from raytracing_c_b200._ffi import Scene, isize

FLOATS = 16
# RT_GPU_AOV: name -> (first float, width)
LAYOUT = {"albedo": (0, 3), "coverage": (3, 1), "normal": (4, 3), "depth": (7, 1),
          "position": (8, 3), "roughness": (11, 1), "emission": (12, 3), "metalness": (15, 1)}

_aov_lib = None


def aov_lib() -> C.CDLL:
    """oracle_render_aov, built with the oracle's flags over its unmodified oracle_trace.c and oracle_shade.c."""
    global _aov_lib
    if _aov_lib is None:
        oracle_ffi.lib()                                   # builds liboracle.so if it is missing
        o = oracle_ffi.ORACLE_DIR
        path = oracle_ffi.build_lib("libaov_oracle.so", [
            "-O2", "-std=gnu11", "-mavx2", "-mfma", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"),
            "-I", o, os.path.join(CSRC, "aov_oracle.c"), "-lpthread", "-lm"])
        lib = C.CDLL(path)
        lib.oracle_render_aov.argtypes = [C.POINTER(Scene), isize, isize, isize, isize, isize, C.c_void_p, C.c_void_p,
                                          C.c_int32]
        lib.oracle_render_aov.restype = None
        _aov_lib = lib
    return _aov_lib


def fields(records) -> dict:
    return {k: (records[..., a:a + n] if n == 3 else records[..., a]) for k, (a, n) in LAYOUT.items()}


def oracle_aov(loaded, width, height, sample_begin, sample_end, max_bounces=8, n_threads=8) -> dict:
    """{"records": (H, W, 16) float32 sums, "counters": the eight work counters}"""
    rec = np.zeros((height, width, FLOATS), dtype=np.float32)
    ctr = np.zeros(8, dtype=np.uint64)
    aov_lib().oracle_render_aov(C.byref(loaded.scene), width, height, sample_begin, sample_end, max_bounces,
                                rec.ctypes.data, ctr.ctypes.data, n_threads)
    return {"records": rec, "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr)))}


def device_aov(loaded, width, height, sample_begin, sample_end, max_bounces=8, aov=None, accumulate=False,
               stream=None) -> dict:
    """rt_gpu_render_aov_device on a torch buffer, on `stream` (default: torch's current stream).  `aov` (a CUDA float32
    tensor of width * height * 16) is continued from with accumulate; a fresh one is filled with 7.0 first, so a record
    the call does not write shows.  Returns the records as numpy and the eight counters."""
    import torch
    from raytracing_c_b200 import driver, gpu_lib
    from raytracing_c_b200._ffi import gpu_check
    buf = aov if aov is not None else torch.full((width * height * FLOATS,), 7.0, dtype=torch.float32, device="cuda")
    ctr = torch.zeros(8, dtype=torch.int64, device="cuda")
    st = stream or torch.cuda.current_stream()
    driver.register_callbacks(loaded)
    gpu_check(gpu_lib().rt_gpu_render_aov_device(C.byref(loaded.scene), width, height, sample_begin, sample_end,
                                                 max_bounces, int(accumulate), buf.data_ptr(), ctr.data_ptr(),
                                                 st.cuda_stream))
    st.synchronize()
    return {"records": buf.cpu().numpy().reshape(height, width, FLOATS),
            "counters": dict(zip(oracle_ffi.COUNTER_NAMES, map(int, ctr.cpu().numpy())))}


def load_default_camera(name):
    """A shipped model with the camera its loader sets (helpers.load overrides quad's and tower's, DESIGN.md §6
    deviation 6: the default camera sits inside those models, so camera rays meet back faces)."""
    from raytracing_c_b200 import driver
    return driver.load_scene(os.path.join(MODELS, name), shader_proc=oracle_ffi.shader_proc(),
                             background_proc=oracle_ffi.background_proc())
