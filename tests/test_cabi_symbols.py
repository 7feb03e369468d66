"""The C-ABI libraries load without a GPU and export every function include/*.h and rt_host.h declare.
No compute call is made here."""
import ctypes as C
import os
import re

import pytest

from helpers import ROOT
from raytracing_c_b200 import _ffi

DECL = re.compile(r"^\s*(?:extern\s+)?(?:[A-Za-z_][\w\s\*]*?[\s\*])([a-z_][a-z0-9_]*)\s*\([^;{]*\)\s*;", re.M)


def declared(header: str) -> set[str]:
    text = open(os.path.join(ROOT, header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"static inline[^{]*\{.*?\n\}", "", text, flags=re.S)
    names = set(DECL.findall(text))
    return {n for n in names if not n.startswith("bvh_n_")}


def test_gpu_library_exports_every_declared_entry_point():
    lib = _ffi.gpu_lib()
    want = declared("include/raytracer.h") | declared("include/denoiser.h") | declared("include/rt_gpu.h")
    assert {"render_thread_proc", "rendering_context_is_finished", "rendering_context_finish", "lightmap_bake",
            "denoise_image", "rt_gpu_scene_upload", "rt_gpu_render_accum_device"} <= want
    for name in sorted(want):
        assert hasattr(lib, name), f"libraytracer_gpu.so does not export {name}"
    assert want == set(_ffi.GPU_EXPORTS), "the ctypes export list and the headers disagree"


def test_host_library_exports_every_declared_entry_point():
    lib = _ffi.host_lib()
    want = declared("raytracing_c_b200/host/rt_host.h") | {"scene_init", "scene_destroy"}
    for name in sorted(want):
        assert hasattr(lib, name), f"librt_host.so does not export {name}"
    assert want == set(_ffi.HOST_EXPORTS)


def test_struct_layouts_match_the_headers():
    assert C.sizeof(_ffi.Triangle) == 112 and C.sizeof(_ffi.Scene) == 208 and C.sizeof(_ffi.RenderingContext) == 80
    assert C.sizeof(_ffi.Image) == 48 and C.sizeof(_ffi.PBRShaderData) == 80 and C.sizeof(_ffi.GPUOptions) == 44


def test_no_gpu_means_a_loud_error_not_a_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = _ffi.gpu_lib()
    assert lib.rt_gpu_init(0) != 0
    assert b"no CPU fallback" in lib.rt_gpu_last_error()


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "raytracing_c_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".cuh", ".h")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                # comments may mention the oracle; code may not reach it
                for needle in ("liboracle", "oracle_ffi", "oracle/", '#include "oracle', "oracle_"):
                    assert needle not in text, f"{os.path.join(dirpath, f)} references {needle}"
