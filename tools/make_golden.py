"""Generate tests/golden/reference_vectors.npz from the reference's OWN code.

Needs a reference checkout named by RT_REFERENCE_DIR: builds oracle/_ref/libref.so — the
reference's raytracer.c / scene.c / denoiser.c / driver.c compiled unmodified over the Codin
stand-in — and records small input/output vectors of the hot path:

  bvh_sha256/<model>          sha256 of scene_init's node bytes, SoA bytes and the non-pointer part
                              of every Triangle_AOS (reference scene.c:416)
  radiance/<case>             cast_ray (raytracer.c:505) per (pixel, sample), rt_path_seed seeding,
                              exact primary rays
  denoise_in / denoise_out    denoise_image (denoiser.c:129)
  hash12_xy / hash12_out      hash12x8 lane 0 (raytracer.c:584)
  bilinear_uv / bilinear_out  sample_texture_bilinear (driver.c:49) on the procedural environment
  background_dir / _out       sample_background (driver.c:95)
  lightmap/<case>             lightmap_bake (raytracer.c:722), u8 image, both generator copies started from the
                              recorded states (the sequential "reference" seed mode)
  reference_mode/<case>       render_thread_proc as shipped (one thread, one RNG stream from 0, _mm256_rsqrt_ps primary
                              rays), u8 image; rsqrt_in / rsqrt_out fingerprint the recording CPU's _mm256_rsqrt_ps
  per_sample/<case>           cast_ray per (pixel, sample) with a non-zero user seed; denoise_frame_in / _out:
                              denoise_image on the oracle's u8 frame of the same render

quad.obj and fov_test.obj are absent from bvh_sha256: the reference's builder has undefined
behaviour on them (SURVEY.md §2.3 Q1/Q2).
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_ffi  # noqa: E402
import ref_ffi  # noqa: E402
from helpers import CAMERAS  # noqa: E402
from raytracing_c_b200 import driver  # noqa: E402
from raytracing_c_b200._ffi import Vec2, Vec3  # noqa: E402

MODELS = os.path.join(ROOT, "assets", "models")
OUT = os.path.join(ROOT, "tests", "golden")

RADIANCE_CASES = {
    # name: (model, width, height, spp, bounces, material override, camera)
    "spheres_24x24x4": ("spheres.glb", 24, 24, 4, 8, {}, None),
    "helmet_24x16x2": ("helmet.glb", 24, 16, 2, 8, {}, None),
    "sheen_injected_16x16x4": ("sheen.glb", 16, 16, 4, 8, {"sheen": 1.0, "sheen_tint": 0.5}, None),
    "tower_16x16x2": ("tower.obj", 16, 16, 2, 8, {}, dict(eye=(0.0, 12.5, 40.0), target=(0.0, 12.5, 0.0))),
    "spheres_2bounce_16x16x2": ("spheres.glb", 16, 16, 2, 2, {"anisotropic_strength": 0.6}, None),
}


LIGHTMAP_CASES = {
    # name: (model, width, height, samples, emission override, dir_state, shader_state)
    "tower_64x48x3": ("tower.obj", 64, 48, 3, (30.0, 20.0, 10.0), 123, 7),
    "spheres_48x48x2": ("spheres.glb", 48, 48, 2, (30.0, 20.0, 10.0), 99, 5),
}


# tests/test_oracle_vs_ref.py reads these under the same keys: (model, width, height, spp, material override)
REFERENCE_MODE_CASES = [("spheres.glb", 96, 64, 4, {}), ("helmet.glb", 64, 48, 3, {}),
                        ("sheen.glb", 48, 48, 4, {"sheen": 1.0, "sheen_tint": 1.0}), ("tower.obj", 48, 32, 2, {})]
SEEDED_CASE = ("spheres.glb", 20, 12, 3, 99)         # model, width, height, spp, user seed


def reference_mode_key(model, w, h, spp):
    return f"reference_mode/{model}_{w}x{h}x{spp}"


def seeded_key(model, w, h, spp, seed):
    return f"per_sample/{model}_{w}x{h}x{spp}_seed{seed}"


def scene_digest(scene) -> str:
    n_nodes, n_slots = scene.bvh.nodes.len, scene.triangles.len
    h = hashlib.sha256()
    h.update(C.string_at(scene.bvh.nodes.data, n_nodes * 192))
    h.update(C.string_at(scene.triangles.x[0], n_slots * 36))
    aos = np.frombuffer(C.string_at(scene.triangles.aos, n_slots * 112), dtype=np.uint8).reshape(n_slots, 112)
    h.update(np.ascontiguousarray(aos[:, :96]).tobytes())
    return h.hexdigest()


def load_ref(model, override=None, camera=None):
    r = ref_ffi.lib()
    cam = driver.look_at(**camera) if camera else None
    loaded = driver.load_scene(os.path.join(MODELS, model), shader_proc=r.ref_shader_proc(),
                               background_proc=r.ref_background_proc(), builder=ref_ffi.scene_builder(), camera=cam)
    for i in range(loaded.model.n_materials):
        for k, v in (override or {}).items():
            setattr(loaded.model.materials[i], k, v)
    return loaded


def main():
    os.makedirs(OUT, exist_ok=True)
    r = ref_ffi.lib()
    arrays, digests = {}, {}
    for model in ["spheres.glb", "sheen.glb", "tower.obj", "helmet.glb"]:
        loaded = load_ref(model)
        digests[model] = {"sha256": scene_digest(loaded.scene), "depth": int(loaded.scene.bvh.depth),
                          "nodes": int(loaded.scene.bvh.nodes.len), "slots": int(loaded.scene.triangles.len)}
        loaded.close()
    for name, (model, w, h, spp, bounces, override, camera) in RADIANCE_CASES.items():
        loaded = load_ref(model, override, camera)
        arrays["radiance/" + name] = ref_ffi.cast_rays_per_sample(loaded, w, h, spp, bounces)
        loaded.close()

    for name, (model, w, h, n, emission, dir_state, shader_state) in LIGHTMAP_CASES.items():
        loaded = load_ref(model, {"emission": Vec3(*emission)})
        arrays["lightmap/" + name] = ref_ffi.lightmap_bake(loaded, w, h, n, dir_state=dir_state, shader_state=shader_state)
        loaded.close()

    rng = np.random.default_rng(2026)
    img = rng.integers(0, 256, size=(40, 48, 3), dtype=np.uint8)
    img[:20] = (img[:20] // 48) * 48
    img[25:35, 10:30] = 200
    arrays["denoise_in"], arrays["denoise_out"] = img, ref_ffi.denoise(img)

    xy = np.stack([rng.uniform(0, 2000 * 50, 512), rng.uniform(0, 1200, 512)], axis=1).astype(np.float32)
    xy[:16, 0] = np.arange(16) * 50.0
    arrays["hash12_xy"] = xy
    arrays["hash12_out"] = np.array([r.ref_hash12(float(a), float(b)) for a, b in xy], dtype=np.float32)

    loaded = load_ref("quad.obj") if False else load_ref("sheen.glb")
    uv = rng.uniform(-2.5, 2.5, size=(256, 2)).astype(np.float32)
    uv[:8] = [(0, 0), (1, 1), (0.999999, 0.999999), (-0.25, 0.5), (-1e-9, 2.0), (0.5, -3.0), (1.5, 0.25), (0.9995, 0.0005)]
    arrays["bilinear_uv"] = uv
    arrays["bilinear_out"] = np.array([(c.x, c.y, c.z) for c in (r.ref_sample_texture_bilinear(C.byref(loaded.background), Vec2(*p)) for p in uv)], dtype=np.float32)
    d = rng.normal(size=(256, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = d.astype(np.float32)
    d[:6] = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    arrays["background_dir"] = d
    arrays["background_out"] = np.array([(c.x, c.y, c.z) for c in (r.ref_sample_background(C.byref(loaded.background), Vec3(*p)) for p in d)], dtype=np.float32)
    loaded.close()

    for model, w, h, spp, override in REFERENCE_MODE_CASES:
        loaded = load_ref(model, override, CAMERAS.get(model))
        arrays[reference_mode_key(model, w, h, spp)] = ref_ffi.render_reference_mode(loaded, w, h, spp)
        loaded.close()
    rng = np.random.default_rng(663)
    x = np.concatenate([np.geomspace(1e-4, 1e4, 2048), rng.uniform(0.0, 8.0, 2048)]).astype(np.float32)
    arrays["rsqrt_in"], arrays["rsqrt_out"] = x, oracle_ffi.rsqrt_ps(x)
    model, w, h, spp, seed = SEEDED_CASE
    loaded = load_ref(model)
    arrays[seeded_key(*SEEDED_CASE)] = ref_ffi.cast_rays_per_sample(loaded, w, h, spp, user_seed=seed)
    loaded.close()
    loaded = driver.load_scene(os.path.join(MODELS, model), shader_proc=oracle_ffi.shader_proc(),
                               background_proc=oracle_ffi.background_proc())
    frame = oracle_ffi.render(loaded, w, h, spp, 8, n_threads=2, user_seed=seed)["pixels"]
    loaded.close()
    arrays["denoise_frame_in"], arrays["denoise_frame_out"] = frame, ref_ffi.denoise(frame)

    np.savez_compressed(os.path.join(OUT, "reference_vectors.npz"), **arrays)
    meta = {"generator": "tools/make_golden.py", "source": "oracle/_ref/libref.so = $RT_REFERENCE_DIR/{raytracer,scene,denoiser,driver}.c unmodified + oracle/codin_shim",
            "bvh": digests, "radiance_cases": {k: dict(model=v[0], width=v[1], height=v[2], spp=v[3], bounces=v[4], override=v[5], camera=v[6]) for k, v in RADIANCE_CASES.items()},
            "lightmap_cases": {k: dict(model=v[0], width=v[1], height=v[2], samples=v[3], emission=list(v[4]), dir_state=v[5], shader_state=v[6])
                               for k, v in LIGHTMAP_CASES.items()}}
    json.dump(meta, open(os.path.join(OUT, "reference_vectors.json"), "w"), indent=1)
    print("wrote", OUT, {k: v.shape for k, v in arrays.items()})


if __name__ == "__main__":
    main()
