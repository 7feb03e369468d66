"""Ray queries for the tests: the CPU reference of the queries (tests/csrc/query_oracle.c), the reference's own
ray_scene_hit with an initial distance (tests/csrc/ref_query_glue.c, where a reference checkout is available), and the
seeded ray families the CPU and GPU tests share.  TEST INFRASTRUCTURE ONLY.

Both C libraries are compiled on first use into a private temporary directory (the tree is never written).
Rays are (n, 6) float32 arrays laid out as the C Ray (position, direction); t_max is (n,) float32 or None (+inf).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

import oracle_ffi
from helpers import CSRC, ROOT, bits  # noqa: F401  (bits is re-exported)
from raytracing_c_b200._ffi import Scene, isize

EPS = np.float32(0.0001)                 # the reference's EPSILON
SURFACE_FIELDS = {"point": slice(0, 3), "normal": slice(3, 6), "normal_geo": slice(6, 9), "tex_coords": slice(9, 11)}
QUERY_COUNTERS = ["rays", "nodes", "leaves", "accepts"]
HIT_DTYPE = np.dtype([("t", np.float32), ("u", np.float32), ("v", np.float32), ("slot", np.int32)])

_query_lib = None
_ref_lib = None


def query_lib() -> C.CDLL:
    """query_oracle_rays, built with the oracle's flags (no FMA contraction)."""
    global _query_lib
    if _query_lib is None:
        path = oracle_ffi.build_lib("libquery_oracle.so", [
            "-O2", "-std=gnu11", "-mavx2", "-mfma", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"),
            "-I", oracle_ffi.ORACLE_DIR, os.path.join(CSRC, "query_oracle.c"), "-lpthread", "-lm"])
        lib = C.CDLL(path)
        lib.query_oracle_rays.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p, isize, C.c_int32, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        lib.query_oracle_rays.restype = None
        _query_lib = lib
    return _query_lib


def ref_available() -> bool:
    return os.path.isdir(os.environ.get("RT_REFERENCE_DIR", ""))


def ref_query_lib() -> C.CDLL:
    """The sources of oracle/Makefile's `ref` target with ref_query_glue.c in place of ref_glue_rt.c."""
    global _ref_lib
    if _ref_lib is None:
        ref, o = os.environ["RT_REFERENCE_DIR"], oracle_ffi.ORACLE_DIR
        path = oracle_ffi.build_lib("libref_query.so", [
            "-O2", "-g", "-std=gnu11", "-mavx2", "-mfma", "-ffp-contract=off", "-w", "-Dmain=ref_driver_main",
            "-I", os.path.join(o, "codin_shim"), "-I", ref, "-I", os.path.join(ROOT, "include"), "-I", o,
            os.path.join(o, "ref_glue_common.c"), os.path.join(CSRC, "ref_query_glue.c"), os.path.join(o, "ref_glue_driver.c"),
            os.path.join(ref, "scene.c"), os.path.join(ref, "denoiser.c"), "-lpthread", "-lm"])
        _ref_lib = C.CDLL(path)
    return _ref_lib


def _ptr(a):
    return a.ctypes.data if a is not None else None


def oracle_query(loaded, rays, t_max=None, any_hit=False, surface=False, n_threads=8) -> dict:
    """query_oracle_rays: closest hit (t, u, v, slot, optional surface (n, 11)) or, with any_hit, the early-exit walk's
    occluded (bool); always the four counters."""
    rays = np.ascontiguousarray(rays, dtype=np.float32)
    n = len(rays)
    if t_max is not None:
        t_max = np.ascontiguousarray(t_max, dtype=np.float32)
    hits = None if any_hit else np.zeros(n, dtype=HIT_DTYPE)
    surf = np.zeros((n, 11), dtype=np.float32) if surface and not any_hit else None
    occ = np.zeros(n, dtype=np.uint8)
    ctr = np.zeros(4, dtype=np.uint64)
    query_lib().query_oracle_rays(C.byref(loaded.scene), rays.ctypes.data, _ptr(t_max), n, int(any_hit), _ptr(hits),
                                  _ptr(surf), occ.ctypes.data, ctr.ctypes.data, n_threads)
    out = {"occluded": occ.astype(bool), "counters": dict(zip(QUERY_COUNTERS, map(int, ctr)))}
    if hits is not None:
        out.update({k: np.ascontiguousarray(hits[k]) for k in ("t", "u", "v", "slot")})
    if surf is not None:
        out["surface"] = surf
    return out


def oracle_trace_ray(loaded, ray):
    """The oracle's oracle_trace_ray (the renderer's own walk from +inf): (slot, t)."""
    t = C.c_float()
    r = oracle_ffi.Ray()
    r.position.x, r.position.y, r.position.z, r.direction.x, r.direction.y, r.direction.z = map(float, ray)
    slot = oracle_ffi.lib().oracle_trace_ray(C.byref(loaded.scene), r, C.byref(t))
    return slot, np.float32(t.value)


def ref_query(loaded, ray, t_max):
    """The reference's ray_scene_hit with hit.distance = t_max before the walk."""
    import ref_ffi
    lib = ref_query_lib()
    lib.ref_query_ray.argtypes = [C.POINTER(Scene), oracle_ffi.Ray, C.c_float, C.POINTER(ref_ffi.RefHit)]
    lib.ref_query_ray.restype = None
    r = oracle_ffi.Ray()
    r.position.x, r.position.y, r.position.z, r.direction.x, r.direction.y, r.direction.z = map(float, ray)
    h = ref_ffi.RefHit()
    lib.ref_query_ray(C.byref(loaded.scene), r, C.c_float(float(t_max)), C.byref(h))
    return h


# ------------------------------------------------------------------------------------------------ ray families
def root_box(scene):
    """Union of the root's non-empty child boxes (BVH_Node: mins[3][8], maxs[3][8])."""
    node = np.frombuffer(C.string_at(scene.bvh.nodes.data, 192), dtype=np.float32).reshape(2, 3, 8)
    lo, hi = node[0], node[1]
    used = (hi > lo).any(axis=0)
    return lo[:, used].min(axis=1), hi[:, used].max(axis=1)


def camera_rays(scene, width, height):
    """Pinhole rays through the pixel centres of the scene camera (unit directions, raytracer.c:652-667 without jitter)."""
    m = np.array([[scene.camera.view_matrix[r][c] for c in range(4)] for r in range(3)], dtype=np.float32)
    ys, xs = np.mgrid[0:height, 0:width].astype(np.float32)
    cx = ((xs + 0.5) * 2 / width - 1) * (width / height)
    cy = -((ys + 0.5) * 2 / height - 1)
    cam = np.stack([cx, cy, np.full_like(cx, -scene.camera.focal_length)], axis=-1).reshape(-1, 3)
    d = cam @ m[:, :3].T
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = np.broadcast_to(m[:, 3], d.shape)
    return np.concatenate([o, d], axis=1).astype(np.float32)


def sphere_dirs(rng, n):
    d = rng.normal(size=(n, 3))
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def interior_rays(scene, rng, n, normalised=True):
    """Origins uniform in the root box, directions uniform on the sphere; not normalised: scaled by 10^U(-1, 1)."""
    lo, hi = root_box(scene)
    o = (lo + rng.random((n, 3)) * (hi - lo)).astype(np.float32)
    d = sphere_dirs(rng, n)
    if not normalised:
        d = (d * 10.0 ** rng.uniform(-1, 1, size=(n, 1))).astype(np.float32)
    return np.concatenate([o, d], axis=1).astype(np.float32)


def axis_rays(scene, rng, n):
    """Axis-aligned directions and directions with one zero component (infinite reciprocals: the general box test)."""
    lo, hi = root_box(scene)
    o = (lo + rng.random((n, 3)) * (hi - lo)).astype(np.float32)
    d = np.zeros((n, 3), dtype=np.float32)
    axis = rng.integers(0, 3, size=n)
    d[np.arange(n), axis] = rng.choice([-1.0, 1.0], size=n)
    half = np.arange(n) % 2 == 1                      # every second ray: one zero component, the other two random
    rnd = sphere_dirs(rng, n)
    rnd[np.arange(n), axis] = 0
    d[half] = rnd[half]
    return np.concatenate([o, d], axis=1).astype(np.float32)


def surface_rays(ray_in, hit_t, rng):
    """Rays that start exactly on the surfaces the rays `ray_in` hit (hit_t finite): half continue along the incoming
    direction (re-hit / self-intersection of the start triangle), half leave in a random direction."""
    keep = np.isfinite(hit_t)
    r, t = ray_in[keep], hit_t[keep]
    p = (r[:, :3] + r[:, 3:] * t[:, None]).astype(np.float32)
    d = r[:, 3:].copy()
    flip = np.arange(len(r)) % 2 == 1
    d[flip] = sphere_dirs(rng, int(flip.sum()))
    return np.concatenate([p, d], axis=1).astype(np.float32)


def t_max_mix(closest_t, rng):
    """Per-ray t_max cycling through: +inf, a random fraction of the closest t (misses, prunes), exactly the closest t
    (misses: the bound is exclusive), EPSILON, 0, negative, NaN, and the closest t times 1 + U(0, 1) (hits, prunes)
    (closest_t = the t_max = inf closest hit, +inf for a miss)."""
    n = len(closest_t)
    kind = np.arange(n) % 8
    frac = rng.random(n).astype(np.float32)
    finite = np.where(np.isfinite(closest_t), closest_t, np.float32(1e3)).astype(np.float32)
    t = np.empty(n, dtype=np.float32)
    t[kind == 0] = np.inf
    t[kind == 1] = (finite * frac)[kind == 1]
    t[kind == 2] = closest_t[kind == 2]
    t[kind == 3] = EPS
    t[kind == 4] = 0.0
    t[kind == 5] = -rng.random(int((kind == 5).sum())).astype(np.float32) - np.float32(1e-3)
    t[kind == 6] = np.nan
    t[kind == 7] = (finite * (np.float32(1.001) + frac))[kind == 7]
    return t


def mixed_rays(loaded, seed, n_each=2048, grid=(64, 48)):
    """Every family for one scene: camera grid, interior (normalised and not), axis-aligned / zero components, and rays
    starting on surfaces.  Returns (rays, closest t at t_max = inf from the oracle)."""
    rng = np.random.default_rng(seed)
    sc = loaded.scene
    cam = camera_rays(sc, *grid)
    base = np.concatenate([cam, interior_rays(sc, rng, n_each), interior_rays(sc, rng, n_each, normalised=False),
                           axis_rays(sc, rng, n_each)])
    t0 = oracle_query(loaded, base)["t"]
    surf = surface_rays(base, t0, rng)[:n_each]
    rays = np.concatenate([base, surf])
    return rays, oracle_query(loaded, rays)["t"]
