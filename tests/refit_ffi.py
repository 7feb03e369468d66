"""Refit of a resident scene, for the tests: the CPU restatement (refit_oracle, tests/csrc/refit_oracle.c) and the
motions the tests apply.  TEST INFRASTRUCTURE ONLY.

Positions are (3, 3, n_slots) float32 arrays indexed [axis][vertex][slot] (driver.scene_positions), normals
(n_slots, 3, 3) float32 (driver.scene_normals).  Every motion is computed in float32 elementwise, so a vertex shared
by several slots moves to the same place in each of them.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

import oracle_ffi
from helpers import CSRC, ROOT
from raytracing_c_b200._ffi import Scene

_lib = None


def refit_lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = oracle_ffi.build_lib("librefit_oracle.so", [
            "-O2", "-std=gnu11", "-mavx2", "-mfma", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"),
            os.path.join(CSRC, "refit_oracle.c"), "-lm"])
        lib = C.CDLL(path)
        lib.refit_oracle.argtypes = [C.POINTER(Scene), C.c_void_p, C.c_void_p]
        lib.refit_oracle.restype = None
        _lib = lib
    return _lib


def oracle_refit(loaded, positions, normals=None) -> None:
    """Rewrites the host Scene of `loaded` in place as a refit to `positions` (and `normals`) leaves it."""
    positions = np.ascontiguousarray(positions, dtype=np.float32)
    normals = np.ascontiguousarray(normals, dtype=np.float32) if normals is not None else None
    refit_lib().refit_oracle(C.byref(loaded.scene), positions.ctypes.data,
                             normals.ctypes.data if normals is not None else None)


def rotation(angle_y, angle_x):
    cy, sy, cx, sx = np.cos(angle_y), np.sin(angle_y), np.cos(angle_x), np.sin(angle_x)
    ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    return (rx @ ry).astype(np.float32)


def rigid(positions, normals, rot, shift):
    """p' = R p + t and n' = R n, in float32 with the products summed left to right."""
    rot = np.asarray(rot, dtype=np.float32)
    shift = np.asarray(shift, dtype=np.float32)
    p = positions
    new_p = np.stack([rot[a, 0] * p[0] + rot[a, 1] * p[1] + rot[a, 2] * p[2] + shift[a] for a in range(3)])
    new_n = None
    if normals is not None:
        n = normals
        new_n = np.stack([rot[a, 0] * n[..., 0] + rot[a, 1] * n[..., 1] + rot[a, 2] * n[..., 2] for a in range(3)], axis=-1)
    return new_p.astype(np.float32), new_n


def deform(positions, amount=0.05, freq=3.0):
    """p += amount * sin(freq * p.yzx)."""
    p = positions.astype(np.float32)
    a, f = np.float32(amount), np.float32(freq)
    return np.stack([p[0] + a * np.sin(f * p[1]), p[1] + a * np.sin(f * p[2]), p[2] + a * np.sin(f * p[0])]).astype(np.float32)
