"""ORACLE binding (test infrastructure, NOT product code): the scalar restatement of the volume queries.

ctypes wrapper over oracle/librr_oracle_query.so (ro_query.cpp, built by query.mk). Import this only from tests/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

WORLD, VOLUME = 0, 1

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")

_VOLUME_ARGS = [f32p, u32p, C.c_float, C.c_int, C.c_void_p, i32p, C.c_void_p, i32p, C.c_void_p, C.c_int, C.c_int,
                C.c_void_p, C.c_void_p, C.c_int, C.c_int, f32p, f32p]


def build(force=False):
    so = os.path.join(_HERE, "librr_oracle_query.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-f", "query.mk", "librr_oracle_query.so"])
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(build())
    L.ro_sample_points.argtypes = _VOLUME_ARGS + [C.c_int, f32p, C.c_uint32, f32p, f32p, f32p]
    L.ro_sample_points.restype = None
    L.ro_cast_rays.argtypes = _VOLUME_ARGS + [C.c_int, C.c_void_p, C.c_uint32, u32p, C.c_float, C.c_int, f32p, f32p, C.c_uint32,
                                              f32p, f32p, f32p, u32p]
    L.ro_cast_rays.restype = None
    _LIB = L
    return L


class _Volume:
    """The volume block every entry point takes: tsdf float32 [Z][Y][X] (res = (X, Y, Z)), and optionally the inverse volumes,
    scene (cv_uv, colour) and pre-processed stage images blendColors reads (all three or none)."""

    def __init__(self, tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max):
        self.keep = []
        tsdf = np.ascontiguousarray(tsdf, np.float32)
        bmin = np.ascontiguousarray(bbox_min, np.float32)
        bmax = np.ascontiguousarray(bbox_max, np.float32)
        head = (tsdf, np.ascontiguousarray(res, np.uint32), np.float32(limit))
        if inv is not None:
            N, IZ, IY, IX, _ = inv.shape
            X, Y, Z = scene.cv_res
            _, H, W = pre["quality"].shape
            self.args = head + (N, self._ptr(inv, np.float32), np.array([IX, IY, IZ], np.int32), self._ptr(scene.cv_uv, np.float32),
                                np.array([X, Y, Z], np.int32), self._ptr(scene.color, np.uint8), scene.CW, scene.CH,
                                self._ptr(pre["depth_b"], np.float32), self._ptr(pre["quality"], np.float32), W, H, bmin, bmax)
        else:
            z3 = np.zeros(3, np.int32)
            self.args = head + (0, None, z3, None, z3, None, 0, 0, None, None, 0, 0, bmin, bmax)

    def _ptr(self, a, dt):
        a = np.ascontiguousarray(a, dt)
        self.keep.append(a)
        return a.ctypes.data


def sample_points(tsdf, res, limit, bbox_min, bbox_max, points, space=WORLD, inv=None, scene=None, pre=None):
    """rr_sample_points: (values [n], normals [n, 3], rgba [n, 4])."""
    v = _Volume(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max)
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
    n = len(pts)
    val, nrm, rgba = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 4), np.float32)
    lib().ro_sample_points(*v.args, int(space), pts, n, val, nrm, rgba)
    return val, nrm, rgba


def cast_rays(tsdf, res, limit, bbox_min, bbox_max, origins, directions, space=WORLD, skip_space=False, occupied=None,
              brick_res=(1, 1, 1), brick_size=0.0, inv=None, scene=None, pre=None):
    """rr_cast_rays: (positions [n, 3], normals [n, 3], rgba [n, 4], steps uint32 [n]). skip_space marches over the hull of
    the occupied bricks (the ordered list of rr_download_bricks)."""
    v = _Volume(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max)
    o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(directions, np.float32).reshape(-1, 3)
    assert o.shape == d.shape
    n = len(o)
    occ = np.ascontiguousarray(occupied if occupied is not None else np.zeros(0), np.uint32)
    pos, nrm, rgba = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 4), np.float32)
    steps = np.zeros(n, np.uint32)
    lib().ro_cast_rays(*v.args, int(bool(skip_space)), occ.ctypes.data if len(occ) else None, len(occ),
                       np.ascontiguousarray(brick_res, np.uint32), np.float32(brick_size), int(space), o, d, n, pos, nrm, rgba, steps)
    return pos, nrm, rgba, steps
