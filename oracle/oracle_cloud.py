"""ORACLE binding (test infrastructure, NOT product code): the scalar restatement of the point-cloud export.

ctypes wrapper over oracle/librr_oracle_cloud.so (ro_cloud.cpp, built by cloud.mk). Import this only from tests/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def build(force=False):
    so = os.path.join(_HERE, "librr_oracle_cloud.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-f", "cloud.mk", "librr_oracle_cloud.so"])
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(build())
    L.ro_extract_points.argtypes = [C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, u8p, C.c_int, C.c_int, f32p, f32p, i32p, f32p, f32p,
                                    C.c_uint32, C.POINTER(C.c_uint32), f32p, f32p, f32p, f32p, u32p]
    L.ro_extract_points.restype = None
    _LIB = L
    return L


def extract_points(depth_b, normal, quality, color, cv_xyz, cv_uv, bbox_min, bbox_max, sensor_mask=None):
    """rr_extract_points on the given images: depth_b [N, H, W, 2], normal [N, H, W, 3] (or the padded [.., 4]), quality
    [N, H, W], colour uint8 [N, CH, CW, 3], cv_xyz [N, Z, Y, X, 3], cv_uv [N, Z, Y, X, 2]. sensor_mask defaults to every
    sensor. Returns (positions [n, 3], normals [n, 3], colors [n, 3], quality [n], pixels uint32 [n])."""
    N, H, W = np.shape(quality)
    _, CH, CW, _ = np.shape(color)
    _, Z, Y, X, _ = np.shape(cv_xyz)
    mask = (1 << N) - 1 if sensor_mask is None else int(sensor_mask)
    n_max = N * W * H
    pos, nrm, rgb = (np.zeros((n_max, 3), np.float32) for _ in range(3))
    q, pix = np.zeros(n_max, np.float32), np.zeros(n_max, np.uint32)
    n = C.c_uint32()
    lib().ro_extract_points(N, W, H, np.ascontiguousarray(depth_b, np.float32), np.ascontiguousarray(np.asarray(normal)[..., :3], np.float32),
                            np.ascontiguousarray(quality, np.float32), np.ascontiguousarray(color, np.uint8), CW, CH,
                            np.ascontiguousarray(cv_xyz, np.float32), np.ascontiguousarray(cv_uv, np.float32), np.array([X, Y, Z], np.int32),
                            np.ascontiguousarray(bbox_min, np.float32), np.ascontiguousarray(bbox_max, np.float32), mask, C.byref(n),
                            pos, nrm, rgb, q, pix)
    k = n.value
    return pos[:k].copy(), nrm[:k].copy(), rgb[:k].copy(), q[:k].copy(), pix[:k].copy()


def extract_points_scene(scene, pre, sensor_mask=None, color=None):
    """extract_points on a synth.Scene and the stage images `pre` (oracle_py.preprocess, or downloaded stages)."""
    return extract_points(pre["depth_b"], pre["normal"], pre["quality"], scene.color if color is None else color, scene.cv_xyz,
                          scene.cv_uv, scene.bbox_min, scene.bbox_max, sensor_mask)
