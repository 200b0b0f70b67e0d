"""ORACLE binding (test infrastructure, NOT product code): the scalar restatement of the surface extraction.

ctypes wrapper over oracle/librr_oracle_mesh.so (ro_mesh.cpp, built by mesh.mk). Import this only from tests/.
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


def build(force=False):
    so = os.path.join(_HERE, "librr_oracle_mesh.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-f", "mesh.mk", "librr_oracle_mesh.so"])
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(build())
    L.ro_mesh_case_table.argtypes = [i32p, i32p]
    L.ro_mesh_case_table.restype = C.c_int
    L.ro_extract_mesh.argtypes = [f32p, u32p, C.c_float, C.c_int, C.c_void_p, i32p, C.c_void_p, i32p, C.c_void_p, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_int, C.c_int, f32p, f32p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
    L.ro_extract_mesh.restype = None
    _LIB = L
    return L


def mesh_case_table():
    """The case table of the surface extraction: (ntri int32[256], tri int32[256][10][3] of cube edges, -1 past ntri), and the
    most triangles any case needs."""
    ntri = np.zeros(256, np.int32)
    tri = np.zeros((256, 10, 3), np.int32)
    most = lib().ro_mesh_case_table(ntri, tri.reshape(-1))
    assert most >= 0, "inconsistent face rule"
    return ntri, tri, most


def extract_mesh(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max):
    """Marching cubes as rr_extract_mesh: tsdf float32 [Z][Y][X] (res = (X, Y, Z)). inv / scene / pre may be None for the
    geometry alone (normals and colours then come back as None). Returns (positions [V,3], normals [V,3], rgba [V,4],
    triangles uint32 [T,3])."""
    L = lib()
    tsdf = np.ascontiguousarray(tsdf, np.float32)
    res = np.ascontiguousarray(res, np.uint32)
    bmin = np.ascontiguousarray(bbox_min, np.float32)
    bmax = np.ascontiguousarray(bbox_max, np.float32)
    attrs = inv is not None
    keep = []

    def ptr(a, dt):
        a = np.ascontiguousarray(a, dt)
        keep.append(a)
        return a.ctypes.data

    if attrs:
        N, IZ, IY, IX, _ = inv.shape
        X, Y, Z = scene.cv_res
        _, H, W = pre["quality"].shape
        args = (N, ptr(inv, np.float32), np.array([IX, IY, IZ], np.int32), ptr(scene.cv_uv, np.float32), np.array([X, Y, Z], np.int32),
                ptr(scene.color, np.uint8), scene.CW, scene.CH, ptr(pre["depth_b"], np.float32), ptr(pre["quality"], np.float32), W, H)
    else:
        z3 = np.zeros(3, np.int32)
        args = (0, None, z3, None, z3, None, 0, 0, None, None, 0, 0)
    counts = np.zeros(2, np.uint64)
    L.ro_extract_mesh(tsdf, res, np.float32(limit), *args, bmin, bmax, counts.ctypes.data, None, None, None, None)
    nv, nt = int(counts[0]), int(counts[1])
    pos = np.zeros((nv, 3), np.float32)
    nrm = np.zeros((nv, 3), np.float32) if attrs else None
    rgba = np.zeros((nv, 4), np.float32) if attrs else None
    tri = np.zeros((nt, 3), np.uint32)
    L.ro_extract_mesh(tsdf, res, np.float32(limit), *args, bmin, bmax, counts.ctypes.data, pos.ctypes.data,
                      nrm.ctypes.data if attrs else None, rgba.ctypes.data if attrs else None, tri.ctypes.data)
    return pos, nrm, rgba, tri
