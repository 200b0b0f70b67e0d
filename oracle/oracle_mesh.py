"""ORACLE binding (test infrastructure, NOT product code): the scalar restatement of the surface extraction.

ctypes wrapper over ro_mesh.cpp in oracle/librr_oracle.so (oracle_py.lib()). Import this only from tests/.
"""
from __future__ import annotations

import numpy as np

import oracle_py


def mesh_case_table():
    """The case table of the surface extraction: (ntri int32[256], tri int32[256][10][3] of cube edges, -1 past ntri), and the
    most triangles any case needs."""
    ntri = np.zeros(256, np.int32)
    tri = np.zeros((256, 10, 3), np.int32)
    most = oracle_py.lib().ro_mesh_case_table(ntri, tri.reshape(-1))
    assert most >= 0, "inconsistent face rule"
    return ntri, tri, most


def extract_mesh(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max):
    """Marching cubes as rr_extract_mesh: tsdf float32 [Z][Y][X] (res = (X, Y, Z)). inv / scene / pre may be None for the
    geometry alone (normals and colours then come back as None). Returns (positions [V,3], normals [V,3], rgba [V,4],
    triangles uint32 [T,3])."""
    v = oracle_py.VolumeArgs(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max)
    attrs = inv is not None
    L = oracle_py.lib()
    counts = np.zeros(2, np.uint64)
    L.ro_extract_mesh(*v.args, counts.ctypes.data, None, None, None, None)
    nv, nt = int(counts[0]), int(counts[1])
    pos = np.zeros((nv, 3), np.float32)
    nrm = np.zeros((nv, 3), np.float32) if attrs else None
    rgba = np.zeros((nv, 4), np.float32) if attrs else None
    tri = np.zeros((nt, 3), np.uint32)
    L.ro_extract_mesh(*v.args, counts.ctypes.data, pos.ctypes.data,
                      nrm.ctypes.data if attrs else None, rgba.ctypes.data if attrs else None, tri.ctypes.data)
    return pos, nrm, rgba, tri
