"""ORACLE binding (test infrastructure, NOT product code): the scalar restatement of the volume queries.

ctypes wrapper over ro_query.cpp in oracle/librr_oracle.so (oracle_py.lib()). Import this only from tests/.
"""
from __future__ import annotations

import numpy as np

import oracle_py

WORLD, VOLUME = 0, 1


def sample_points(tsdf, res, limit, bbox_min, bbox_max, points, space=WORLD, inv=None, scene=None, pre=None):
    """rr_sample_points: (values [n], normals [n, 3], rgba [n, 4])."""
    v = oracle_py.VolumeArgs(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max)
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
    n = len(pts)
    val, nrm, rgba = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 4), np.float32)
    oracle_py.lib().ro_sample_points(*v.args, int(space), pts, n, val, nrm, rgba)
    return val, nrm, rgba


def cast_rays(tsdf, res, limit, bbox_min, bbox_max, origins, directions, space=WORLD, skip_space=False, occupied=None,
              brick_res=(1, 1, 1), brick_size=0.0, inv=None, scene=None, pre=None):
    """rr_cast_rays: (positions [n, 3], normals [n, 3], rgba [n, 4], steps uint32 [n]). skip_space marches over the hull of
    the occupied bricks (the ordered list of rr_download_bricks)."""
    v = oracle_py.VolumeArgs(tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max)
    o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(directions, np.float32).reshape(-1, 3)
    assert o.shape == d.shape
    n = len(o)
    occ = np.ascontiguousarray(occupied if occupied is not None else np.zeros(0), np.uint32)
    pos, nrm, rgba = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 4), np.float32)
    steps = np.zeros(n, np.uint32)
    oracle_py.lib().ro_cast_rays(*v.args, int(bool(skip_space)), occ.ctypes.data if len(occ) else None, len(occ),
                                 np.ascontiguousarray(brick_res, np.uint32), np.float32(brick_size), int(space), o, d, n, pos, nrm, rgba, steps)
    return pos, nrm, rgba, steps
