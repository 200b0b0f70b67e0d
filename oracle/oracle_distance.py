"""ORACLE (test infrastructure, NOT product code): the distance field and distance queries of the fused volume. Import this
only from tests/.

nearest_voxels                 ro_distance.cpp: the sequential separable transform, O(N); compiled on first use into a
                               library of its own under the temporary directory (keyed by the source's hash), with
                               the oracle's compiler flags, so the tree is never written
nearest_bruteforce_separable   an independent numpy restatement: per pass the min-plus over the whole line, np.argmin's
                               first occurrence being the tie rule (small volumes only: O(N * longest axis) memory)
squared_distances              d^2 of every voxel to its nearest voxel, from the indices
sample_distance                the query formulas in float32 numpy, operation by operation (numpy fuses nothing)
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_parts
import oracle_py

NONE = np.uint32(0xFFFFFFFF)
WORLD, VOLUME = 0, 1


_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ro_distance.cpp")
_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-shared"]
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        key = hashlib.sha256(open(_SRC, "rb").read() + " ".join(_FLAGS).encode()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"rr_oracle_distance_{os.getuid()}_{key}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call(["/usr/bin/g++", *_FLAGS, "-o", tmp, _SRC])
            os.replace(tmp, path)                            # atomic: concurrent first uses agree on one file
        L = C.CDLL(path)
        L.ro_distance_field.argtypes = [oracle_py.u8p, C.c_int, C.c_int, C.c_int, oracle_py.u32p]
        _LIB = L
    return _LIB


def nearest_voxels(tsdf):
    """tsdf float32 [Z][Y][X] (the values the raymarch reads) -> nearest uint32 [Z][Y][X]."""
    inside = np.ascontiguousarray(oracle_parts.inside(tsdf), np.uint8)
    Z, Y, X = inside.shape
    out = np.empty((Z, Y, X), np.uint32)
    _lib().ro_distance_field(inside, X, Y, Z, out)
    return out


def nearest_bruteforce_separable(inside):
    """inside bool [Z][Y][X] -> nearest uint32 [Z][Y][X], one axis at a time: for every voxel the line's argmin of
    g(s) + (v - s)^2, g being the squared distance over the axes already done (inf: no candidate)."""
    inside = np.asarray(inside, bool)
    Z, Y, X = inside.shape
    lin = np.arange(X * Y * Z, dtype=np.int64).reshape(Z, Y, X)
    g = np.where(inside, 0.0, np.inf)
    idx = np.where(inside, lin, -1)
    for axis in (2, 1, 0):                                   # x, then y, then z
        gm, im = np.moveaxis(g, axis, -1), np.moveaxis(idx, axis, -1)
        n = gm.shape[-1]
        v = np.arange(n)
        cost = gm[..., None, :] + ((v[:, None] - v[None, :]) ** 2).astype(np.float64)   # [..., v, s]
        best = np.argmin(cost, axis=-1)                      # the first (smallest) s on ties
        g_new = np.take_along_axis(cost, best[..., None], -1)[..., 0]
        i_new = np.take_along_axis(im, best, -1)
        i_new = np.where(np.isfinite(g_new), i_new, -1)
        g, idx = np.moveaxis(g_new, -1, axis), np.moveaxis(i_new, -1, axis)
    return np.where(idx < 0, NONE, idx).astype(np.uint32)


def squared_distances(nearest):
    """int64 [Z][Y][X]: dx^2 + dy^2 + dz^2 from every voxel to its nearest voxel (-1 where there is none); slice by slice."""
    Z, Y, X = nearest.shape
    y, x = np.arange(Y)[:, None], np.arange(X)[None, :]
    out = np.empty((Z, Y, X), np.int64)
    for z in range(Z):
        f = nearest[z].astype(np.int64)
        d2 = (x - f % X) ** 2 + (y - (f // X) % Y) ** 2 + (z - f // (X * Y)) ** 2
        out[z] = np.where(nearest[z] == NONE, -1, d2)
    return out


def _near_coord(s, n):
    """floor(s * n) in binary32, clamped to [0, n - 1] (rr_math.cuh near_coord)."""
    return np.clip(np.floor(s * np.float32(n)), 0, n - 1).astype(np.int64)


def sample_distance(nearest, bbox_min, bbox_max, points, space=WORLD):
    """rr_sample_distance against the field `nearest`: (distances float32 [n], nearest_points float32 [n, 3], nearest_voxels
    uint32 [n])."""
    Z, Y, X = nearest.shape
    R = (X, Y, Z)
    bmin = np.asarray(bbox_min, np.float32)
    dims = (np.asarray(bbox_max, np.float32) - bmin).astype(np.float32)
    v = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
    n = len(v)
    with np.errstate(invalid="ignore", over="ignore"):
        q = (v - bmin) / dims if space == WORLD else v
        ok = np.all((q >= 0) & (q <= 1), axis=1)             # false for NaN
    dist = np.full(n, np.nan, np.float32)
    pts = np.full((n, 3), np.nan, np.float32)
    vox = np.full(n, NONE, np.uint32)
    if not ok.any():
        return dist, pts, vox
    qa = q[ok]
    a = (_near_coord(qa[:, 2], Z) * Y + _near_coord(qa[:, 1], Y)) * X + _near_coord(qa[:, 0], X)
    f = nearest.reshape(-1)[a]
    vox[ok] = f
    has = f != NONE
    d = np.full(len(f), np.inf, np.float32)
    c = np.full((len(f), 3), np.nan, np.float32)
    fi = f[has].astype(np.int64)
    fk = np.stack([fi % X, (fi // X) % Y, fi // (X * Y)], 1).astype(np.float32)
    cv = (fk + np.float32(0.5)) / np.asarray(R, np.float32)
    cw = bmin + cv * dims
    vin = v[ok][has]
    pw = vin if space == WORLD else bmin + vin * dims
    dd = pw - cw
    d[has] = np.sqrt((dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2])
    c[has] = cw if space == WORLD else cv
    dist[ok] = d
    pts[ok] = c
    return dist, pts, vox
