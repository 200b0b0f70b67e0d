"""ORACLE (test infrastructure, NOT product code): the connected parts of the fused volume, restated with numpy and
scipy.ndimage.label (an independent labelling implementation). Import this only from tests/.

label_parts   6-connected parts of the inside voxels (v > 0, finite), numbered by ascending key (the smallest linear
              index z*X*Y + y*X + x of the part), with voxel counts, half-open boxes and centroids;
mesh_edges    the mesh's vertices as crossed edges, by edge key, with the linear index of each edge's inside end;
mesh_parts    the part of every vertex and triangle of a mesh from the labels.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

OUTSIDE = np.uint32(0xFFFFFFFF)


def inside(tsdf):
    t = np.asarray(tsdf, np.float32)
    with np.errstate(invalid="ignore"):
        return np.isfinite(t) & (t > 0)


def centroids(sums, counts, res, bbox_min, bbox_max):
    """c_k = (float)(bmin_k + ((S_k / n) + 0.5) / R_k * (bmax_k - bmin_k)) in binary64, operands widened from float32 / int."""
    bmin = np.asarray(bbox_min, np.float32).astype(np.float64)
    bmax = np.asarray(bbox_max, np.float32).astype(np.float64)
    R = np.asarray(res, np.float64)
    S = np.asarray(sums, np.int64).astype(np.float64)          # exact: every sum is below 2^53
    n = np.asarray(counts, np.float64)[:, None]
    return (bmin + ((S / n) + 0.5) / R * (bmax - bmin)).astype(np.float32)


def label_parts(tsdf, bbox_min, bbox_max):
    """tsdf float32 [Z][Y][X] -> (labels uint32 [Z][Y][X] (0xFFFFFFFF outside), voxels uint32 [P], boxes int32 [P][6] =
    x0, x1, y0, y1, z0, z1 half-open, centroids float32 [P][3] in metres)."""
    tsdf = np.asarray(tsdf, np.float32)
    Z, Y, X = tsdf.shape
    lab, n = ndimage.label(inside(tsdf), structure=ndimage.generate_binary_structure(3, 1))
    flat = lab.ravel()
    idx = np.flatnonzero(flat)                                 # inside voxels in ascending linear index
    labels = np.full(flat.shape, OUTSIDE, np.uint32)
    if n == 0:
        return labels.reshape(Z, Y, X), np.zeros(0, np.uint32), np.zeros((0, 6), np.int32), np.zeros((0, 3), np.float32)
    _, first = np.unique(flat[idx], return_index=True)         # scipy label l = 1..n: its first voxel in index order
    rank = np.empty(n + 1, np.int64)
    rank[1:] = np.argsort(np.argsort(idx[first], kind="stable"), kind="stable")   # part number = rank of the key
    part = rank[flat[idx]]
    labels[idx] = part.astype(np.uint32)
    order = np.argsort(part, kind="stable")
    p_sorted, v_sorted = part[order], idx[order]
    starts = np.flatnonzero(np.r_[True, p_sorted[1:] != p_sorted[:-1]])
    x, y, z = v_sorted % X, (v_sorted // X) % Y, v_sorted // (X * Y)
    counts = np.diff(np.r_[starts, len(v_sorted)])
    boxes = np.stack([np.minimum.reduceat(x, starts), np.maximum.reduceat(x, starts) + 1,
                      np.minimum.reduceat(y, starts), np.maximum.reduceat(y, starts) + 1,
                      np.minimum.reduceat(z, starts), np.maximum.reduceat(z, starts) + 1], axis=1).astype(np.int32)
    sums = np.stack([np.add.reduceat(a.astype(np.int64), starts) for a in (x, y, z)], axis=1)
    return labels.reshape(Z, Y, X), counts.astype(np.uint32), boxes, centroids(sums, counts, (X, Y, Z), bbox_min, bbox_max)


def mesh_edges(tsdf):
    """The mesh's vertices under the header's vertex rule - edges with one end > 0, both ends finite, on at least one cell
    whose eight corners are finite - in edge-key order (key = linear index of the lower end * 3 + axis). Returns (keys
    uint64 [V], linear index of each edge's inside end int64 [V])."""
    t = np.asarray(tsdf, np.float32)
    Z, Y, X = t.shape
    fin = np.isfinite(t)
    pos = inside(t)
    cell = np.zeros((Z + 1, Y + 1, X + 1), bool)               # cell (x, y, z) at [z + 1, y + 1, x + 1]; False off the grid
    if X > 1 and Y > 1 and Z > 1:
        c = np.ones((Z - 1, Y - 1, X - 1), bool)
        for dz in (0, 1):
            for dy in (0, 1):
                for dx in (0, 1):
                    c &= fin[dz:Z - 1 + dz, dy:Y - 1 + dy, dx:X - 1 + dx]
        cell[1:Z, 1:Y, 1:X] = c
    keys, ends = [], []
    lin = np.arange(X * Y * Z, dtype=np.int64).reshape(Z, Y, X)
    for k in range(3):
        sl_a = [slice(None)] * 3
        sl_b = [slice(None)] * 3
        sl_a[2 - k] = slice(0, t.shape[2 - k] - 1)
        sl_b[2 - k] = slice(1, None)
        a, b = tuple(sl_a), tuple(sl_b)
        crossed = fin[a] & fin[b] & (pos[a] != pos[b])
        zz, yy, xx = np.nonzero(crossed)
        # the up to four cells around the edge: one step back (or not) along each of the two other axes
        near = np.zeros(len(xx), bool)
        for du in (0, 1):
            for dw in (0, 1):
                cx = xx - (du if k != 0 else 0)
                cy = yy - (du if k == 0 else (dw if k == 2 else 0))
                cz = zz - (dw if k != 2 else 0)
                near |= cell[cz + 1, cy + 1, cx + 1]
        zz, yy, xx = zz[near], yy[near], xx[near]
        la = lin[zz, yy, xx]
        lb = la + (1, X, X * Y)[k]
        keys.append(la.astype(np.uint64) * 3 + k)
        ends.append(np.where(pos[zz, yy, xx], la, lb))
    keys, ends = np.concatenate(keys), np.concatenate(ends)
    order = np.argsort(keys, kind="stable")
    return keys[order], ends[order]


def mesh_parts(labels, tsdf, triangles):
    """(vertex_parts uint32 [V], triangle_parts uint32 [T]) of the mesh of tsdf: a vertex's part is its inside end's label,
    a triangle's the part of its first vertex."""
    _, ends = mesh_edges(tsdf)
    vp = np.asarray(labels, np.uint32).ravel()[ends]
    tri = np.asarray(triangles, np.int64).reshape(-1, 3)
    return vp, vp[tri[:, 0]] if len(tri) else np.zeros(0, np.uint32)
