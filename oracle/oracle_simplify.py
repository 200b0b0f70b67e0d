"""ORACLE (test infrastructure, NOT product code): mesh simplification by vertex clustering, restated with numpy,
independently of the device algorithm (no sorts of rank triples, no scans). Import this only from tests/.

clusters         the cluster id of every vertex from its edge key;
simplify_arrays  the geometry of the contract from edge keys, positions and triangles: mean positions, triangles, sources;
simplify_mesh    the whole contract for the mesh of a volume: edge keys from oracle_parts.mesh_edges, normals and colours
                 from oracle_query.sample_points (world space) at the mean positions.
"""
from __future__ import annotations

import numpy as np

import oracle_parts
import oracle_query


def clusters(keys, res, cluster_voxels):
    """Cluster id (z/c * CY + y/c) * CX + x/c of the lower corner (x, y, z) of each edge key (linear index * 3 + axis)."""
    X, Y, Z = (int(r) for r in res)
    c = int(cluster_voxels)
    CX, CY = -(-X // c), -(-Y // c)
    lin = np.asarray(keys, np.uint64).astype(np.int64) // 3
    x, y, z = lin % X, (lin // X) % Y, lin // (X * Y)
    return ((z // c) * CY + y // c) * CX + x // c


def simplify_arrays(keys, res, positions, triangles, cluster_voxels):
    """keys uint64 [V] in ascending order with the mesh's vertices (positions float32 [V, 3]), triangles [T, 3] ->
    (positions float32 [V', 3], triangles uint32 [T', 3], sources uint32 [T'])."""
    keys = np.asarray(keys, np.uint64)
    pos = np.asarray(positions, np.float32).reshape(-1, 3)
    tri = np.asarray(triangles, np.int64).reshape(-1, 3)
    assert len(keys) == len(pos) and (len(keys) < 2 or (np.diff(keys.astype(np.int64)) > 0).all())
    cid = clusters(keys, res, cluster_voxels)
    ids, member = np.unique(cid, return_inverse=True)          # every non-empty cluster, ascending id
    sums = np.zeros((len(ids), 3), np.float64)
    np.add.at(sums, member, pos.astype(np.float64))            # in index order = ascending edge key, from +0.0
    count = np.bincount(member, minlength=len(ids)).astype(np.float64)
    mean = (sums / count[:, None]).astype(np.float32)
    ct = cid[tri] if len(tri) else np.zeros((0, 3), np.int64)
    ok = (ct[:, 0] != ct[:, 1]) & (ct[:, 1] != ct[:, 2]) & (ct[:, 0] != ct[:, 2])
    src = np.flatnonzero(ok)
    ct = ct[ok]
    first = np.argmin(ct, axis=1)                              # rotate the smallest id to the front, keeping the cycle
    rot = np.stack([ct[np.arange(len(ct)), (first + k) % 3] for k in range(3)], axis=1) if len(ct) else ct
    if len(rot):
        _, at = np.unique(rot, axis=0, return_index=True)      # first occurrence = smallest source index
        at = np.sort(at)
    else:
        at = np.zeros(0, np.int64)
    rot, src = rot[at], src[at]
    used = np.unique(rot.ravel())                              # referenced clusters, ascending id
    new_tri = np.searchsorted(used, rot).astype(np.uint32).reshape(-1, 3)
    new_pos = mean[np.searchsorted(ids, used)].reshape(-1, 3)
    return new_pos, new_tri, src.astype(np.uint32)


def simplify_mesh(tsdf, positions, triangles, cluster_voxels, limit, bbox_min, bbox_max, inv=None, scene=None, pre=None):
    """rr_simplify_mesh of the mesh (positions, triangles) of tsdf float32 [Z][Y][X]: (positions [V', 3], normals [V', 3],
    rgba [V', 4], triangles uint32 [T', 3], sources uint32 [T']). inv / scene / pre as for oracle_query.sample_points;
    without them the normals and colours come back as None."""
    t = np.asarray(tsdf, np.float32)
    Z, Y, X = t.shape
    keys, _ = oracle_parts.mesh_edges(t)
    pos, tri, src = simplify_arrays(keys, (X, Y, Z), positions, triangles, cluster_voxels)
    if inv is None:
        return pos, None, None, tri, src
    _, nrm, rgba = oracle_query.sample_points(t, (X, Y, Z), limit, bbox_min, bbox_max, pos, oracle_query.WORLD, inv, scene, pre)
    return pos, nrm, rgba, tri, src
