"""The connected parts' contract on the oracle alone (oracle/oracle_parts.py): the mesh's case table keeps every triangle
within one face-connected group of inside corners, hand-made volumes, a plain breadth-first search on random fields, and
the numpy vertex enumeration against the mesh oracle. The device kernels are held to the oracle by test_parts_gpu.py."""
from collections import deque

import numpy as np
import oracle_mesh
import oracle_parts
import pytest

BMIN, BMAX = (-1.0, 0.0, -1.0), (1.0, 2.0, 1.0)


def _edge_ends(e):
    axis, bits = e // 4, e % 4
    other = [a for a in range(3) if a != axis]
    lo = ((bits & 1) << other[0]) | (((bits >> 1) & 1) << other[1])
    return lo, lo | (1 << axis)


def _corner_groups(cs):
    """Face-connected groups of the inside corners of case cs: corner -> group id."""
    group = {}
    for c in range(8):
        if not (cs >> c) & 1 or c in group:
            continue
        stack = [c]
        group[c] = c
        while stack:
            a = stack.pop()
            for k in range(3):
                b = a ^ (1 << k)
                if (cs >> b) & 1 and b not in group:
                    group[b] = c
                    stack.append(b)
    return group


def test_every_triangle_stays_in_one_corner_group():
    ntri, tri, _ = oracle_mesh.mesh_case_table()
    for cs in range(256):
        group = _corner_groups(cs)
        for t in range(ntri[cs]):
            ends = []
            for e in tri[cs, t]:
                a, b = _edge_ends(int(e))
                assert ((cs >> a) & 1) != ((cs >> b) & 1), f"case {cs}: edge {e} is not crossed"
                ends.append(a if (cs >> a) & 1 else b)
            assert len({group[c] for c in ends}) == 1, f"case {cs} triangle {t} spans two corner groups"


def _bfs(tsdf):
    """Plain-Python 6-connected labelling, keys and statistics (no scipy)."""
    Z, Y, X = tsdf.shape
    ins = oracle_parts.inside(tsdf)
    seen = np.zeros(ins.shape, bool)
    parts = []
    for z in range(Z):
        for y in range(Y):
            for x in range(X):
                if not ins[z, y, x] or seen[z, y, x]:
                    continue
                seen[z, y, x] = True
                q, vox = deque([(z, y, x)]), []
                while q:
                    c = q.popleft()
                    vox.append(c)
                    for d in ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)):
                        n = (c[0] + d[0], c[1] + d[1], c[2] + d[2])
                        if 0 <= n[0] < Z and 0 <= n[1] < Y and 0 <= n[2] < X and ins[n] and not seen[n]:
                            seen[n] = True
                            q.append(n)
                parts.append(vox)                      # found in raster order: ascending key
    labels = np.full(tsdf.shape, 0xFFFFFFFF, np.uint32)
    voxels, boxes, sums = [], [], []
    for p, vox in enumerate(parts):
        a = np.array(vox)
        labels[a[:, 0], a[:, 1], a[:, 2]] = p
        voxels.append(len(vox))
        boxes.append([a[:, 2].min(), a[:, 2].max() + 1, a[:, 1].min(), a[:, 1].max() + 1, a[:, 0].min(), a[:, 0].max() + 1])
        sums.append([int(a[:, 2].sum()), int(a[:, 1].sum()), int(a[:, 0].sum())])
    cen = np.array([[(np.float64(np.float32(BMIN[k])) + ((s[k] / n) + 0.5) / (X, Y, Z)[k]
                      * (np.float64(np.float32(BMAX[k])) - np.float64(np.float32(BMIN[k])))) for k in range(3)]
                    for s, n in zip(sums, voxels)], np.float64).astype(np.float32).reshape(-1, 3)
    return labels, np.array(voxels, np.uint32), np.array(boxes, np.int32).reshape(-1, 6), cen


def _same(got, want):
    for g, w, n in zip(got, want, ("labels", "voxels", "boxes", "centroids")):
        assert g.shape == w.shape and g.dtype == w.dtype, n
        if n == "centroids":
            assert np.array_equal(g.view(np.uint32), w.view(np.uint32)), n
        else:
            assert np.array_equal(g, w), n


def _field(shape, boxes):
    t = np.full(shape, -0.01, np.float32)
    for z0, z1, y0, y1, x0, x1 in boxes:
        t[z0:z1, y0:y1, x0:x1] = 0.01
    return t


@pytest.mark.parametrize("second, parts", [((2, 4, 2, 4, 4, 6), 1),     # shares a face with the first block
                                           ((4, 6, 4, 6, 2, 4), 2),     # along an edge only
                                           ((4, 6, 4, 6, 4, 6), 2)])    # at a corner only
def test_blocks_touching(second, parts):
    t = _field((8, 8, 8), [(2, 4, 2, 4, 2, 4), second])
    got = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(got[1]) == parts
    _same(got, _bfs(t))


def test_torus_is_one_part():
    z, y, x = np.mgrid[0:12, 0:20, 0:20].astype(np.float32)
    r = np.hypot(x - 9.5, y - 9.5)
    t = (2.5 - np.hypot(r - 6.0, z - 5.5)).astype(np.float32)
    got = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(got[1]) == 1 and got[0][5, 9, 3] == 0 and got[0][5, 9, 9] == 0xFFFFFFFF   # the hole is outside
    _same(got, _bfs(t))


def test_u_joined_high_in_z_has_the_lowest_voxel_as_key():
    # two arms standing on z = 1 .. 7 at x = 1 and x = 6, joined by a bridge at z = 7; the right arm goes lower (z = 0)
    t = _field((9, 4, 9), [(1, 8, 1, 3, 1, 2), (0, 8, 1, 3, 6, 7), (7, 8, 1, 3, 1, 7), (3, 4, 1, 2, 3, 4)])
    labels, voxels, boxes, _ = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(voxels) == 2
    assert labels[0, 1, 6] == 0 and labels[3, 1, 3] == 1                 # the U's key (z = 0) is lower than the blob's
    assert list(boxes[0]) == [1, 7, 1, 3, 0, 8]
    _same((labels, voxels, boxes, oracle_parts.label_parts(t, BMIN, BMAX)[3]), _bfs(t))


def test_parts_on_the_volume_border():
    t = _field((6, 5, 7), [(0, 1, 0, 5, 0, 7), (5, 6, 4, 5, 6, 7), (2, 4, 0, 1, 3, 4)])
    got = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(got[1]) == 3 and list(got[2][1]) == [3, 4, 0, 1, 2, 4] and list(got[2][2]) == [6, 7, 4, 5, 5, 6]
    _same(got, _bfs(t))


def test_non_finite_voxels_are_never_inside():
    t = _field((5, 5, 5), [(1, 4, 1, 4, 1, 4)])
    t[2, 2, 2] = np.nan                           # splits nothing: the ring around it stays connected
    t[2, 2, 1] = np.inf
    t[0, 0, 0] = np.inf
    t[4, 4, 4] = -np.inf
    labels, voxels, boxes, cen = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(voxels) == 1 and voxels[0] == 27 - 2
    assert labels[2, 2, 2] == labels[2, 2, 1] == labels[0, 0, 0] == 0xFFFFFFFF
    _same((labels, voxels, boxes, cen), _bfs(t))


def test_all_outside_volume_has_no_parts():
    t = np.full((4, 5, 6), -0.01, np.float32)
    t[1, 1, 1] = 0.0                              # v > 0 is inside, 0 is not
    labels, voxels, boxes, cen = oracle_parts.label_parts(t, BMIN, BMAX)
    assert (labels == 0xFFFFFFFF).all() and voxels.shape == (0,) and boxes.shape == (0, 6) and cen.shape == (0, 3)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_breadth_first_search(seed):
    rng = np.random.default_rng(seed)
    shape = tuple(int(s) for s in rng.integers(3, 12, 3))
    t = rng.normal(-0.3 + 0.1 * seed, 1.0, shape).astype(np.float32)
    t[rng.random(shape) < 0.03] = np.nan
    got = oracle_parts.label_parts(t, BMIN, BMAX)
    assert len(got[1]) > 1
    _same(got, _bfs(t))


@pytest.mark.parametrize("seed", range(6))
def test_mesh_vertices_and_triangles_get_one_part(seed):
    rng = np.random.default_rng(100 + seed)
    shape = tuple(int(s) for s in rng.integers(4, 14, 3))
    t = rng.normal(-0.2, 1.0, shape).astype(np.float32)
    t[rng.random(shape) < 0.02] = np.nan
    Z, Y, X = shape
    pos, _, _, tri = oracle_mesh.extract_mesh(t, (X, Y, Z), 0.01, None, None, None, BMIN, BMAX)
    keys, ends = oracle_parts.mesh_edges(t)
    assert len(keys) == len(pos) > 0 and len(tri) > 0
    assert oracle_parts.inside(t).ravel()[ends].all()
    labels = oracle_parts.label_parts(t, BMIN, BMAX)[0]
    vp, tp = oracle_parts.mesh_parts(labels, t, tri)
    assert (vp != 0xFFFFFFFF).all()
    assert (vp[tri[:, 0]] == vp[tri[:, 1]]).all() and (vp[tri[:, 0]] == vp[tri[:, 2]]).all()
    assert np.array_equal(tp, vp[tri[:, 0]])
