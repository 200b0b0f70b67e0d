"""Mesh simplification's contract on the oracle alone (oracle/oracle_simplify.py): a hand-made mesh with its simplified
arrays written out, the oracle against a plain per-triangle loop of the same rules, and properties of the simplified
meshes of an analytic sphere and a wall. The device kernels are held to the oracle by test_simplify_gpu.py."""
import numpy as np
import oracle_mesh
import oracle_parts
import oracle_simplify
import pytest

BMIN, BMAX = (-1.0, 0.0, -1.0), (1.0, 2.0, 1.0)


def _loop(keys, res, positions, triangles, c):
    """The rules one triangle and one vertex at a time, with Python floats (binary64) for the sums."""
    X, Y, Z = res
    CX, CY = -(-X // c), -(-Y // c)

    def cluster(key):
        lin = int(key) // 3
        x, y, z = lin % X, (lin // X) % Y, lin // (X * Y)
        return ((z // c) * CY + y // c) * CX + x // c
    cid = [cluster(k) for k in keys]
    sums, count = {}, {}
    for i in range(len(keys)):                                 # ascending edge key
        s = sums.setdefault(cid[i], [0.0, 0.0, 0.0])
        for k in range(3):
            s[k] = s[k] + float(positions[i][k])
        count[cid[i]] = count.get(cid[i], 0) + 1
    seen, kept = set(), []
    for t, (i, j, k) in enumerate(triangles):
        a, b, cc = cid[i], cid[j], cid[k]
        if a == b or b == cc or a == cc:
            continue
        while a != min(a, b, cc):
            a, b, cc = b, cc, a
        if (a, b, cc) in seen:
            continue
        seen.add((a, b, cc))
        kept.append(((a, b, cc), t))
    used = sorted({x for trip, _ in kept for x in trip})
    index = {u: n for n, u in enumerate(used)}
    pos = np.array([[np.float32(sums[u][k] / count[u]) for k in range(3)] for u in used], np.float32).reshape(-1, 3)
    tri = np.array([[index[x] for x in trip] for trip, _ in kept], np.uint32).reshape(-1, 3)
    return pos, tri, np.array([t for _, t in kept], np.uint32)


def _same(got, want):
    for g, w, n in zip(got, want, ("positions", "triangles", "sources")):
        assert g.shape == w.shape and g.dtype == w.dtype, n
        assert np.array_equal(g.view(np.uint32), w.view(np.uint32)), n


def test_hand_made_mesh():
    # a 4 x 2 x 1 grid (X, Y, Z), clusters of 2 voxels: corners x = 0, 1 -> cluster 0, x = 2, 3 -> cluster 1 (CX = 2, CY = 1)
    res = (4, 2, 1)
    keys = np.array([0 * 3, 1 * 3 + 1, 2 * 3, 3 * 3 + 1, 5 * 3, 6 * 3 + 2, 7 * 3], np.uint64)   # lower corners 0, 1, 2, 3, 5, 6, 7
    pos = np.array([[0.0, 0, 0], [1.0, 0, 0], [2.0, 0, 0], [3.0, 0, 0], [1.0, 1, 0], [2.0, 1, 0], [3.0, 1, 0]], np.float32)
    # clusters:        0            0            1            1            0            1            1
    tri = np.array([[0, 1, 4],      # (0, 0, 0): dropped
                    [1, 2, 5],      # (0, 1, 1): dropped
                    [2, 3, 6]],     # (1, 1, 1): dropped
                   np.uint32)
    got = oracle_simplify.simplify_arrays(keys, res, pos, tri, 2)
    assert got[0].shape == (0, 3) and got[1].shape == (0, 3) and got[2].shape == (0,)
    # a 6 x 1 x 1 grid, clusters of 2: three clusters along x
    res = (6, 1, 1)
    keys = np.array([0, 3, 6, 9 + 1, 12, 15 + 2], np.uint64)   # corners 0 .. 5; cluster = corner // 2
    pos = np.array([[0.5, 0.25, 0], [1.0, 0.75, 0], [2.0, 0, 1], [3.0, 0, 1], [4.0, 2, 0], [5.0, 2, 2]], np.float32)
    tri = np.array([[0, 2, 4],      # (0, 1, 2): kept, source 0
                    [3, 5, 1],      # (1, 2, 0) -> rotated (0, 1, 2): duplicate of source 0
                    [4, 2, 0],      # (2, 1, 0) -> (0, 2, 1): opposite orientation, kept
                    [0, 1, 2],      # (0, 0, 1): degenerate
                    [5, 0, 3]],     # (2, 0, 1) -> (0, 1, 2): duplicate
                   np.uint32)
    p, t, s = oracle_simplify.simplify_arrays(keys, res, pos, tri, 2)
    assert np.array_equal(s, [0, 2])
    assert np.array_equal(t, [[0, 1, 2], [0, 2, 1]])
    assert np.array_equal(p, np.array([[0.75, 0.5, 0.0], [2.5, 0.0, 1.0], [4.5, 2.0, 1.0]], np.float32))
    _same((p, t, s), _loop(keys, res, pos, tri, 2))


def test_mean_is_the_rounded_binary64_sum_in_key_order():
    # three members whose binary32 sum would round differently: 1, 2^-24, 2^-24 (binary64 keeps both small terms)
    res = (2, 1, 1)
    keys = np.array([0, 1, 2], np.uint64)                      # one corner, three axes: one cluster for c = 1
    pos = np.array([[1.0, 0, 0], [2.0 ** -24, 0, 0], [2.0 ** -24, 0, 0]], np.float32)
    keys2 = np.array([3, 4, 5], np.uint64)                     # corner 1: a second cluster
    keys, pos = np.r_[keys, keys2], np.r_[pos, np.array([[5, 0, 0], [6, 0, 0], [7, 0, 0]], np.float32)]
    tri = np.array([[0, 3, 4], [1, 4, 5], [2, 3, 5]], np.uint32)
    # clusters (0, 1, 1) for every triangle: all degenerate, no output; with a third cluster the first survives
    assert len(oracle_simplify.simplify_arrays(keys, res, pos, tri, 1)[1]) == 0
    res = (3, 1, 1)
    keys = np.r_[keys, np.array([6], np.uint64)]
    pos = np.r_[pos, np.array([[9, 9, 9]], np.float32)]
    tri = np.array([[0, 3, 6]], np.uint32)
    p, _, _ = oracle_simplify.simplify_arrays(keys, res, pos, tri, 1)
    want = np.float32((1.0 + 2.0 ** -24 + 2.0 ** -24) / 3.0)
    assert p[0, 0] == want and np.float32(np.float32(np.float32(1.0) + np.float32(2.0 ** -24)) + np.float32(2.0 ** -24)) / 3 != want
    _same((p,) + oracle_simplify.simplify_arrays(keys, res, pos, tri, 1)[1:], _loop(keys, res, pos, tri, 1))


def _random_mesh(seed):
    rng = np.random.default_rng(seed)
    shape = tuple(int(s) for s in rng.integers(5, 16, 3))
    t = rng.normal(-0.1, 1.0, shape).astype(np.float32)
    Z, Y, X = shape
    pos, _, _, tri = oracle_mesh.extract_mesh(t, (X, Y, Z), 0.01, None, None, None, BMIN, BMAX)
    keys, _ = oracle_parts.mesh_edges(t)
    return t, (X, Y, Z), keys, pos, tri


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("c", [1, 2, 3, 5])
def test_oracle_equals_a_plain_loop(seed, c):
    t, res, keys, pos, tri = _random_mesh(seed)
    assert len(keys) == len(pos) > 0 and len(tri) > 0
    got = oracle_simplify.simplify_arrays(keys, res, pos, tri, c)
    _same(got, _loop(keys, res, pos, tri, c))
    assert len(got[1]) > 0
    # simplify_mesh finds the same keys from the volume
    full = oracle_simplify.simplify_mesh(t, pos, tri, c, 0.01, BMIN, BMAX)
    _same((full[0], full[3], full[4]), got)


def _sphere(n=40, r=13.0):
    z, y, x = np.mgrid[0:n, 0:n, 0:n].astype(np.float32)
    return (r - np.sqrt((x - 19.3) ** 2 + (y - 20.1) ** 2 + (z - 18.7) ** 2)).astype(np.float32)


def _wall(n=40):
    z, y, x = np.mgrid[0:n, 0:n, 0:24].astype(np.float32)
    return (np.minimum(z - 10.4, 17.6 - z) + 0.3 * np.sin(x * 0.7) * np.cos(y * 0.3)).astype(np.float32)


@pytest.mark.parametrize("shape", ["sphere", "wall"])
@pytest.mark.parametrize("c", [1, 2, 3, 4, 8])
def test_properties(shape, c):
    t = _sphere() if shape == "sphere" else _wall()
    Z, Y, X = t.shape
    res = (X, Y, Z)
    pos, _, _, tri = oracle_mesh.extract_mesh(t, res, 0.01, None, None, None, BMIN, BMAX)
    keys, _ = oracle_parts.mesh_edges(t)
    p, nt, src = oracle_simplify.simplify_arrays(keys, res, pos, tri, c)
    assert len(nt) > 0
    # no degenerate or duplicate triangles, every vertex used, smallest index first
    assert ((nt[:, 0] != nt[:, 1]) & (nt[:, 1] != nt[:, 2]) & (nt[:, 0] != nt[:, 2])).all()
    assert len(np.unique(nt, axis=0)) == len(nt)
    assert ((nt[:, 0] < nt[:, 1]) & (nt[:, 0] < nt[:, 2])).all()
    assert np.array_equal(np.unique(nt), np.arange(len(p)))
    # sources ascending; each maps to its output triangle: the clusters of its corners, rotated
    assert (np.diff(src.astype(np.int64)) > 0).all()
    cid = oracle_simplify.clusters(keys, res, c)
    used = np.unique(cid[tri[src]].ravel())
    for k in range(len(src)):
        trip = list(cid[tri[src[k]]])
        r = int(np.argmin(trip))
        assert list(used[nt[k]]) == trip[r:] + trip[:r]
    # each position inside the box of its cluster's members
    for v, u in enumerate(used):
        m = pos[cid == u]
        assert (m.min(axis=0) <= p[v]).all() and (p[v] <= m.max(axis=0)).all()
    # fewer vertices and triangles than the mesh
    assert len(p) <= len(pos) and len(nt) <= len(tri)
    if c >= 2:
        assert len(p) < len(pos) and len(nt) < len(tri)


def test_one_cluster_gives_no_triangles():
    t = _sphere()
    Z, Y, X = t.shape
    pos, _, _, tri = oracle_mesh.extract_mesh(t, (X, Y, Z), 0.01, None, None, None, BMIN, BMAX)
    keys, _ = oracle_parts.mesh_edges(t)
    for c in (max(X, Y, Z), max(X, Y, Z) + 7, 2 ** 31):
        p, nt, src = oracle_simplify.simplify_arrays(keys, (X, Y, Z), pos, tri, c)
        assert p.shape == (0, 3) and nt.shape == (0, 3) and src.shape == (0,)


@pytest.mark.parametrize("shape", ["sphere", "wall"])
def test_cluster_of_one_voxel_merges_only_shared_lower_corners(shape):
    t = _sphere() if shape == "sphere" else _wall()
    Z, Y, X = t.shape
    pos, _, _, tri = oracle_mesh.extract_mesh(t, (X, Y, Z), 0.01, None, None, None, BMIN, BMAX)
    keys, _ = oracle_parts.mesh_edges(t)
    cid = oracle_simplify.clusters(keys, (X, Y, Z), 1)
    assert np.array_equal(cid, keys.astype(np.int64) // 3)     # the cluster is the lower corner
    p, nt, src = oracle_simplify.simplify_arrays(keys, (X, Y, Z), pos, tri, 1)
    # a triangle survives unless two of its vertices share a lower corner; a kept triangle's vertex is its cluster's mean
    corner = keys.astype(np.int64) // 3
    ct = corner[tri]
    survives = (ct[:, 0] != ct[:, 1]) & (ct[:, 1] != ct[:, 2]) & (ct[:, 0] != ct[:, 2])
    assert len(src) <= survives.sum() and set(src.tolist()) <= set(np.flatnonzero(survives).tolist())
    single = np.bincount(np.searchsorted(np.unique(corner), corner)) == 1
    lone = np.unique(corner)[single]
    used = np.unique(corner[tri[src]].ravel())
    at = np.searchsorted(used, lone[np.isin(lone, used)])
    assert np.array_equal(p[at], pos[np.isin(corner, lone[np.isin(lone, used)])])
