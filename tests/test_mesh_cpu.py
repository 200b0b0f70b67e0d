"""The surface extraction's contract on the oracle alone (oracle/ro_mesh.cpp): the generated case table, watertightness on
random fields, analytic shapes and NaN handling. The device kernels are held to the oracle bit for bit by test_mesh_gpu.py."""
import os
import re

import numpy as np
import oracle_mesh
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _corner(c):
    return np.array([c & 1, (c >> 1) & 1, (c >> 2) & 1])


def _edge_corners(e):
    axis, bits = e // 4, e % 4
    other = [a for a in range(3) if a != axis]
    lo = ((bits & 1) << other[0]) | (((bits >> 1) & 1) << other[1])
    return lo, lo | (1 << axis)


def _faces():
    """Per face: (axis, side, its four edges)."""
    out = []
    for axis in range(3):
        for side in range(2):
            edges = [e for e in range(12) if all(_corner(c)[axis] == side for c in _edge_corners(e))]
            out.append((axis, side, edges))
    return out


@pytest.fixture(scope="module")
def table():
    return oracle_mesh.mesh_case_table()


def test_case_table_rule(table):
    ntri, tri, most = table
    assert ntri[0] == 0 and ntri[255] == 0
    faces = _faces()
    by_face_pattern = {}
    for cs in range(256):
        inside = [(cs >> c) & 1 for c in range(8)]
        crossed = {e for e in range(12) if inside[_edge_corners(e)[0]] != inside[_edge_corners(e)[1]]}
        tris = tri[cs][: ntri[cs]]
        assert (tri[cs][ntri[cs]:] == -1).all()
        # directed boundary edges of the fans = the loops; every crossed edge is on exactly one loop, no other edge is used
        directed = {}
        for a, b, c in tris:
            for u, v in ((a, b), (b, c), (c, a)):
                directed[(u, v)] = directed.get((u, v), 0) + 1
        boundary = [(u, v) for (u, v), k in directed.items() if directed.get((v, u), 0) == 0]
        used = {e for t in tris for e in t}
        assert used == crossed, cs
        succ = {}
        for u, v in boundary:
            assert u not in succ, cs
            succ[u] = v
        assert set(succ) == crossed and set(succ.values()) == crossed, f"case {cs}: loops not closed"
        # each face's segments (boundary edges with both ends on the face) depend on the face's four signs alone
        for axis, side, edges in faces:
            corners = [c for c in range(8) if _corner(c)[axis] == side]
            key = (axis, side, tuple(inside[c] for c in corners))
            segs = frozenset((u, v) for u, v in boundary if u in edges and v in edges)
            assert by_face_pattern.setdefault(key, segs) == segs, f"case {cs}: face {axis}/{side} disagrees"
    # the kernels size their constant table for this many triangles per cell
    src = open(os.path.join(ROOT, "rgbd-recon_b200", "csrc", "rr_mesh.cu")).read()
    bound = int(re.search(r"constexpr int kMaxCellTris = (\d+);", src).group(1))
    assert most == ntri.max() and most <= bound


def _mesh(field, bmin=(0.0, 0.0, 0.0), bmax=(1.0, 1.0, 1.0)):
    Z, Y, X = field.shape
    pos, _, _, tri = oracle_mesh.extract_mesh(field.astype(np.float32), np.array([X, Y, Z], np.uint32), 0.01, None, None, None,
                                    np.array(bmin, np.float32), np.array(bmax, np.float32))
    return pos, tri


def _directed_edges(tri):
    e = np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]]).astype(np.int64)
    return e[:, 0] << 32 | e[:, 1], e[:, 1] << 32 | e[:, 0]


def _assert_watertight(tri, pos):
    """Every directed edge (i, j) is matched by as many (j, i): a crack or a flipped triangle breaks that. A directed edge
    occurs twice only where both cells on a face with four crossed edges fan across it between the same two vertices (a
    diagonal lying in the face, so its two ends share the face's coordinate); nowhere more often."""
    fwd, rev = _directed_edges(tri)
    u, k = np.unique(fwd, return_counts=True)
    ur, kr = np.unique(rev, return_counts=True)
    assert np.array_equal(u, ur) and np.array_equal(k, kr), "a directed edge has no opposite: the mesh has a crack or a flipped triangle"
    assert k.max() <= 2
    twice = u[k == 2]
    a, b = twice >> 32, twice & 0xffffffff
    assert (pos[a] == pos[b]).any(axis=1).all(), "a doubled edge that is not a diagonal in a cube face"
    assert len(np.unique(tri)) == len(pos), "unreferenced vertices"


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_watertight_on_random_fields(seed):
    rng = np.random.default_rng(seed)
    f = rng.uniform(-1.0, 1.0, (24, 25, 23)).astype(np.float32)
    f[0], f[-1], f[:, 0], f[:, -1], f[:, :, 0], f[:, :, -1] = -1, -1, -1, -1, -1, -1
    pos, tri = _mesh(f)
    assert len(tri) > 1000
    _assert_watertight(tri, pos)


def _grid(n):
    c = (np.arange(n, dtype=np.float64) + 0.5) / n
    return np.meshgrid(c, c, c, indexing="ij")     # z, y, x in texture coordinates


def _euler(pos, tri):
    fwd, _ = _directed_edges(tri)
    lo = np.minimum(fwd >> 32, fwd & 0xffffffff) << 32 | np.maximum(fwd >> 32, fwd & 0xffffffff)
    return len(pos) - len(np.unique(lo)) + len(tri)


def _face_normals(pos, tri):
    p = pos.astype(np.float64)
    return np.cross(p[tri[:, 1]] - p[tri[:, 0]], p[tri[:, 2]] - p[tri[:, 0]])


def test_sphere():
    n, r = 40, 0.3
    z, y, x = _grid(n)
    d = np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2 + (z - 0.5) ** 2)
    f = np.clip(r - d, -0.05, 0.05).astype(np.float32)           # TSDF, positive inside
    pos, nrm, _, tri = _with_normals(f)
    _assert_watertight(tri, pos)
    assert _euler(pos, tri) == 2
    h = 1.0 / n
    dist = np.abs(np.linalg.norm(pos.astype(np.float64) - 0.5, axis=1) - r)
    assert dist.max() <= h * h / r
    fn = _face_normals(pos, tri)
    centre = pos[tri].astype(np.float64).mean(axis=1) - 0.5
    assert ((fn * centre).sum(axis=1) > 0).all(), "a face normal points into the sphere"
    vn = np.zeros((len(pos), 3))
    for k in range(3):
        np.add.at(vn, tri[:, k], fn)
    vn /= np.linalg.norm(vn, axis=1, keepdims=True)
    assert ((vn * nrm).sum(axis=1) > 0.9).all(), "gradient normals disagree with the faces"


def _with_normals(f):
    """Extraction with the gradient normals, without sensors (no colour)."""
    from rrpy import synth
    Z, Y, X = f.shape
    sc = synth.make_scene(N=1, W=16, H=16, CW=16, CH=16, cv_res=(4, 4, 4), bbox=((0.0, 0.0, 0.0), (1.0, 1.0, 1.0)))
    inv = np.zeros((1, 4, 4, 4, 4), np.float32)
    pre = dict(depth_b=np.zeros((1, 16, 16, 2), np.float32), quality=np.zeros((1, 16, 16), np.float32))
    return oracle_mesh.extract_mesh(f, np.array([X, Y, Z], np.uint32), 0.01, inv, sc, pre, np.zeros(3, np.float32), np.ones(3, np.float32))


def test_torus():
    n, R, r = 48, 0.28, 0.1
    z, y, x = _grid(n)
    q = np.sqrt((x - 0.5) ** 2 + (z - 0.5) ** 2) - R
    f = np.clip(r - np.sqrt(q ** 2 + (y - 0.5) ** 2), -0.05, 0.05).astype(np.float32)
    pos, tri = _mesh(f)
    _assert_watertight(tri, pos)
    assert _euler(pos, tri) == 0


def test_nan_corners_emit_nothing():
    n, r = 32, 0.3
    z, y, x = _grid(n)
    f = np.clip(r - np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2 + (z - 0.5) ** 2), -0.05, 0.05).astype(np.float32)
    rng = np.random.default_rng(7)
    near = np.argwhere(np.abs(f) < 0.03)
    bad = near[rng.choice(len(near), 40, replace=False)]
    f[tuple(bad.T)] = np.nan
    pos, tri = _mesh(f)
    assert len(tri) > 100 and (tri < len(pos)).all()
    assert len(np.unique(tri)) == len(pos)
    assert np.isfinite(pos).all()
    # no triangle lies in a cell with a NaN corner: each triangle's cell is the floor of its centroid in voxel units
    cell = np.floor(pos[tri].astype(np.float64).mean(axis=1) * n - 0.5).astype(int)
    nanv = np.isnan(f)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                assert not nanv[cell[:, 2] + dz, cell[:, 1] + dy, cell[:, 0] + dx].any()
