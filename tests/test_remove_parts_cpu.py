"""Removing connected parts (rr_remove_parts) on the oracle alone (oracle/oracle_remove.py): hand-made volumes with their
expected arrays written out, and the mesh of a removed volume against the --min-part-voxels filter of the mesh before the
removal. The device is held to the oracle bit for bit by test_remove_parts_gpu.py."""
import numpy as np
import oracle_mesh
import oracle_parts
import oracle_remove
import pytest

from conftest import bits_equal

L = np.float32(0.01)
O = np.float32(-0.01)      # outside


def _vol(shape, inside):
    t = np.full(shape, O, np.float32)
    for (x, y, z), v in inside.items():
        t[z, y, x] = v
    return t


def test_cleared_voxel_per_format():
    bits, t, w = oracle_remove.cleared_voxel(oracle_remove.VOXELS_F32, L)
    assert bits == np.float32(-L).view(np.uint32) and t == -L and w == 0
    bits, t, w = oracle_remove.cleared_voxel(oracle_remove.VOXELS_F32_WEIGHT, L)
    assert t == -L and w == 0
    bits, t, w = oracle_remove.cleared_voxel(oracle_remove.VOXELS_HALF2, L)
    # __floats2half2_rn(-0.01, 0): low half = half(-0.01) = 0xA11F (round to nearest even), high half +0
    assert bits == 0x0000A11F and t == np.float32(np.float16(-0.01)) and w == 0


def test_parts_touching_at_an_edge_and_a_corner():
    # A: two voxels along x; B touches A only along an edge, C only at a corner: three parts
    a = {(1, 1, 1): 0.5, (2, 1, 1): 0.25}
    b = {(3, 2, 1): 0.125}
    c = {(3, 2, 2): 0.0625}      # touches B across a face: B and C are one part
    d = {(0, 0, 0): 1.0}         # touches A at a corner only
    t = _vol((4, 4, 4), {**a, **b, **c, **d})
    labels, voxels, _, _ = oracle_parts.label_parts(t, (0, 0, 0), (1, 1, 1))
    assert voxels.tolist() == [1, 2, 2]            # D (key 0), A (key 21), B+C (key 27)
    got, _, k, v = oracle_remove.remove_parts(t, L, min_voxels=2)
    want = t.copy()
    want[0, 0, 0] = -L                             # D goes, A and B+C stay
    assert (k, v) == (1, 1) and bits_equal(got, want).all()
    got, _, k, v = oracle_remove.remove_parts(t, L, keep=np.array([1, 0, 1], np.uint8))
    want = t.copy()
    want[1, 1, 1] = want[1, 1, 2] = -L             # A goes; D at its corner and B at its edge stay
    assert (k, v) == (1, 2) and bits_equal(got, want).all()
    got, _, k, v = oracle_remove.remove_parts(t, L, min_voxels=2, keep=np.array([1, 1, 0], bool))
    want = t.copy()
    want[0, 0, 0] = want[1, 2, 3] = want[2, 2, 3] = -L
    assert (k, v) == (2, 3) and bits_equal(got, want).all()


def test_non_finite_voxels_are_never_touched():
    t = _vol((3, 3, 5), {(1, 1, 1): 0.5, (2, 1, 1): 0.5, (4, 2, 2): 0.5})
    t[1, 1, 3] = np.inf                            # next to the first part: not inside, not removed
    t[1, 1, 0] = np.nan
    t[2, 2, 3] = -np.inf
    w = np.arange(t.size, dtype=np.float32).reshape(t.shape) + 1
    got, got_w, k, v = oracle_remove.remove_parts(t, L, oracle_remove.VOXELS_F32_WEIGHT, min_voxels=3, weight=w)
    want, want_w = t.copy(), w.copy()
    for x, y, z in ((1, 1, 1), (2, 1, 1), (4, 2, 2)):
        want[z, y, x] = -L
        want_w[z, y, x] = 0
    assert (k, v) == (2, 3)
    assert bits_equal(got, want).all() and bits_equal(got_w, want_w).all()
    assert np.isnan(got[1, 1, 0]) and got[1, 1, 3] == np.inf and got[2, 2, 3] == -np.inf


def test_nothing_to_remove():
    t = _vol((3, 3, 3), {(1, 1, 1): 0.5})
    got, _, k, v = oracle_remove.remove_parts(t, L)
    assert (k, v) == (0, 0) and bits_equal(got, t).all()
    got, _, k, v = oracle_remove.remove_parts(_vol((3, 3, 3), {}), L, min_voxels=5, keep=np.zeros(0, np.uint8))
    assert (k, v) == (0, 0)


def _filtered_mesh(mesh, tparts, voxels, n):
    """fusion_playback's --min-part-voxels N filter: the triangles of parts of at least n voxels and the vertices they use, in
    their original order, re-indexed."""
    pos, nrm, rgba, tri = mesh
    keep_t = voxels[tparts] >= n
    used = np.zeros(len(pos), bool)
    used[tri[keep_t].ravel()] = True
    index = np.cumsum(used) - 1
    return pos[used], None if nrm is None else nrm[used], None if rgba is None else rgba[used], index[tri[keep_t]].astype(np.uint32)


def _mesh_after_equals_filter(t, n, inv=None, scene=None, pre=None, bmin=(0, 0, 0), bmax=(1, 1, 1)):
    res = (t.shape[2], t.shape[1], t.shape[0])
    labels, voxels, _, _ = oracle_parts.label_parts(t, bmin, bmax)
    before = oracle_mesh.extract_mesh(t, res, L, inv, scene, pre, bmin, bmax)
    _, tparts = oracle_parts.mesh_parts(labels, t, before[3])
    want = _filtered_mesh(before, tparts, voxels, n)
    removed, _, k, _ = oracle_remove.remove_parts(t, L, min_voxels=n, labels=labels, voxels=voxels)
    got = oracle_mesh.extract_mesh(removed, res, L, inv, scene, pre, bmin, bmax)
    assert bits_equal(got[0], want[0]).all(), "vertex positions"
    assert np.array_equal(got[3], want[3]), "triangles"
    if inv is not None:
        assert bits_equal(got[2], want[2]).all(), "colours"
    return k, len(want[3]), len(before[3])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_mesh_of_removed_volume_equals_filtered_mesh(seed):
    """Random blobs of every size, many of them touching at edges and corners: the removed voxels were inside, so none is the
    outside end of a kept part's crossed edge, and the face rule keeps each group's loop of a cell independent."""
    rng = np.random.default_rng(seed)
    t = np.where(rng.random((24, 20, 28)) < 0.3, rng.uniform(0.001, 0.01, (24, 20, 28)), rng.uniform(-0.01, -0.001, (24, 20, 28)))
    t = t.astype(np.float32)
    k, kept, total = _mesh_after_equals_filter(t, 4)
    assert k > 10 and 0 < kept < total


def test_mesh_colours_of_removed_scene_equal_filtered_mesh():
    """The oracle's own pre-process and integrate of a small scene, with floaters written in front of the surface: positions,
    triangles and colours of the kept parts are those of the mesh before the removal."""
    import oracle_py as O
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    inv = synth.analytic_inverse(sc, (40, 44, 40))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.02, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    t = O.integrate(inv, pre, grid, L, True, O.occupied_bricks(pre["bricks"], 10)).copy()
    rng = np.random.default_rng(4)
    Z, Y, X = t.shape
    for _ in range(12):                            # 1- to 8-voxel floaters
        z, y, x = rng.integers(2, Z - 4), rng.integers(2, Y - 4), rng.integers(2, X - 4)
        s = rng.integers(1, 3, 3)
        t[z:z + s[0], y:y + s[1], x:x + s[2]] = np.float32(0.005)
    k, kept, total = _mesh_after_equals_filter(t, 9, inv, sc, pre, sc.bbox_min, sc.bbox_max)
    assert k >= 5 and kept < total
