"""The distance-field oracle (oracle/oracle_distance.py, oracle/ro_distance.cpp) without a GPU: the separable argmin
restatement against a brute force over every inside voxel on small volumes full of ties, the C++ transform against the
argmin restatement bit for bit, d^2 against scipy's Euclidean distance transform, and hand-worked queries."""
import numpy as np
import oracle_distance as D
import pytest
from scipy import ndimage

from conftest import bits_equal

NONE = D.NONE


def brute_force(inside):
    """For every voxel, the smallest linear index among the inside voxels at the least squared index distance."""
    Z, Y, X = inside.shape
    cand = np.flatnonzero(inside.reshape(-1))
    out = np.full(inside.size, NONE, np.uint32)
    if len(cand) == 0:
        return out.reshape(Z, Y, X)
    cz, cy, cx = cand // (X * Y), (cand // X) % Y, cand % X
    for i in range(inside.size):
        z, y, x = i // (X * Y), (i // X) % Y, i % X
        d2 = (cx - x) ** 2 + (cy - y) ** 2 + (cz - z) ** 2
        out[i] = cand[np.argmin(d2)]                         # candidates ascend: the first minimum is the smallest index
    return out.reshape(Z, Y, X)


def _tsdf(inside, rng=None):
    """A volume whose inside voxels are `inside`: positive values there, -0.01, 0, -inf or NaN elsewhere."""
    t = np.full(inside.shape, -0.01, np.float32)
    if rng is not None:
        t = rng.choice(np.array([-0.01, 0.0, -np.inf, np.nan], np.float32), inside.shape)
    t[inside] = 0.005
    return t


def _cases():
    out = {}
    a = np.zeros((5, 6, 7), bool)
    a[2, 3, 1] = a[2, 3, 5] = True                           # equidistant from the plane x = 3
    out["two_on_a_line"] = a
    b = np.zeros((7, 7, 7), bool)
    b[3, 1, 3] = b[3, 5, 3] = b[1, 3, 3] = b[5, 3, 3] = True   # four voxels around the centre
    out["four_around_a_centre"] = b
    z, y, x = np.meshgrid(*(np.arange(9),) * 3, indexing="ij")
    r2 = (x - 4) ** 2 + (y - 4) ** 2 + (z - 4) ** 2
    out["hollow_shell"] = (r2 >= 9) & (r2 <= 12)
    out["checkerboard"] = ((x + y + z) % 2 == 0)[:6, :5, :7]
    e = np.zeros((6, 5, 4), bool)
    e[0, 0, 0] = e[5, 4, 3] = e[0, 4, 3] = e[5, 0, 0] = True   # corners only
    out["border_voxels"] = e
    out["empty"] = np.zeros((4, 5, 6), bool)
    out["full"] = np.ones((4, 5, 6), bool)
    rng = np.random.default_rng(3)
    out["non_cubic_7x11x13"] = rng.random((13, 11, 7)) < 0.03
    out["single"] = np.pad(np.ones((1, 1, 1), bool), ((2, 3), (1, 4), (0, 5)))
    return out


@pytest.mark.parametrize("name", sorted(_cases()))
def test_separable_argmin_equals_brute_force(name):
    inside = _cases()[name]
    want = brute_force(inside)
    assert np.array_equal(D.nearest_bruteforce_separable(inside), want), name
    # the C++ transform too, from a volume whose outside holds the values that are never inside (0, -limit, -inf, NaN)
    assert np.array_equal(D.nearest_voxels(_tsdf(inside, np.random.default_rng(1))), want), name


def test_inside_rule():
    t = np.array([[[0.0, -0.0, np.nan, np.inf, -np.inf, 1e-30, 3.0]]], np.float32)
    n = D.nearest_voxels(t)
    assert n.reshape(-1).tolist() == [5, 5, 5, 5, 5, 5, 6]   # only the finite positive values are inside; ties to the left


def _blobs(shape, n, seed, radius=(2, 9)):
    rng = np.random.default_rng(seed)
    Z, Y, X = shape
    z, y, x = np.meshgrid(np.arange(Z), np.arange(Y), np.arange(X), indexing="ij")
    inside = np.zeros(shape, bool)
    for _ in range(n):
        c = rng.uniform(0, 1, 3) * (X, Y, Z)
        r = rng.uniform(*radius)
        inside |= (x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2 <= r * r
    return inside


@pytest.mark.parametrize("shape", [(64, 64, 64), (80, 64, 48)])
def test_cpp_oracle_equals_argmin_oracle(shape):
    inside = _blobs(shape, 6, 7, (1, 5))
    inside |= np.random.default_rng(11).random(shape) < 2e-4   # isolated voxels: many exact ties between them
    got = D.nearest_voxels(_tsdf(inside))
    assert np.array_equal(got, D.nearest_bruteforce_separable(inside))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_squared_distances_equal_scipy(seed):
    inside = _blobs((128, 128, 128), 5 + 3 * seed, seed)
    d2 = D.squared_distances(D.nearest_voxels(_tsdf(inside)))
    want = np.rint(ndimage.distance_transform_edt(~inside) ** 2).astype(np.int64)
    assert np.array_equal(d2, want)
    assert (d2[inside] == 0).all()


# ---- queries -----------------------------------------------------------------------------------------------------------
BMIN, BMAX = np.array([-1.0, 0.0, -1.0], np.float32), np.array([1.0, 2.0, 1.0], np.float32)   # 4x4x4 voxels of 0.5 m


def _field():
    inside = np.zeros((4, 4, 4), bool)
    inside[1, 2, 3] = True                                   # voxel (x 3, y 2, z 1), centre (0.75, 1.25, -0.25)
    return D.nearest_voxels(_tsdf(inside))


def test_query_on_a_voxel_centre():
    nearest = _field()
    d, c, v = D.sample_distance(nearest, BMIN, BMAX, [[0.75, 1.25, -0.25], [-0.75, 0.25, -0.75]])
    assert v.tolist() == [1 * 16 + 2 * 4 + 3] * 2
    assert bits_equal(c, np.array([[0.75, 1.25, -0.25]] * 2, np.float32)).all()
    assert d[0] == 0.0
    assert d[1] == np.float32(np.sqrt(np.float32(1.5 * 1.5 + 1.0 * 1.0) + np.float32(0.5 * 0.5)))


def test_query_on_boundaries_and_volume_space():
    nearest = _field()
    # on the cell boundary x = 0.5 (q = 0.75): the voxel above (floor(0.75 * 4) = 3); at q = 1 the last voxel (clamped)
    d, c, v = D.sample_distance(nearest, BMIN, BMAX, [[0.75, 0.5, 0.375], [1.0, 1.0, 1.0], [0.0, 0.0, 0.0]], space=D.VOLUME)
    assert v.tolist() == [27, 27, 27]
    assert bits_equal(c, np.array([[0.875, 0.625, 0.375]] * 3, np.float32)).all()   # volume space
    p = BMIN + np.array([1.0, 1.0, 1.0], np.float32) * (BMAX - BMIN)
    dd = p - np.array([0.75, 1.25, -0.25], np.float32)
    assert d[1] == np.sqrt((dd[0] * dd[0] + dd[1] * dd[1]) + dd[2] * dd[2])
    assert d[2] > d[0] > 0


def test_query_outside_nan_and_empty():
    nearest = _field()
    d, c, v = D.sample_distance(nearest, BMIN, BMAX, [[1.01, 1.0, 0.0], [np.nan, 1.0, 0.0], [0.0, np.inf, 0.0], [0.0, 1.0, 0.0]])
    assert np.isnan(d[:3]).all() and np.isnan(c[:3]).all() and (v[:3] == NONE).all()
    assert np.isfinite(d[3]) and v[3] != NONE
    empty = D.nearest_voxels(np.full((4, 4, 4), -0.01, np.float32))
    assert (empty == NONE).all()
    d, c, v = D.sample_distance(empty, BMIN, BMAX, [[0.0, 1.0, 0.0], [5.0, 1.0, 0.0]])
    assert d[0] == np.inf and np.isnan(c[0]).all() and v[0] == NONE
    assert np.isnan(d[1]) and v[1] == NONE
