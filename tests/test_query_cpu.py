"""The query contract on the oracle alone (oracle/ro_query.cpp), on an analytic sphere TSDF: where rays hit, which way the
normals face, rays that miss, rays starting inside, and point samples inside, outside and beyond the volume. The device kernels
are held to the oracle bit for bit by test_query_gpu.py."""
import numpy as np
import oracle_query as Q
import pytest

RES = (48, 44, 40)
BMIN, BMAX = np.array([-1.0, -0.9, -0.8], np.float32), np.array([1.0, 1.1, 0.8], np.float32)
SIZE = BMAX - BMIN
CENTRE, RADIUS, LIMIT = np.array([0.1, 0.05, -0.02], np.float32), np.float32(0.45), 0.02
STEP_M = float(LIMIT / 2 * SIZE.max())          # the longest a march step can be, in metres


def _voxel_centres():
    X, Y, Z = RES
    z, y, x = np.meshgrid((np.arange(Z) + 0.5) / Z, (np.arange(Y) + 0.5) / Y, (np.arange(X) + 0.5) / X, indexing="ij")
    return BMIN + np.stack([x, y, z], -1).astype(np.float32) * SIZE


@pytest.fixture(scope="module")
def sphere():
    """tsdf [Z][Y][X]: positive inside the sphere (the raymarch's hit test is density > 0), clamped to +-0.1 m."""
    d = np.linalg.norm(_voxel_centres() - CENTRE, axis=-1)
    return np.clip(RADIUS - d, -0.1, 0.1).astype(np.float32)


def _cast(tsdf, origins, directions, **kw):
    return Q.cast_rays(tsdf, RES, LIMIT, BMIN, BMAX, origins, directions, **kw)


def _sphere_rays(n, seed=1):
    """Origins on a shell outside the sphere but inside the volume, aimed at the centre."""
    rng = np.random.default_rng(seed)
    u = rng.normal(size=(n, 3)).astype(np.float32)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    o = (CENTRE + u * np.float32(0.7)).astype(np.float32)
    o = np.clip(o, BMIN + 0.01, BMAX - 0.01)
    return o, (CENTRE - o).astype(np.float32)


@pytest.mark.parametrize("space", ["world", "volume"])
def test_rays_aimed_at_the_centre_hit_the_sphere(sphere, space):
    o, d = _sphere_rays(500)
    if space == "volume":
        pos, nrm, rgba, steps = _cast(sphere, (o - BMIN) / SIZE, d / SIZE, space=Q.VOLUME)
        pos = BMIN + pos * SIZE
    else:
        pos, nrm, rgba, steps = _cast(sphere, o, d)
    assert (steps != 0xFFFFFFFF).all() and (steps >= 1).all()
    r = np.linalg.norm(pos - CENTRE, axis=1)
    assert np.abs(r - RADIUS).max() < STEP_M
    # the hit lies between the origin and the centre
    assert (np.linalg.norm(pos - o, axis=1) <= np.linalg.norm(CENTRE - o, axis=1)).all()


def test_normals_point_outward(sphere):
    o, d = _sphere_rays(500, seed=2)
    pos, nrm, _, _ = _cast(sphere, o, d)
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1.0, atol=1e-5)
    radial = (pos - CENTRE) / np.linalg.norm(pos - CENTRE, axis=1, keepdims=True)
    assert ((nrm * radial).sum(1) > 0.95).all()
    # the point sample's normal is the same formula (in volume space the hit position is the march's q itself)
    qpos, qnrm, _, _ = _cast(sphere, (o - BMIN) / SIZE, d / SIZE, space=Q.VOLUME)
    _, pn, _ = Q.sample_points(sphere, RES, LIMIT, BMIN, BMAX, qpos, space=Q.VOLUME)
    assert np.array_equal(pn.view(np.uint32), qnrm.view(np.uint32))


def test_rays_that_miss_get_no_hit(sphere):
    o = np.array([[-1.5, 0.0, 0.0], [0.0, 2.0, 0.0], [-0.9, 0.0, 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0], [np.nan, 0.0, 0.0]], np.float32)
    d = np.array([[-1.0, 0.0, 0.0],    # outside, pointing away from the cube
                  [0.0, 1.0, 0.1],     # outside, away
                  [0.0, 1.0, 0.0],     # inside the volume, passing beside the sphere
                  [0.0, 0.0, 0.0],     # zero direction
                  [np.inf, 0.0, 0.0],  # non-finite direction
                  [1.0, 0.0, 0.0]], np.float32)   # non-finite origin
    pos, nrm, rgba, steps = _cast(sphere, o, d)
    assert (steps == 0xFFFFFFFF).all()
    assert np.isnan(pos).all() and np.isnan(nrm).all() and (rgba == 0).all()


def test_ray_starting_inside_the_surface_hits_at_step_one(sphere):
    o = np.array([CENTRE, CENTRE + np.float32(0.2)], np.float32)
    d = np.array([[0.3, -1.0, 0.2], [1.0, 1.0, 1.0]], np.float32)
    pos, _, _, steps = _cast(sphere, o, d)
    assert (steps == 1).all()
    assert np.isfinite(pos).all()


def test_skip_space_hull_gives_the_same_hits(sphere):
    """With the occupied bricks covering the sphere the march over their hull finds the same surface."""
    brick = np.float32(0.25)
    rb = np.ceil(SIZE / brick).astype(np.uint32)
    lo = BMIN + np.stack(np.meshgrid(*[np.arange(n) for n in rb[::-1]], indexing="ij")[::-1], -1).reshape(-1, 3) * brick
    near = np.linalg.norm(np.clip(CENTRE, lo, lo + brick) - CENTRE, axis=1) <= RADIUS + 0.1
    occ = np.nonzero(near)[0].astype(np.uint32)
    o, d = _sphere_rays(300, seed=3)
    full = _cast(sphere, o, d)
    hull = _cast(sphere, o, d, skip_space=True, occupied=occ, brick_res=rb, brick_size=brick)
    assert (hull[3] != 0xFFFFFFFF).all()
    assert np.abs(np.linalg.norm(hull[0] - CENTRE, axis=1) - RADIUS).max() < STEP_M
    assert np.abs(hull[0] - full[0]).max() < STEP_M


def test_point_value_sign_matches_inside_and_outside(sphere):
    rng = np.random.default_rng(4)
    p = (BMIN + rng.random((4000, 3)).astype(np.float32) * SIZE).astype(np.float32)
    val, nrm, rgba = Q.sample_points(sphere, RES, LIMIT, BMIN, BMAX, p)
    d = np.linalg.norm(p - CENTRE, axis=1)
    clear = np.abs(d - RADIUS) > 0.05            # away from the surface, where trilinear filtering cannot flip the sign
    assert (val[clear & (d < RADIUS)] > 0).all() and (val[clear & (d > RADIUS)] < 0).all()
    assert np.isfinite(val).all()
    vol = Q.sample_points(sphere, RES, LIMIT, BMIN, BMAX, (p - BMIN) / SIZE, space=Q.VOLUME)[0]
    assert np.allclose(vol, val, atol=1e-6)


def test_points_outside_the_unit_cube_are_nan(sphere):
    p = np.array([BMIN - 0.01, BMAX + 0.01, [0.0, 0.0, 5.0], [np.nan, 0.0, 0.0], [np.inf, 0.0, 0.0], BMIN, BMAX], np.float32)
    val, nrm, rgba = Q.sample_points(sphere, RES, LIMIT, BMIN, BMAX, p)
    assert np.isnan(val[:5]).all() and np.isnan(nrm[:5]).all() and (rgba[:5] == 0).all()
    assert np.isfinite(val[5:]).all()            # the bbox corners are in the closed cube


@pytest.mark.parametrize("space", ["world", "volume"])
def test_huge_and_tiny_directions_are_rays(sphere, space):
    """A finite non-zero direction is a ray whatever its length: one whose squared length overflows binary32 (which would
    normalise to the zero vector and march in place) or underflows is scaled by a power of two first, so it casts exactly
    as the same direction of ordinary length."""
    o, d = _sphere_rays(200, seed=6)
    d = np.where(np.abs(d) < 0.1, np.copysign(np.float32(0.1), d), d).astype(np.float32)   # no component near 0 or denormal when scaled
    if space == "volume":
        o, d, sp = ((o - BMIN) / SIZE).astype(np.float32), (d / SIZE).astype(np.float32), Q.VOLUME
    else:
        sp = Q.WORLD
    want = _cast(sphere, o, d, space=sp)
    assert (want[3] != 0xFFFFFFFF).all()
    for scale in (np.float32(2.0 ** 70), np.float32(2.0 ** 100), np.float32(2.0 ** -110)):
        got = _cast(sphere, o, (d * scale).astype(np.float32), space=sp)
        for g, w in zip(got, want):
            assert np.array_equal(np.asarray(g).view(np.uint32), np.asarray(w).view(np.uint32)), f"scale {scale}"
    # a direction 1e20 long along +x, from outside the sphere
    pos, _, _, steps = _cast(sphere, np.array([[-0.8, 0.05, -0.02]], np.float32), np.array([[1e20, 0.0, 0.0]], np.float32))
    assert steps[0] != 0xFFFFFFFF and abs(pos[0, 0] - (CENTRE[0] - RADIUS)) < STEP_M


def test_origins_beyond_2_24_bbox_sizes_are_not_cast(sphere):
    """The march's step count comes from binary32 ray parameters; an origin farther than 2^24 bbox sizes is not cast (no hit)
    instead of marching for billions of steps."""
    far = np.float32(2.0 ** 25)
    o = np.array([[-far, 0.05, -0.02], [0.1, 0.05, 1e30], [-0.8, 0.05, -0.02]], np.float32)
    d = np.array([[1.0, 0.0, 0.0], [0.001, 0.0, -1.0], [1.0, 0.0, 0.0]], np.float32)
    pos, nrm, rgba, steps = _cast(sphere, (o - BMIN) / SIZE, d, space=Q.VOLUME)
    assert (steps[:2] == 0xFFFFFFFF).all() and np.isnan(pos[:2]).all()
    assert steps[2] != 0xFFFFFFFF
