"""Queries of the fused volume on the device (rr_sample_points / rr_cast_rays and their group forms) against the oracle's
scalar restatement (oracle/ro_query.cpp) and against the raymarch itself, bit for bit (NaN == NaN): values, positions,
normals, colours and steps. The oracle reads the volume, stage images and brick tables the context holds at the call."""
import ctypes as C
import os
import subprocess

import numpy as np
import oracle_query as Q
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10
NO_HIT = 0xFFFFFFFF


def _same(what, got, want):
    names = ("positions", "normals", "rgba", "steps") if len(want) == 4 else ("values", "normals", "rgba")
    for n, g, w in zip(names, got, want):
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n == "steps":
            assert np.array_equal(g, w), f"{what} steps: {(g != w).sum()} of {len(w)} differ"
        else:
            assert bits_equal(g, w).all(), mismatch_report(f"{what} {n}", g, w)


def _context(sc, inv, use_bricks=True, store_weight=0, skip_space=True, frame=True, limit=LIMIT):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=limit, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, skip_space=skip_space,
                 store_weight=store_weight)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame()
    return fu


class _Oracle:
    """The oracle over what a context holds now: volume, stage images, limit and brick tables."""

    def __init__(self, fu, sc, inv, limit, skip_space):
        self.sc, self.inv, self.limit, self.skip = sc, inv, limit, skip_space
        self.tsdf, self.res = fu.download_tsdf(), fu.volume_res()
        self.pre = dict(depth_b=fu.download_stage("depth_b"), quality=fu.download_stage("quality"))
        info = fu.brick_info()
        self.occ = fu.download_bricks()[1]
        self.rb, self.bs = info["res_bricks"], info["brick_size"]

    def points(self, p, space=Q.WORLD):
        return Q.sample_points(self.tsdf, self.res, self.limit, self.sc.bbox_min, self.sc.bbox_max, p, space, self.inv, self.sc, self.pre)

    def rays(self, o, d, space=Q.WORLD):
        return Q.cast_rays(self.tsdf, self.res, self.limit, self.sc.bbox_min, self.sc.bbox_max, o, d, space, self.skip, self.occ,
                           self.rb, self.bs, self.inv, self.sc, self.pre)


def _bbox(sc):
    return np.asarray(sc.bbox_min, np.float32), np.asarray(sc.bbox_max, np.float32)


def _random_points(sc, n, seed):
    lo, hi = _bbox(sc)
    return (lo + np.random.default_rng(seed).random((n, 3)).astype(np.float32) * (hi - lo)).astype(np.float32)


def _odd_points(sc):
    """Outside the bbox, on its faces and corners, and non-finite."""
    lo, hi = _bbox(sc)
    mid = (lo + hi) / 2
    return np.array([lo - 0.01, hi + 0.01, lo, hi, [mid[0], hi[1] + 1e-3, mid[2]], [mid[0], mid[1], lo[2]],
                     [np.nan, mid[1], mid[2]], [mid[0], np.inf, mid[2]], [-np.inf, 0, 0], mid], np.float32)


def _camera_rays(fu, sc, n, seed):
    """From every sensor's camera towards random points of the bbox (world space)."""
    cams = fu.camera_positions()
    rng = np.random.default_rng(seed)
    o = cams[rng.integers(0, len(cams), n)].astype(np.float32)
    return o, (_random_points(sc, n, seed + 1) - o).astype(np.float32)


def _inside_rays(sc, n, seed):
    rng = np.random.default_rng(seed)
    return _random_points(sc, n, seed), rng.normal(size=(n, 3)).astype(np.float32)


def _special_rays(sc):
    """Axis-parallel rays (both signs, through the middle), rays that miss the cube, zero and non-finite directions."""
    lo, hi = _bbox(sc)
    mid = (lo + hi) / 2
    o, d = [], []
    for a in range(3):
        for s in (1.0, -1.0):
            start = mid.copy()
            start[a] = lo[a] - 0.5 if s > 0 else hi[a] + 0.5
            for off in (-0.2, 0.0, 0.17):
                q = start.copy()
                q[(a + 1) % 3] += off
                e = np.zeros(3, np.float32)
                e[a] = s
                o.append(q); d.append(e)
    o += [lo - 1.0, hi + 1.0, mid, mid, mid]
    d += [[-1.0, 0.0, 0.0], [0.0, 1.0, 1.0], [0.0, 0.0, 0.0], [np.nan, 1.0, 0.0], [np.inf, 0.0, 0.0]]
    return np.array(o, np.float32), np.array(d, np.float32)


@pytest.fixture(scope="module")
def scene2():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("store_weight", [0, 1, 2])
@pytest.mark.parametrize("mode", ["bricks", "dense"])
def test_points_match_oracle(scene2, store_weight, mode):
    sc, inv = scene2
    fu = _context(sc, inv, use_bricks=mode == "bricks", store_weight=store_weight)
    orc = _Oracle(fu, sc, inv, LIMIT, False)
    p = _random_points(sc, 20000, 1)
    got = fu.sample_points(p)
    _same(f"random {mode} {store_weight}", got, orc.points(p))
    assert (got[0] > 0).any() and (got[0] < 0).any() and (got[2][:, 3] == 1.0).any()
    mesh_pos = fu.extract_mesh()[0]
    _same("mesh vertices", fu.sample_points(mesh_pos), orc.points(mesh_pos))
    odd = _odd_points(sc)
    got = fu.sample_points(odd)
    _same("odd points", got, orc.points(odd))
    assert np.isnan(got[0][[0, 1, 6, 7, 8]]).all() and np.isfinite(got[0][[2, 3, 5, 9]]).all()
    lo, hi = _bbox(sc)
    q = (p - lo) / (hi - lo)
    _same("volume space", fu.sample_points(q, space="volume"), orc.points(q, Q.VOLUME))
    fu.close()


@pytest.mark.parametrize("store_weight", [0, 1, 2])
@pytest.mark.parametrize("mode", ["skip", "noskip", "dense"])
def test_rays_match_oracle(scene2, store_weight, mode):
    sc, inv = scene2
    fu = _context(sc, inv, use_bricks=mode != "dense", skip_space=mode == "skip", store_weight=store_weight)
    orc = _Oracle(fu, sc, inv, LIMIT, mode == "skip")
    for what, (o, d) in (("camera", _camera_rays(fu, sc, 6000, 2)), ("inside", _inside_rays(sc, 6000, 3)), ("special", _special_rays(sc))):
        got = fu.cast_rays(o, d)
        _same(f"{what} {mode} {store_weight}", got, orc.rays(o, d))
        if what == "camera":
            assert (got[3] != NO_HIT).sum() > 300
    o, d = _special_rays(sc)
    steps = fu.cast_rays(o, d)[3]
    assert (steps[-5:] == NO_HIT).all()
    # directions whose squared length overflows or underflows binary32 cast exactly as the same direction of ordinary
    # length; origins beyond 2^24 bbox sizes are not cast
    o, d = _camera_rays(fu, sc, 2000, 5)
    d = np.where(np.abs(d) < 0.1, np.copysign(np.float32(0.1), d), d).astype(np.float32)
    want = fu.cast_rays(o, d)
    for scale in (np.float32(2.0 ** 70), np.float32(2.0 ** 100), np.float32(2.0 ** -110)):
        got = fu.cast_rays(o, (d * scale).astype(np.float32))
        _same(f"direction x {scale}", got, want)
        _same(f"direction x {scale} oracle", got, orc.rays(o, (d * scale).astype(np.float32)))
    lo, hi = _bbox(sc)
    far = np.array([[lo[0] - 2.0 ** 25 * (hi[0] - lo[0]), lo[1], lo[2]], [0.0, 1e30, 0.0]], np.float32)
    fd = np.array([[1.0, 0.01, 0.01], [0.0, -1.0, 0.001]], np.float32)
    got = fu.cast_rays(far, fd)
    _same("far origins", got, orc.rays(far, fd))
    assert (got[3] == NO_HIT).all()
    lo, hi = _bbox(sc)
    o, d = _camera_rays(fu, sc, 3000, 4)
    _same("volume space", fu.cast_rays((o - lo) / (hi - lo), d, space="volume"), orc.rays((o - lo) / (hi - lo), d, Q.VOLUME))
    fu.close()


def _view_rays(mv, pr, sc, w, h, limit):
    """The raymarch's own rays of a w x h view in volume space: origin = the camera, direction = screenToVol(pixel, 1) - camera."""
    import oracle_py as O
    cam = O.raymarch_uniforms(mv, pr, sc.bbox_min, sc.bbox_max, w, h)[80:83]
    pts, _ = O.raymarch_rays(mv, pr, sc.bbox_min, sc.bbox_max, w, h, limit)
    pts = pts.reshape(-1, 3)
    return np.broadcast_to(cam, pts.shape).astype(np.float32), (pts - cam).astype(np.float32)


def _check_against_raymarch(fu, mv, pr, w, h, what, o, d):
    view = fu.raymarch(mv, pr, w, h, shade_mode=0)
    hitpos = fu.download_hit_positions(w, h).reshape(-1, 4)
    nsamp = fu.download_num_samples(w, h).reshape(-1)
    pos, nrm, rgba, steps = fu.cast_rays(o, d, space="volume")
    hit = steps != NO_HIT
    assert np.array_equal(hit, hitpos[:, 3] == 1.0), f"{what}: hit pixels differ"
    assert hit.sum() > 500
    assert bits_equal(pos[hit], hitpos[hit, :3]).all(), mismatch_report(f"{what} positions", pos[hit], hitpos[hit, :3])
    want_ns = steps[hit].astype(np.float32) * np.float32(0.0027)
    assert bits_equal(want_ns, nsamp[hit]).all(), mismatch_report(f"{what} samples", want_ns, nsamp[hit])
    assert bits_equal(rgba, view[0].reshape(-1, 4)).all(), mismatch_report(f"{what} rgba", rgba, view[0].reshape(-1, 4))


@pytest.mark.parametrize("skip", [True, False])
def test_rays_equal_the_raymarch_headline(skip):
    import bench
    from rrpy import capi, synth
    scenes, inv, voxel = bench.make_inputs()
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True, skip_space=skip)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    w, h = 1280, 720
    mv, pr = synth.look_at((1.6, 1.5, 2.2), (0.0, 1.1, 0.0)), synth.perspective(50.0, w / h, 0.1, 10.0)
    o, d = _view_rays(mv, pr, sc, w, h, bench.LIMIT)
    _check_against_raymarch(fu, mv, pr, w, h, f"headline skip={skip}", o, d)
    fu.close()


def test_headline_and_eight_sensors_match_oracle():
    import bench
    from rrpy import capi, synth
    scenes, inv, voxel = bench.make_inputs()
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    orc = _Oracle(fu, sc, inv, bench.LIMIT, True)
    o, d = _camera_rays(fu, sc, 4000, 5)
    got = fu.cast_rays(o, d)
    _same("512^3 rays", got, orc.rays(o, d))
    assert (got[3] != NO_HIT).sum() > 500
    p = np.concatenate([_random_points(sc, 5000, 6), got[0][got[3] != NO_HIT]])
    _same("512^3 points", fu.sample_points(p), orc.points(p))
    fu.close()

    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv, store_weight=2)
    orc = _Oracle(fu, sc, inv, LIMIT, True)
    o, d = _camera_rays(fu, sc, 4000, 7)
    _same("8 sensors rays", fu.cast_rays(o, d), orc.rays(o, d))
    p = _random_points(sc, 4000, 8)
    _same("8 sensors points", fu.sample_points(p), orc.points(p))
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "configure_limit", "bricks_clear"])
def test_query_after_call_orders_equals_raymarch(scene2, order):
    """A call between the integrate and the query: the query marches with what rr_raymarch would use now (the same code
    path), so it equals the raymarch's hits, samples and colours; the oracle is checked too."""
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    limit = LIMIT
    if order == "bricks_update_other":       # brick tables of another frame set than the volume was integrated with
        other = synth.rerender(sc, 7)
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
        sc_pre = other
    elif order == "configure_limit":
        limit = 0.02
        fu.configure(limit=limit, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
        sc_pre = sc
    else:
        fu.bricks_clear()
        sc_pre = sc
    w, h = 200, 120
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, w / h, 0.1, 10.0)
    o, d = _view_rays(mv, pr, sc, w, h, limit)
    _check_against_raymarch(fu, mv, pr, w, h, order, o, d)
    orc = _Oracle(fu, sc_pre, inv, limit, True)
    o, d = _camera_rays(fu, sc, 3000, 9)
    got, want = fu.cast_rays(o, d), orc.rays(o, d)
    if order == "bricks_update_other":
        # stale tables: empty-space fetch skipping may skip samples of bricks that are occupied in the volume but not in
        # the new tables; the oracle samples every step. Report, do not hide, a difference.
        same = bits_equal(got[0], want[0]).all(axis=1) & (got[3] == want[3])
        print(f"stale brick tables: {int((~same).sum())} of {len(same)} rays differ from the oracle")
    else:
        _same(order, got, want)
    fu.close()


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


def test_refusals_and_limits(scene2):
    from rrpy import capi
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    p = np.zeros((4, 3), np.float32)
    pp = p.ctypes.data
    out = np.zeros((4, 4), np.float32)
    op = out.ctypes.data
    assert _status(fu, "rr_sample_points", 0, pp, 4, op, None, None) == -1                # nothing integrated yet
    assert _status(fu, "rr_cast_rays", 0, pp, pp, 4, op, None, None, None) == -1
    fu.frame()
    assert _status(fu, "rr_sample_points", 2, pp, 4, op, None, None) == -1                # bad space
    assert _status(fu, "rr_cast_rays", -1, pp, pp, 4, op, None, None, None) == -1
    assert _status(fu, "rr_sample_points", 0, None, 4, op, None, None) == -1              # null inputs
    assert _status(fu, "rr_cast_rays", 0, pp, None, 4, op, None, None, None) == -1
    assert _status(fu, "rr_sample_points", 0, pp, 1 << 31, op, None, None) == -4          # 2^31 entries
    assert _status(fu, "rr_cast_rays", 0, pp, pp, 0xFFFFFFFF, op, None, None, None) == -4
    assert _status(fu, "rr_sample_points", 0, None, 0, None, None, None) == 0             # count 0: nothing to do
    assert _status(fu, "rr_cast_rays", 1, None, None, 0, None, None, None, None) == 0
    # NULL outputs: any subset
    o, d = _camera_rays(fu, sc, 1000, 10)
    full = fu.cast_rays(o, d)
    steps = np.zeros(1000, np.uint32)
    assert _status(fu, "rr_cast_rays", 0, o.ctypes.data, d.ctypes.data, 1000, None, None, None, steps.ctypes.data) == 0
    assert np.array_equal(steps, full[3])
    assert _status(fu, "rr_cast_rays", 0, o.ctypes.data, d.ctypes.data, 1000, None, None, None, None) == 0
    pts = _random_points(sc, 1000, 11)
    fullp = fu.sample_points(pts)
    nrm = np.zeros((1000, 3), np.float32)
    assert _status(fu, "rr_sample_points", 0, pts.ctypes.data, 1000, None, nrm.ctypes.data, None) == 0
    assert bits_equal(nrm, fullp[1]).all()
    # a new voxel format is a new volume; a slab-restricted context is refused
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True, store_weight=capi.VOXELS_HALF2)
    assert _status(fu, "rr_sample_points", 0, pp, 4, op, None, None) == -1
    fu.frame()
    assert _status(fu, "rr_sample_points", 0, pp, 4, op, None, None) == 0
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_cast_rays", 0, pp, pp, 4, op, None, None, None) == -1
    assert "group" in fu.L.rr_last_error(fu.h).decode()
    fu.close()


def test_buffers_grow_and_shrink_back(scene2):
    sc, inv = scene2
    fu = _context(sc, inv)
    orc = _Oracle(fu, sc, inv, LIMIT, True)
    o, d = _camera_rays(fu, sc, 1, 12)
    first = fu.cast_rays(o, d)
    _same("1 ray", first, orc.rays(o, d))
    big_o, big_d = _camera_rays(fu, sc, 1000000, 13)
    big = fu.cast_rays(big_o, big_d)
    sel = np.random.default_rng(14).choice(1000000, 20000, replace=False)
    _same("1e6 rays (a sample)", tuple(a[sel] for a in big), orc.rays(big_o[sel], big_d[sel]))
    p = _random_points(sc, 1000000, 15)
    bigp = fu.sample_points(p)
    _same("1e6 points (a sample)", tuple(a[sel] for a in bigp), orc.points(p[sel]))
    _same("1 ray again", fu.cast_rays(o, d), first)
    fu.close()


def test_queries_have_no_side_effects(scene2):
    """The volume, the last view's raymarch and fill, the mesh, the next fused frame's volume and the launches per fused
    frame are the same with and without queries in between (captured frame graphs stay valid)."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 3)
    w, h = 200, 120
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, w / h, 0.1, 10.0)
    runs = []
    for query in (False, True):
        fu = _context(sc, inv, frame=False)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        view = fu.raymarch(mv, pr, w, h, shade_mode=1)
        counts = fu.extract_mesh_counts()
        if query:
            fu.cast_rays(*_camera_rays(fu, sc, 5000, 16))
            fu.sample_points(_random_points(sc, 5000, 17))
        mesh = fu.download_mesh(*counts)
        filled = fu.fill_colors()
        tsdf = fu.download_tsdf()
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        assert fu.launch_count() - l0 == per_frame
        runs.append((view, filled, mesh, tsdf, fu.download_tsdf(), per_frame))
        fu.close()
    a, b = runs
    assert bits_equal(a[0][0], b[0][0]).all() and bits_equal(a[0][1], b[0][1]).all()
    assert bits_equal(a[1], b[1]).all()
    for x, y in zip(a[2], b[2]):
        assert bits_equal(x, y).all() if x.dtype == np.float32 else np.array_equal(x, y)
    assert bits_equal(a[3], b[3]).all() and bits_equal(a[4], b[4]).all()
    assert a[5] == b[5]


def test_torch_tensors_equal_numpy(scene2):
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    o, d = _camera_rays(fu, sc, 5000, 18)
    p = _random_points(sc, 5000, 19)
    want_r, want_p = fu.cast_rays(o, d), fu.sample_points(p)
    dev = torch.device("cuda", 0)
    got_r = fu.cast_rays(torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev))
    got_p = fu.sample_points(torch.from_numpy(p).to(dev))
    assert all(t.is_cuda for t in got_r + got_p)
    _same("torch rays", tuple(t.cpu().numpy() for t in got_r), want_r)
    _same("torch points", tuple(t.cpu().numpy() for t in got_p), want_p)
    _same("torch host rays", fu.cast_rays(torch.from_numpy(o), torch.from_numpy(d)), want_r)
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_queries_equal_single_context(scene2, n):
    from rrpy import capi, synth
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    Z = int(fu.volume_res()[2])
    lo, hi = _bbox(sc)
    o1, d1 = _camera_rays(fu, sc, 20000, 20)
    o2, d2 = _inside_rays(sc, 5000, 21)
    o3, d3 = _special_rays(sc)
    # rays along z through the whole volume cross every slab boundary
    xy = _random_points(sc, 2000, 22)
    o4 = np.concatenate([xy[:, :2], np.full((2000, 1), lo[2] - 0.1, np.float32)], 1)
    d4 = np.tile(np.array([[0.01, -0.02, 1.0]], np.float32), (2000, 1))
    o, d = np.concatenate([o1, o2, o3, o4]), np.concatenate([d1, d2, d3, d4])
    # points on every slice centre and boundary (where the owner changes) and on the slices just beside them
    zs = np.concatenate([(np.arange(Z) + 0.5) / Z, np.arange(Z + 1) / Z, np.nextafter(np.arange(1, Z) / Z, 0).astype(np.float32)]).astype(np.float32)
    pz = _random_points(sc, len(zs), 23)
    pz[:, 2] = lo[2] + zs * (hi[2] - lo[2])
    p = np.concatenate([_random_points(sc, 20000, 24), pz, _odd_points(sc), fu.extract_mesh()[0]])
    want_r, want_p = fu.cast_rays(o, d), fu.sample_points(p)
    want_v = fu.sample_points(np.stack([np.full(len(zs), 0.5, np.float32), np.full(len(zs), 0.5, np.float32), zs], 1), space="volume")
    fu.close()

    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    _same(f"group of {n} rays", g.cast_rays(o, d), want_r)
    _same(f"group of {n} points", g.sample_points(p), want_p)
    zv = np.stack([np.full(len(zs), 0.5, np.float32), np.full(len(zs), 0.5, np.float32), zs], 1)
    _same(f"group of {n} slice points", g.sample_points(zv, space="volume"), want_v)
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_pick(tmp_path, small_scene, devices):
    """fusion_playback --pick prints the world ray through a view pixel and its hit; replaying the printed ray through
    Fusion.cast_rays on the same frame set gives the printed hit bit for bit (on one device and through a group)."""
    from test_host_cpp import BIN, write_scene_files
    from rrpy import capi, synth, volume_io
    sc = small_scene
    ks, streams = write_scene_files(str(tmp_path), sc)
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    for i in range(sc.N):
        volume_io.write_volume(str(tmp_path / f"sensor{i}.cv_xyz_inv"), inv[i])
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame()
    # a pixel the playback's own last view covers (--dump-image: rgba float32 [h][w][4], then depth [h][w], row 0 = bottom)
    w, h = 96, 72
    base = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
            "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", str(w), str(h)]
    img = str(tmp_path / "view.bin")
    r = subprocess.run(base + ["--dump-image", img], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    covered = np.fromfile(img, np.float32)[w * h * 4:].reshape(h, w) < 1.0
    inner = covered & np.roll(covered, 1, 0) & np.roll(covered, -1, 0) & np.roll(covered, 1, 1) & np.roll(covered, -1, 1)
    ys, xs = np.nonzero(inner if inner.any() else covered)
    assert len(ys), "the playback's view shows no surface"
    k = np.argmin((ys - ys.mean()) ** 2 + (xs - xs.mean()) ** 2)
    px, py = int(xs[k]), int(ys[k])
    lines = {}
    for dev in (None, devices) if devices else (None,):
        r = subprocess.run(base + ["--pick", str(px), str(py)] + (["--devices", dev] if dev else []), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        lines[dev] = next(l for l in r.stdout.splitlines() if l.startswith("pick "))
    if devices:
        assert lines[devices] == lines[None], "the multi-device run picked another hit"
    tok = lines[None].split()
    val = lambda key, k: np.array([float(x) for x in tok[tok.index(key) + 1: tok.index(key) + 1 + k]], np.float32)
    o, d = val("origin", 3), val("direction", 3)
    pos, nrm, rgba, steps = fu.cast_rays(o[None], d[None])
    fu.close()
    assert steps[0] != NO_HIT, lines[None]
    assert int(tok[tok.index("step") + 1]) == int(steps[0])
    assert bits_equal(val("hit", 3), pos[0]).all() and bits_equal(val("normal", 3), nrm[0]).all()
    assert bits_equal(val("rgba", 4), rgba[0]).all()
