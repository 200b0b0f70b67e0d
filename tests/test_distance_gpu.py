"""Distances on the device (rr_distance_field / rr_download_distance_field / rr_sample_distance and the group forms) against
the oracle (oracle/oracle_distance.py), bit for bit: the field against the C++ transform of the volume the context holds,
the queries against the float32 restatement of their formulas over that field. Every scene is fused both by separate
calls and by a replayed frame graph."""
import ctypes as C

import numpy as np
import oracle_distance as D
import pytest

from conftest import bits_equal

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10
NONE = int(D.NONE)


def _scene(n_sensors=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), **kw):
    from rrpy import synth
    sc = synth.make_scene(N=n_sensors, W=W, H=H, CW=CW, CH=CH, cv_res=cv_res, **kw)
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.fixture(scope="module")
def scene2():
    return _scene()


def _context(sc, inv, use_bricks=True, store_weight=0, voxel=VOXEL, brick=BRICK):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=voxel, brick_size=brick, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    return fu


def _fuse(fu, sc, graph):
    fu.upload_frames(sc.color, sc.depth)
    if graph:
        fu.fuse_frame()
        fu.fuse_frame()                                      # the second is a replay of the captured graph
    else:
        fu.frame()


def _query_points(sc, n, seed=0, margin=0.1):
    """n world points over the bbox and a margin around it (some outside), plus a few special ones."""
    rng = np.random.default_rng(seed)
    lo, hi = sc.bbox_min - margin, sc.bbox_max + margin
    p = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    p[:4] = [sc.bbox_min, sc.bbox_max, [np.nan, 1.0, 0.0], [np.inf, 0.0, 0.0]]
    return p


def _same_query(what, got, want):
    for name, g, w in zip(("distances", "nearest_points", "nearest_voxels"), got, want):
        g = g.cpu().numpy() if hasattr(g, "cpu") else np.asarray(g)
        assert g.shape == w.shape, f"{what} {name}: shape {g.shape} != {w.shape}"
        ok = bits_equal(g, w) if w.dtype.kind == "f" else g == w
        assert ok.all(), f"{what} {name}: {int((~ok).sum())} of {ok.size} differ"


def _check(fu, sc, what, points=None, field=None):
    """The field and queries of the context's current volume against the oracle; returns the field."""
    n_inside = fu.distance_field() if field is None else field()
    tsdf = fu.download_tsdf()
    want = D.nearest_voxels(tsdf)
    got = fu.nearest_voxels()
    assert np.array_equal(got, want), f"{what}: nearest differs on {int((got != want).sum())} voxels"
    assert n_inside == int((want.reshape(-1) == np.arange(want.size)).sum()), what
    pts = _query_points(sc, 4096) if points is None else points
    bmin, bmax = sc.bbox_min, sc.bbox_max
    _same_query(f"{what} world", fu.sample_distance(pts), D.sample_distance(want, bmin, bmax, pts, D.WORLD))
    q = ((pts - bmin) / (bmax - bmin)).astype(np.float32)
    _same_query(f"{what} volume", fu.sample_distance(q, "volume"), D.sample_distance(want, bmin, bmax, q, D.VOLUME))
    return want


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("mode", ["f32", "f32_weight", "half2", "dense"])
def test_field_matches_oracle(scene2, mode, graph):
    sc, inv = scene2
    fu = _context(sc, inv, use_bricks=mode != "dense", store_weight={"f32": 0, "f32_weight": 1, "half2": 2, "dense": 0}[mode])
    _fuse(fu, sc, graph)
    want = _check(fu, sc, mode)
    assert (want != D.NONE).all() and fu.distance_field() > 100
    fu.close()


@pytest.mark.parametrize("graph", [False, True])
def test_eight_sensors(graph):
    sc, inv = _scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    fu = _context(sc, inv)
    _fuse(fu, sc, graph)
    _check(fu, sc, "8 sensors")
    fu.close()


@pytest.mark.parametrize("graph", [False, True])
def test_non_cubic_bbox(graph):
    sc, inv = _scene(bbox=((-0.9, 0.1, -0.6), (1.1, 2.0, 0.7)))
    fu = _context(sc, inv, voxel=0.023)
    _fuse(fu, sc, graph)
    X, Y, Z = (int(v) for v in fu.volume_res())
    assert len({X, Y, Z}) == 3
    _check(fu, sc, "non-cubic")
    fu.close()


@pytest.mark.parametrize("use_bricks", [True, False])
def test_headline_frame_set(use_bricks):
    import bench
    from rrpy import capi
    from scipy import ndimage
    scenes, inv, voxel = bench.make_inputs(n_frames=1)
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks)
    for graph in (False, True):
        _fuse(fu, sc, graph)
        assert tuple(fu.volume_res()) == (512, 512, 512)
        want = _check(fu, sc, f"512^3 bricks={use_bricks} graph={graph}", points=_query_points(sc, 1 << 20, seed=3))
    if use_bricks:
        d2 = D.squared_distances(want)
        inside = d2 == 0
        assert np.array_equal(d2, np.rint(ndimage.distance_transform_edt(~inside) ** 2).astype(np.int64))
    fu.close()


def test_surface_queries(scene2):
    """1 M points on the surface (mesh vertices, jittered) in world and volume space, from host and device arrays."""
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    _fuse(fu, sc, True)
    pos = fu.extract_mesh()[0]
    rng = np.random.default_rng(4)
    pts = (pos[rng.integers(0, len(pos), 1 << 20)] + rng.normal(0, 0.01, ((1 << 20), 3))).astype(np.float32)
    want = _check(fu, sc, "surface", points=pts)
    got = fu.sample_distance(torch.from_numpy(pts).cuda())
    _same_query("surface, device inputs", got, D.sample_distance(want, sc.bbox_min, sc.bbox_max, pts))
    assert isinstance(got[0], torch.Tensor) and got[0].is_cuda
    d = got[0].cpu().numpy()
    assert np.isfinite(d).all() and np.median(d) < 0.03   # near the surface
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "configure_brick_size"])
def test_stale_brick_tables(scene2, order):
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    _fuse(fu, sc, False)
    other = synth.rerender(sc, 9)
    if order == "bricks_update_other":
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
    else:
        fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=0.08, min_voxels=MIN_VOX, use_bricks=True)
    _check(fu, sc, order)
    fu.close()


def test_empty_frame_set(scene2):
    sc, inv = scene2
    for graph in (False, True):
        fu = _context(sc, inv)
        fu.upload_frames(sc.color, np.zeros_like(sc.depth))
        if graph:
            fu.fuse_frame()
            fu.fuse_frame()
        else:
            fu.frame()
        want = _check(fu, sc, f"empty graph={graph}")
        assert (want == D.NONE).all() and fu.distance_field() == 0
        d, c, v = fu.sample_distance(np.array([[0.0, 1.0, 0.0], [5.0, 1.0, 0.0]], np.float32))
        assert d[0] == np.inf and np.isnan(c).all() and (v == D.NONE).all() and np.isnan(d[1])
        fu.close()


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


def test_refusals_and_epoch(scene2):
    sc, inv = scene2
    fu = _context(sc, inv)
    n = C.c_uint32()
    pts = np.zeros((4, 3), np.float32)
    out = np.empty(4, np.float32)
    assert _status(fu, "rr_distance_field", C.byref(n)) == -1                       # nothing integrated yet
    assert _status(fu, "rr_download_distance_field", None) == -1                    # no field yet
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, out.ctypes.data, None, None) == -1
    _fuse(fu, sc, False)
    assert _status(fu, "rr_distance_field", None) == -1                             # null count pointer
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, out.ctypes.data, None, None) == -1   # no field yet
    assert _status(fu, "rr_distance_field", C.byref(n)) == 0 and n.value > 0
    assert _status(fu, "rr_sample_distance", 2, pts.ctypes.data, 4, out.ctypes.data, None, None) == -1   # bad space
    assert _status(fu, "rr_sample_distance", 0, None, 4, out.ctypes.data, None, None) == -1              # null points
    assert _status(fu, "rr_sample_distance", 0, None, 0, None, None, None) == 0                          # count 0
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 1 << 31, None, None, None) == -4
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, None, None, None) == 0               # outputs may be NULL
    field = fu.nearest_voxels()
    _fuse(fu, sc, False)                                     # the next integrate: the field is of an older volume state
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, out.ctypes.data, None, None) == -1
    assert np.array_equal(fu.nearest_voxels(), field)        # the download still returns the last field
    fu.distance_field()
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, out.ctypes.data, None, None) == 0
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_distance_field", C.byref(n)) == -1
    assert "rr_group_distance_field" in fu.L.rr_last_error(fu.h).decode()
    assert _status(fu, "rr_sample_distance", 0, pts.ctypes.data, 4, out.ctypes.data, None, None) == 0   # the field stays
    assert fu.L.rr_distance_field(None, C.byref(n)) == -1
    assert fu.L.rr_download_distance_field(None, None) == -1
    assert fu.L.rr_sample_distance(None, 0, None, 0, None, None, None) == -1
    fu.close()


def test_no_side_effects(scene2):
    """Against a twin context that never computes distances: volume, brick tables, view, fill_colors, mesh, simplified mesh,
    parts, tracks, cloud; after the next fused frame (a replayed graph) the volume, the launches per frame and
    rr_integrator_last."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 2)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    runs = []
    for dist in (False, True):
        fu = _context(sc, inv)
        fu.upload_frames(sc.color, sc.depth)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        mesh = fu.extract_mesh()
        simple = fu.simplify_mesh(2)
        cloud = fu.extract_points()
        parts = fu.label_parts()
        tracks = fu.track_parts()
        if dist:
            fu.distance_field()
            fu.sample_distance(_query_points(sc, 1000))
        out = dict(view=view, tsdf=fu.download_tsdf(), bricks=fu.download_bricks(), fill=fu.fill_colors(),
                   mesh=fu.download_mesh(len(mesh[0]), len(mesh[3])), cloud=fu.download_points(len(cloud[0])),
                   simple=fu.download_simplified_mesh(len(simple[0]), len(simple[3])),
                   parts=parts + (fu.part_labels(),) + fu.mesh_parts(),
                   tracks=fu.download_part_tracks(len(tracks[0]), len(tracks[6])))
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        out["per_frame"], out["next_frame"] = (per_frame, fu.launch_count() - l0), fu.download_tsdf()
        out["last"] = fu.integrator_last()
        out["next_tracks"] = fu.track_parts()
        runs.append(out)
        fu.close()
    a, b = runs
    for key in ("view", "mesh", "cloud", "bricks", "simple", "parts", "tracks", "next_tracks"):
        for x, y in zip(a[key], b[key]):
            assert (bits_equal(x, y).all() if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y)), key
    for key in ("tsdf", "next_frame", "fill"):
        assert bits_equal(a[key], b[key]).all(), key
    assert a["per_frame"] == b["per_frame"] and b["per_frame"][0] == b["per_frame"][1]
    assert a["last"] == b["last"]


def test_release_and_regrow(scene2):
    """A new resolution releases the field (no download), and the next field has the new size and is right."""
    sc, inv = scene2
    fu = _context(sc, inv)
    _fuse(fu, sc, False)
    _check(fu, sc, "first")
    fu.configure(limit=LIMIT, voxel_size=0.03, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    assert _status(fu, "rr_download_distance_field", None) == -1
    _fuse(fu, sc, True)
    _check(fu, sc, "coarser")
    fu.configure(limit=LIMIT, voxel_size=0.015, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    _fuse(fu, sc, True)
    _check(fu, sc, "finer")
    fu.close()


def test_cuda_tensor_and_pinned_outputs(scene2):
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    _fuse(fu, sc, False)
    fu.distance_field()
    host = fu.nearest_voxels()
    dev = fu.nearest_voxels(device=True)
    assert isinstance(dev, torch.Tensor) and dev.is_cuda and np.array_equal(dev.cpu().numpy(), host)
    pinned = torch.empty(host.size, dtype=torch.int32).pin_memory()
    assert _status(fu, "rr_download_distance_field", C.c_void_p(pinned.data_ptr())) == 0
    assert np.array_equal(pinned.numpy().view(np.uint32).reshape(host.shape), host)
    pts = _query_points(sc, 5000)
    want = D.sample_distance(host, sc.bbox_min, sc.bbox_max, pts)
    pin_in = torch.from_numpy(pts).pin_memory()
    outs = [torch.empty(5000, dtype=torch.float32).pin_memory(), torch.empty((5000, 3), dtype=torch.float32).pin_memory(),
            torch.empty(5000, dtype=torch.int32).pin_memory()]
    assert _status(fu, "rr_sample_distance", 0, C.c_void_p(pin_in.data_ptr()), 5000, *[C.c_void_p(t.data_ptr()) for t in outs]) == 0
    _same_query("pinned", (outs[0].numpy(), outs[1].numpy(), outs[2].numpy().view(np.uint32)), want)
    dev_outs = [torch.empty(5000, dtype=torch.float32, device="cuda"), torch.empty((5000, 3), dtype=torch.float32, device="cuda"),
                torch.empty(5000, dtype=torch.int32, device="cuda")]
    assert _status(fu, "rr_sample_distance", 0, C.c_void_p(pin_in.data_ptr()), 5000, *[C.c_void_p(t.data_ptr()) for t in dev_outs]) == 0
    _same_query("device outputs", (dev_outs[0].cpu().numpy(), dev_outs[1].cpu().numpy(), dev_outs[2].cpu().numpy().view(np.uint32)), want)
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_equals_single_context(scene2, n):
    from rrpy import capi
    sc, inv = scene2
    pts = _query_points(sc, 20000, seed=5)
    fu = _context(sc, inv)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    want_n = fu.distance_field()
    want = fu.nearest_voxels()
    want_q = fu.sample_distance(pts)
    fu.close()

    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    if n > 1:
        Z = int(g.member(0).volume_res()[2])       # slab boundaries through the middle of the scene, where the objects are
        g.set_slabs([0] + [int(b) for b in np.linspace(Z // 2 - 5, Z // 2 + 5, n - 1)] + [Z])
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    assert g.distance_field() == want_n
    assert np.array_equal(g.nearest_voxels(), want)
    _same_query(f"group of {n}", g.sample_distance(pts), tuple(np.asarray(x) for x in want_q))
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    with pytest.raises(Exception):
        g.sample_distance(pts)                               # the field is of the previous frame set
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_distance(tmp_path, devices):
    """fusion_playback --distance X Y Z over stream files of several frame sets prints Fusion.sample_distance of each."""
    import os
    import subprocess
    from test_host_cpp import BIN, write_scene_files
    from rrpy import capi, synth, volume_io
    first = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    frames = [first] + [synth.rerender(first, 5 * f) for f in range(1, 3)]
    sc = frames[0]
    ks, streams = write_scene_files(str(tmp_path), sc, frames=frames)
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    for i in range(sc.N):
        volume_io.write_volume(str(tmp_path / f"sensor{i}.cv_xyz_inv"), inv[i])
    point = np.array([[0.55, 1.4, 0.3]], np.float32)
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    want = []
    for fr in frames:
        fu.upload_frames(fr.color, fr.depth)
        fu.frame()
        fu.distance_field()
        d, c, v = fu.sample_distance(point)
        want.append((d[0], *c[0], int(v[0])))
    fu.close()
    assert all(np.isfinite(w[0]) and w[4] != NONE for w in want)
    args = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
            "--streams", ";".join(streams), "--frames", str(len(frames)), "--voxel", "0.02", "--view", "64", "64",
            "--distance"] + [repr(float(x)) for x in point[0]] + (["--devices", devices] if devices else [])
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [l.split() for l in r.stdout.splitlines() if l.startswith("frame ") and " distance " in l]
    assert len(lines) == len(frames), r.stdout
    for f, (l, w) in enumerate(zip(lines, want)):
        assert l[1] == str(f) and l[2] == "distance" and l[4] == "nearest" and l[8] == "voxel"
        got = np.array([float(l[3]), float(l[5]), float(l[6]), float(l[7])], np.float32)
        assert bits_equal(got, np.array(w[:4], np.float32)).all(), (l, w)
        assert int(l[9]) == w[4]
