"""Removing connected parts from the volume on the device (rr_remove_parts / rr_group_remove_parts) against the oracle
(oracle/oracle_remove.py on the labels of scipy.ndimage.label), bit for bit: the volume and weight volume after the
removal, the counts, the consumers of the removed volume (view, mesh, labelling), what follows a removal (the next fuses,
the incremental clear, tracking), keep flags in host, pinned and device memory, refusals, the epoch rule, side effects
against a twin context, groups and fusion_playback."""
import ctypes as C
import math

import numpy as np
import oracle_parts
import oracle_remove
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10


@pytest.fixture(scope="module")
def scene2():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    return sc, synth.analytic_inverse(sc, INV_RES)


def _context(sc, inv, use_bricks=True, store_weight=0, frame=True, voxel=VOXEL):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=voxel, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame()
    return fu


def _volume(fu, store_weight):
    return fu.download_tsdf(), (fu.download_weight() if store_weight in (1, 2) else None)


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


def _check_removal(fu, what, store_weight=0, min_voxels=0, keep=None, limit=LIMIT):
    """Label, remove, and hold the volume, weight volume and counts to the oracle on the volume before the removal. Returns
    (voxels of the labelling, removed flags, volume after)."""
    tsdf, weight = _volume(fu, store_weight)
    voxels, _, _ = fu.label_parts()
    labels, w_voxels, _, _ = oracle_parts.label_parts(tsdf, (0, 0, 0), (1, 1, 1))
    assert np.array_equal(voxels, w_voxels), f"{what}: labelling differs from the oracle"
    got_counts = fu.remove_parts(min_voxels, keep)
    want_t, want_w, k, v = oracle_remove.remove_parts(tsdf, limit, store_weight, min_voxels, keep, weight, labels, voxels)
    assert got_counts == (k, v), f"{what}: counts {got_counts} != {(k, v)}"
    got_t, got_w = _volume(fu, store_weight)
    assert bits_equal(got_t, want_t).all(), mismatch_report(f"{what} tsdf", got_t, want_t)
    if want_w is not None:
        assert bits_equal(got_w, want_w).all(), mismatch_report(f"{what} weight", got_w, want_w)
    return voxels, oracle_remove.removed_flags(voxels, min_voxels, keep), got_t


def _floater_threshold(voxels):
    """A threshold that removes some parts and keeps others (the largest always stays)."""
    s = np.sort(voxels)
    return int(s[len(s) // 2]) + 1 if len(s) > 1 else 0


@pytest.mark.parametrize("store_weight,use_bricks", [(0, True), (1, True), (2, True), (0, False)])
def test_removal_matches_oracle(scene2, store_weight, use_bricks):
    sc, inv = scene2
    fu = _context(sc, inv, use_bricks=use_bricks, store_weight=store_weight, frame=False)
    fu.fuse_frame()
    fu.fuse_frame()                                                  # the captured graph's replay
    voxels, _, _ = fu.label_parts()
    assert len(voxels) >= 2, "the scene should hold several parts"
    _, flags, _ = _check_removal(fu, f"format {store_weight} bricks {use_bricks}", store_weight, _floater_threshold(voxels))
    assert 0 < flags.sum() < len(flags)
    fu.close()


def _three_objects(p, frame=0):
    a = np.linalg.norm(p - np.array([0.5, 1.1, 0.0]), axis=-1) - 0.25
    b = np.linalg.norm(p - np.array([-0.5, 1.1, 0.0]), axis=-1) - 0.25
    c = np.linalg.norm(p - np.array([0.0, 1.6, 0.0]), axis=-1) - 0.05
    return np.minimum(np.minimum(a, b), c)


@pytest.fixture(scope="module")
def three():
    from rrpy import synth
    sc = synth.make_scene(N=4, W=512, H=424, CW=640, CH=540, cv_res=(32, 32, 64), sdf=_three_objects)
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("which", ["none", "some", "all"])
def test_three_objects(three, which):
    sc, inv = three
    fu = _context(sc, inv)
    voxels, _, _ = fu.label_parts()
    big = np.sort(voxels)[-3:]                                       # the two big spheres and the small one are the largest
    th = dict(none=0, some=int(big[0]) + 1, all=int(voxels.max()) + 1)[which]
    _, flags, after = _check_removal(fu, f"three objects, {which}", 0, th)
    assert flags.sum() == dict(none=0, some=len(voxels) - 2, all=len(voxels))[which]
    if which == "all":
        assert not oracle_parts.inside(after).any()
        assert fu.label_parts_count() == 0
    fu.close()


def test_removal_eight_sensors():
    from rrpy import synth
    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv)
    voxels, _, _ = fu.label_parts()
    _check_removal(fu, "8 sensors", 0, _floater_threshold(voxels))
    fu.close()


def test_removal_headline_frame_set():
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs()
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    assert tuple(fu.volume_res()) == (512, 512, 512)
    voxels, _, _ = fu.label_parts()
    _check_removal(fu, "512^3 floaters", 0, 64, limit=bench.LIMIT)
    fu.fuse_frame()
    voxels, _, _ = fu.label_parts()
    keep = np.zeros(len(voxels), np.uint8)
    keep[int(np.argmax(voxels))] = 1                                 # keep only the largest part (the floaters go)
    _check_removal(fu, "512^3 keep only", 0, 0, keep, limit=bench.LIMIT)
    fu.fuse_frame()
    voxels, boxes, _ = fu.label_parts()
    big = int(np.argmax(voxels))
    keep = np.ones(len(voxels), bool)
    keep[big] = False                                                # remove the subject: a box of millions of voxels
    assert np.prod((boxes[big, 1::2] - boxes[big, 0::2]).astype(np.int64)) > 1000000
    _check_removal(fu, "512^3 largest", 0, 0, keep, limit=bench.LIMIT)
    fu.close()


def test_removal_with_stale_brick_tables(scene2):
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    other = synth.rerender(sc, 7)
    fu.upload_frames(other.color, other.depth)
    fu.bricks_clear()
    fu.preprocess()
    fu.bricks_update()
    voxels, _, _ = fu.label_parts()
    keep = (np.arange(len(voxels)) % 2).astype(np.uint8)
    _check_removal(fu, "stale tables", 0, 0, keep)
    fu.close()


def test_removal_of_an_empty_frame_set(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.upload_frames(sc.color, np.zeros_like(sc.depth))
    fu.frame()
    before = fu.download_tsdf()
    assert fu.label_parts_count() == 0
    assert fu.remove_parts(100) == (0, 0)
    assert fu.remove_parts(1, np.zeros(0, np.uint8)) == (0, 0)
    assert bits_equal(fu.download_tsdf(), before).all()
    fu.close()


def test_consumers_see_the_removed_volume(scene2):
    """The view equals the raymarch oracle over the removed volume, the mesh the mesh oracle, and a new labelling gives the
    kept parts with their voxel counts."""
    import oracle_mesh
    import oracle_py as O
    from rrpy import synth
    from test_raymarch_gpu import _compare
    sc, inv = scene2
    fu = _context(sc, inv)
    fu.frame(sync_bricks=True)
    voxels, flags, after = _check_removal(fu, "consumers", 0, _floater_threshold(fu.label_parts()[0]))
    pre = dict(depth_b=fu.download_stage("depth_b"), quality=fu.download_stage("quality"))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
    _, occupied = fu.download_bricks()
    exact, _ = _compare(sc, fu, dict(tsdf=after, inv=inv, pre=pre, grid=grid, occ=occupied), (1.4, 1.5, 2.0), 1, True)
    assert exact, "the view differs from the raymarch oracle over the removed volume"
    got = fu.extract_mesh()
    want = oracle_mesh.extract_mesh(after, fu.volume_res(), LIMIT, inv, sc, pre, sc.bbox_min, sc.bbox_max)
    for name, g, w in zip(("positions", "normals", "rgba", "triangles"), got, want):
        assert g.shape == w.shape and bits_equal(g, w).all(), f"mesh {name} differs from the oracle"
    kept, _, _ = fu.label_parts()
    assert np.array_equal(kept, voxels[~flags])
    o = np.tile(np.asarray(sc.bbox_min, np.float32) - 0.5, (16, 1))
    d = np.tile(np.float32([1.0, 1.0, 1.0]), (16, 1))
    assert fu.cast_rays(o, d)[0].shape == (16, 3)
    fu.close()


@pytest.mark.parametrize("path", ["fuse_frame", "frame"])
def test_fusing_after_removal_equals_a_twin(scene2, path):
    """fuse, label, remove, fuse, ...: after every fuse the volume equals a twin's that never removes, and the staged
    integrate after a removal still runs the incremental clear."""
    from rrpy import synth
    sc, inv = scene2
    frames = [sc, synth.rerender(sc, 3), synth.rerender(sc, 6), sc]
    a, b = _context(sc, inv, frame=False), _context(sc, inv, frame=False)
    for k, f in enumerate(frames):
        for fu in (a, b):
            fu.upload_frames(f.color, f.depth)
            getattr(fu, path)()
        assert bits_equal(a.download_tsdf(), b.download_tsdf()).all(), f"step {k}: the volume differs from the twin's"
        if k > 0:
            assert a.integrator_last()["clear"] == "incremental", f"step {k}: the incremental clear did not run after a removal"
        voxels, _, _ = a.label_parts()
        _check_removal(a, f"step {k}", 0, _floater_threshold(voxels))
    a.close()
    b.close()


def test_tracks_of_removed_parts_end(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    voxels, _, _, ids, _, _, _ = fu.track_parts(1)
    th = _floater_threshold(voxels)
    gone = voxels < th
    got = fu.remove_parts(th)
    assert got == (int(gone.sum()), int(voxels[gone].sum()))
    tracks_after = fu.track_parts(1)            # the removed volume, tracked against the labelling before the removal
    assert sorted(tracks_after[6].tolist()) == sorted(ids[gone].tolist())
    assert np.array_equal(tracks_after[3], ids[~gone])
    fu.fuse_frame()
    fu.track_parts(1)
    fu.close()


def test_keep_in_host_pinned_and_device_memory(scene2):
    import torch
    sc, inv = scene2
    results = []
    for kind in ("numpy", "bool", "pinned", "cuda"):
        fu = _context(sc, inv)
        voxels, _, _ = fu.label_parts()
        k = (np.arange(len(voxels)) % 3 != 1).astype(np.uint8)
        keep = dict(numpy=k, bool=k.astype(bool), pinned=torch.from_numpy(k).pin_memory(),
                    cuda=torch.from_numpy(k).cuda())[kind]
        counts = fu.remove_parts(0, keep)
        results.append((counts, fu.download_tsdf()))
        fu.close()
    for counts, t in results[1:]:
        assert counts == results[0][0] and bits_equal(t, results[0][1]).all()
    assert results[0][0][0] > 0
    # the library reads one byte per part: another length or element type is refused before the call
    fu = _context(sc, inv)
    n = fu.label_parts_count()
    for bad in (np.ones(n + 1, np.uint8), np.ones(max(0, n - 1), np.uint8), np.ones(n, np.int32),
                torch.ones(n, dtype=torch.int32), torch.ones(n + 1, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            fu.remove_parts(0, bad)
    fresh = _context(sc, inv)
    with pytest.raises(ValueError):                                  # no labelling through this object yet
        fresh.remove_parts(0, np.ones(n, np.uint8))
    fresh.close()
    assert fu.remove_parts(0, np.ones(n, np.uint8)) == (0, 0)
    fu.close()


def test_refusals_and_epochs(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    p, v = C.c_uint32(), C.c_uint32()
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), C.byref(v)) == -1      # nothing integrated, nothing labelled
    fu.frame()
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), C.byref(v)) == -1      # no labelling
    voxels, _, _ = fu.label_parts()
    assert _status(fu, "rr_remove_parts", 1, None, None, C.byref(v)) == -1            # null counts
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), None) == -1
    fu.frame()
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), C.byref(v)) == -1      # a labelling older than an integrate
    fu.label_parts()
    assert _status(fu, "rr_remove_parts", 0, None, C.byref(p), C.byref(v)) == 0 and p.value == 0
    assert _status(fu, "rr_remove_parts", 0, None, C.byref(p), C.byref(v)) == 0       # nothing removed: the labelling stands
    fu.extract_mesh()
    fu.distance_field()
    assert _status(fu, "rr_download_mesh_parts", None, None) == 0
    assert fu.sample_distance(np.zeros((1, 3), np.float32))[0].shape == (1,)
    assert fu.remove_parts(_floater_threshold(voxels))[0] > 0
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), C.byref(v)) == -1      # the labelling is of the state before
    with pytest.raises(Exception):
        fu.sample_distance(np.zeros((1, 3), np.float32))                            # the field is of the state before
    fu.extract_mesh()
    assert _status(fu, "rr_download_mesh_parts", None, None) == -1                   # mesh after, labelling before
    fu.label_parts()
    assert _status(fu, "rr_download_mesh_parts", None, None) == 0
    fu.distance_field()
    fu.sample_distance(np.zeros((1, 3), np.float32))
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_remove_parts", 1, None, C.byref(p), C.byref(v)) == -1
    assert "rr_group_remove_parts" in fu.L.rr_last_error(fu.h).decode()
    fu.close()


def test_removal_has_no_side_effects(scene2):
    """Against a twin context that never removes: brick tables, stage images, view, fill_colors, cloud, tracking state and
    rr_integrator_last, then the next fused frame."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 3)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    runs = []
    for remove in (False, True):
        fu = _context(sc, inv, frame=False)
        fu.fuse_frame()
        fu.fuse_frame()
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        cloud = fu.extract_points()
        voxels, _, _, ids, _, _, _ = fu.track_parts(1)
        if remove:
            assert fu.remove_parts(_floater_threshold(voxels))[0] > 0
        out = dict(view=view, bricks=fu.download_bricks(), fill=fu.fill_colors(), cloud=fu.download_points(len(cloud[0])),
                   stage=fu.download_stage("quality"), last=fu.integrator_last(), cleared=fu.integrator_cleared(),
                   tracks=fu.download_part_tracks(len(ids), 0))
        fu.upload_frames(other.color, other.depth)
        fu.fuse_frame()
        out["next_frame"], out["next_last"] = fu.download_tsdf(), fu.integrator_last()
        out["next_tracks"] = fu.track_parts(1)
        runs.append(out)
        fu.close()
    a, b = runs
    for key in ("view", "cloud", "bricks", "tracks"):
        for x, y in zip(a[key], b[key]):
            assert (bits_equal(x, y).all() if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y)), key
    for key in ("fill", "stage", "next_frame"):
        assert bits_equal(a[key], b[key]).all(), key
    assert a["last"] == b["last"] and a["next_last"] == b["next_last"] and a["cleared"] == b["cleared"]
    # the next tracking: the same parts; ids continue from the same next_id, the removed parts' tracks have ended
    assert np.array_equal(a["next_tracks"][0], b["next_tracks"][0])


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


def _removal_args(voxels, which):
    """(min_voxels, keep) of a removal: the floaters, or the largest part alone (a box across the slab boundaries)."""
    if which == "floaters":
        return _floater_threshold(voxels), None
    keep = np.ones(len(voxels), np.uint8)
    keep[int(np.argmax(voxels))] = 0
    return 0, keep


@pytest.mark.parametrize("which", ["floaters", "largest"])
@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_removal_equals_single_context(scene2, n, which):
    from rrpy import capi, synth
    sc, inv = scene2
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    voxels, boxes, _ = fu.label_parts()
    args = _removal_args(voxels, which)
    counts = fu.remove_parts(*args)
    assert counts[0] > 0
    want_t = fu.download_tsdf()
    want_view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
    rng = np.random.default_rng(5)
    o = np.tile(np.float32([1.4, 1.5, 2.0]), (4096, 1))
    d = (rng.uniform(-0.5, 0.5, (4096, 3)) + np.float32([-1.4, -0.4, -2.0])).astype(np.float32)
    want_rays = fu.cast_rays(o, d)
    want_mesh = fu.extract_mesh()
    fu.close()

    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    Z = int(g.member(0).volume_res()[2])
    if n > 1:
        g.set_slabs([0] + [int(b) for b in np.linspace(Z // 2 - 5, Z // 2 + 5, n - 1)] + [Z])
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    g_voxels, g_boxes, _ = g.label_parts()
    assert np.array_equal(g_voxels, voxels)
    assert g.remove_parts(*args) == counts
    bounds = g.slabs()
    if n > 1 and which == "largest":
        big = int(np.argmax(voxels))
        assert any(boxes[big, 4] < b < boxes[big, 5] for b in bounds[1:-1]), "the removed part crosses no slab boundary"
    halo = math.ceil(np.float32(LIMIT) * np.float32(Z)) + 2 if n > 1 else 0
    for i in range(n):
        z0, z1 = max(0, int(bounds[i]) - halo), min(Z, int(bounds[i + 1]) + halo)
        t = g.member(i).download_tsdf()
        assert bits_equal(t[z0:z1], want_t[z0:z1]).all(), mismatch_report(f"member {i} rows {z0}..{z1}", t[z0:z1], want_t[z0:z1])
    assert bits_equal(g.download_tsdf(), want_t).all()
    for x, y in zip(g.raymarch(mv, pr, 200, 120, shade_mode=1), want_view):
        assert bits_equal(x, y).all(), "group view"
    for x, y in zip(g.cast_rays(o, d), want_rays):
        assert bits_equal(x, y).all() if x.dtype.kind == "f" else np.array_equal(x, y), "group rays"
    for x, y in zip(g.extract_mesh(), want_mesh):
        assert bits_equal(x, y).all() if x.dtype.kind == "f" else np.array_equal(x, y), "group mesh"
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_remove_parts(tmp_path, small_scene, devices):
    """fusion_playback --remove-parts N prints the counts of label_parts + remove_parts per frame set, and --dump-tsdf writes
    the oracle's removed volume."""
    import os
    import subprocess
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
    tsdf = fu.download_tsdf()
    voxels, _, _ = fu.label_parts()
    fu.close()
    th = _floater_threshold(voxels)
    want_t, _, k, v = oracle_remove.remove_parts(tsdf, 0.01, 0, th)
    assert k > 0
    out = str(tmp_path / "tsdf.bin")
    args = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
            "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", "64", "64", "--remove-parts", str(th),
            "--dump-tsdf", out] + (["--devices", devices] if devices else [])
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if " removed " in l]
    assert lines == [f"frame {f} removed {k} parts {v} voxels" for f in range(2)]
    got = np.fromfile(out, np.float32).reshape(want_t.shape)
    assert bits_equal(got, want_t).all(), mismatch_report("--dump-tsdf", got, want_t)
