"""Part tracking on the device (rr_track_parts / rr_download_part_tracks / rr_reset_part_tracks / rr_group_track_parts)
against the oracle (oracle/oracle_track.py over oracle_parts.label_parts), bit for bit over sequences of frame sets of
moving objects: two spheres that approach, merge and separate again, and a small sphere that appears and vanishes. The
oracle is fed the volume the context holds after each frame set (the labelling of that volume is pinned to the oracle's
integrate by test_parts_gpu.py)."""
import ctypes as C

import numpy as np
import oracle_track
import pytest

from conftest import bits_equal

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10
GAPS = (0.45, 0.32, 0.19, 0.12, 0.3, 0.45)          # half the distance between the big spheres' centres, per frame set


def moving_sdf(p, frame=0):
    """Two 20 cm spheres at x = +-GAPS[frame] (apart, touching, merged, apart again) and a 12 cm sphere in frames 1 to 3."""
    g = GAPS[int(frame) % len(GAPS)]
    a = np.linalg.norm(p - np.array([g, 1.1, 0.0]), axis=-1) - 0.2
    b = np.linalg.norm(p - np.array([-g, 1.1, 0.05]), axis=-1) - 0.2
    d = np.minimum(a, b)
    if 1 <= int(frame) <= 3:
        d = np.minimum(d, np.linalg.norm(p - np.array([0.1, 1.65, 0.0]), axis=-1) - 0.12)
    return d


def _frames(n_sensors=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), n=len(GAPS)):
    from rrpy import synth
    first = synth.make_scene(N=n_sensors, W=W, H=H, CW=CW, CH=CH, cv_res=cv_res, sdf=moving_sdf)
    return [first] + [synth.rerender(first, f, sdf=moving_sdf) for f in range(1, n)]


@pytest.fixture(scope="module")
def seq2():
    from rrpy import synth
    frames = _frames()
    return frames, synth.analytic_inverse(frames[0], INV_RES)


def _context(sc, inv, use_bricks=True, store_weight=0):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    return fu


def _fuse(fu, fr):
    fu.upload_frames(fr.color, fr.depth)
    fu.frame()


def _same(what, got, want):
    names = ("voxels", "boxes", "centroids", "track_ids", "prev_parts", "overlaps", "ended")
    for n, g, w in zip(names, got, want):
        g = g.cpu().numpy() if hasattr(g, "cpu") else np.asarray(g)
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n == "centroids":
            assert bits_equal(g, w).all(), f"{what}: centroids differ"
        else:
            assert np.array_equal(g, w), f"{what} {n}: {g.tolist()[:12]} != {w.tolist()[:12]}"


def _step(fu, tracker, what, min_voxels=1, labels=True):
    """One track on the context and on the oracle (fed the context's volume); compares, returns the device's outputs."""
    got = fu.track_parts(min_voxels)
    want = tracker.step(fu.download_tsdf(), min_voxels)
    _same(what, got, want[1:])
    if labels:
        assert np.array_equal(fu.part_labels(), want[0]), f"{what}: labels differ"
    return got


def _sequence(fu, frames, sc, what, min_voxels=1):
    tracker = oracle_track.Tracker(sc.bbox_min, sc.bbox_max)
    outs = []
    for f, fr in enumerate(frames):
        _fuse(fu, fr)
        outs.append(_step(fu, tracker, f"{what} frame {f}", min_voxels))
    return outs


def _check_story(outs):
    """What the scene does: the spheres keep their ids while apart, one id ends at the merge and a new one starts at the
    split; the small sphere gets an id and loses it."""
    ids0 = set(outs[0][3].tolist()) - {oracle_track.NONE}
    assert len(ids0) >= 2
    assert sum(len(o[6]) for o in outs) >= 2, "no track ended"
    assert max(int(o[3][o[3] != oracle_track.NONE].max()) for o in outs if len(o[3])) >= 3, "no new track after the first frame set"
    assert any((o[4] != oracle_track.NONE).sum() >= 2 for o in outs[1:]), "nothing was matched"


@pytest.mark.parametrize("mode", ["f32", "f32_weight", "half2", "dense"])
def test_track_matches_oracle(seq2, mode):
    frames, inv = seq2
    fu = _context(frames[0], inv, use_bricks=mode != "dense", store_weight={"f32": 0, "f32_weight": 1, "half2": 2, "dense": 0}[mode])
    outs = _sequence(fu, frames, frames[0], mode)
    if mode != "dense":                                      # dense mode keeps the band between the spheres: one part
        _check_story(outs)
    fu.close()


def test_track_min_voxels(seq2):
    frames, inv = seq2
    fu = _context(frames[0], inv)
    tracker = oracle_track.Tracker(frames[0].bbox_min, frames[0].bbox_max)
    for f, fr in enumerate(frames[:4]):
        _fuse(fu, fr)
        v = fu.label_parts()[0]
        mv = int(np.sort(v)[len(v) // 2]) if len(v) else 1      # at a part's exact size: that part is tracked, smaller are not
        got = _step(fu, tracker, f"min_voxels {mv} frame {f}", mv)
        assert ((got[0] >= mv) == (got[3] != oracle_track.NONE)).all()
    fu.close()


def test_track_eight_sensors():
    from rrpy import synth
    frames = _frames(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48), n=5)
    fu = _context(frames[0], synth.analytic_inverse(frames[0], INV_RES))
    _sequence(fu, frames, frames[0], "8 sensors")
    fu.close()


def test_track_headline_sequence():
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs(n_frames=3)
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    tracker = oracle_track.Tracker(sc.bbox_min, sc.bbox_max)
    for f, s in enumerate(scenes):
        fu.upload_frames(s.color, s.depth)
        fu.fuse_frame()
        got = _step(fu, tracker, f"512^3 frame {f}", 1000)
        assert (got[3] != oracle_track.NONE).sum() >= 1
        if f:
            assert (got[4] != oracle_track.NONE).sum() >= 1
    assert tuple(fu.volume_res()) == (512, 512, 512)
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "configure_limit"])
def test_track_with_stale_brick_tables(seq2, order):
    """The brick tables no longer describe the volume: the whole volume is visited; a new limit keeps the tracks."""
    frames, inv = seq2
    sc = frames[0]
    fu = _context(sc, inv)
    tracker = oracle_track.Tracker(sc.bbox_min, sc.bbox_max)
    for f in range(2):
        _fuse(fu, frames[f])
        _step(fu, tracker, f"{order} frame {f}")
    if order == "bricks_update_other":
        fu.upload_frames(frames[4].color, frames[4].depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
    else:
        fu.configure(limit=0.02, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    got = _step(fu, tracker, order)
    assert (got[4] != oracle_track.NONE).sum() >= 2          # the tracks continue
    fu.close()


def test_same_volume_twice_is_the_identity(seq2):
    frames, inv = seq2
    fu = _context(frames[0], inv)
    _fuse(fu, frames[1])
    a = fu.track_parts()
    b = fu.track_parts()
    assert np.array_equal(a[3], b[3]) and np.array_equal(b[4], np.arange(len(b[0]), dtype=np.uint32))
    assert np.array_equal(b[5], b[0]) and len(b[6]) == 0
    fu.close()


def test_labelling_between_tracks_changes_nothing(seq2):
    """rr_label_parts, rr_extract_mesh and rr_download_mesh_parts between two tracks: the second track is as without them,
    and after a track rr_download_parts and the mesh parts are those of rr_label_parts."""
    frames, inv = seq2
    runs = []
    for between in (False, True):
        fu = _context(frames[0], inv)
        _fuse(fu, frames[1])
        first = fu.track_parts()
        after = (fu.part_labels(),) + fu.download_parts(len(first[0]))
        fu.extract_mesh()
        mp_track = fu.mesh_parts()
        lab = fu.label_parts()
        for x, y in zip(after[1:], lab):
            assert bits_equal(x, y).all() if x.dtype.kind == "f" else np.array_equal(x, y)
        assert np.array_equal(after[0], fu.part_labels())
        for x, y in zip(mp_track, fu.mesh_parts()):
            assert np.array_equal(x, y)
        _fuse(fu, frames[2])
        if between:
            fu.label_parts()
            fu.extract_mesh()
            fu.mesh_parts()
            fu.label_parts()
        second = fu.track_parts()
        # the downloads stay those of the last track whatever labelling follows
        fu.label_parts()
        again = fu.download_part_tracks(len(second[0]), len(second[6]))
        for x, y in zip(again, second[3:]):
            assert np.array_equal(x, y)
        runs.append(second)
        fu.close()
    _same("label between", runs[1], tuple(np.asarray(x) for x in runs[0]))


def test_reset_and_settings(seq2):
    from rrpy import capi
    frames, inv = seq2
    fu = _context(frames[0], inv)
    _fuse(fu, frames[0])
    first = fu.track_parts()
    _fuse(fu, frames[1])
    fu.track_parts()
    n_before = int(first[3].max())
    fu.configure(limit=0.02, voxel_size=VOXEL, brick_size=0.08, min_voxels=MIN_VOX, use_bricks=True)   # limit, brick size
    kept = fu.track_parts()                                  # the same volume: every track continues
    assert (kept[4] != oracle_track.NONE).all() and np.array_equal(kept[5], kept[0])
    fu.reset_part_tracks()
    assert fu.L.rr_download_part_tracks(fu.h, None, None, None, None) == -1
    again = fu.track_parts()
    assert np.array_equal(again[3], np.arange(len(again[0]), dtype=np.uint32)) and len(again[6]) == 0
    assert (again[4] == oracle_track.NONE).all()
    # a new voxel size is a new volume: nothing integrated, nothing tracked, ids from 0
    fu.configure(limit=LIMIT, voxel_size=0.025, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    assert fu.L.rr_download_part_tracks(fu.h, None, None, None, None) == -1
    _fuse(fu, frames[0])
    fresh = fu.track_parts()
    assert np.array_equal(fresh[3], np.arange(len(fresh[0]), dtype=np.uint32)) and n_before >= 1
    # a new voxel format too
    fu.configure(limit=LIMIT, voxel_size=0.025, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True, store_weight=capi.VOXELS_HALF2)
    assert fu.L.rr_download_part_tracks(fu.h, None, None, None, None) == -1
    fu.close()


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


def test_track_refusals(seq2):
    frames, inv = seq2
    fu = _context(frames[0], inv)
    n, e = C.c_uint32(), C.c_uint32()
    assert _status(fu, "rr_track_parts", 1, C.byref(n), C.byref(e)) == -1                 # nothing integrated yet
    assert _status(fu, "rr_download_part_tracks", None, None, None, None) == -1            # nothing tracked yet
    _fuse(fu, frames[0])
    assert _status(fu, "rr_track_parts", 0, C.byref(n), C.byref(e)) == -1                 # min_voxels 0
    assert _status(fu, "rr_track_parts", 1, None, C.byref(e)) == -1                       # null count pointers
    assert _status(fu, "rr_track_parts", 1, C.byref(n), None) == -1
    assert _status(fu, "rr_download_part_tracks", None, None, None, None) == -1
    fu.label_parts()
    assert _status(fu, "rr_download_part_tracks", None, None, None, None) == -1            # labelling is not tracking
    assert _status(fu, "rr_track_parts", 1, C.byref(n), C.byref(e)) == 0 and n.value > 0
    assert _status(fu, "rr_download_part_tracks", None, None, None, None) == 0
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_track_parts", 1, C.byref(n), C.byref(e)) == -1
    assert "rr_group_track_parts" in fu.L.rr_last_error(fu.h).decode()
    assert _status(fu, "rr_download_part_tracks", None, None, None, None) == 0             # the last tracking stays
    assert fu.L.rr_track_parts(None, 1, C.byref(n), C.byref(e)) == -1
    assert fu.L.rr_reset_part_tracks(None) == -1
    fu.close()


def test_track_has_no_side_effects(seq2):
    """Against a twin context that never tracks: volume, brick tables, view, fill_colors, mesh, simplified mesh and cloud;
    after the next fused frame (a replayed graph) the volume, the launches per frame and rr_integrator_last."""
    from rrpy import synth
    frames, inv = seq2
    sc = frames[0]
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    runs = []
    for track in (False, True):
        fu = _context(sc, inv)
        fu.upload_frames(frames[1].color, frames[1].depth)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        mesh = fu.extract_mesh()
        simple = fu.simplify_mesh(2)
        cloud = fu.extract_points()
        if track:
            fu.track_parts()
            fu.track_parts(5)
        out = dict(view=view, tsdf=fu.download_tsdf(), bricks=fu.download_bricks(), fill=fu.fill_colors(),
                   mesh=fu.download_mesh(len(mesh[0]), len(mesh[3])), cloud=fu.download_points(len(cloud[0])),
                   simple=fu.download_simplified_mesh(len(simple[0]), len(simple[3])))
        fu.upload_frames(frames[2].color, frames[2].depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        out["per_frame"], out["next_frame"] = (per_frame, fu.launch_count() - l0), fu.download_tsdf()
        out["last"] = fu.integrator_last()
        runs.append(out)
        fu.close()
    a, b = runs
    for key in ("view", "mesh", "cloud", "bricks", "simple"):
        for x, y in zip(a[key], b[key]):
            assert (bits_equal(x, y).all() if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y)), key
    for key in ("tsdf", "next_frame", "fill"):
        assert bits_equal(a[key], b[key]).all(), key
    assert a["per_frame"] == b["per_frame"] and b["per_frame"][0] == b["per_frame"][1]
    assert a["last"] == b["last"]


def test_track_buffers_grow(seq2):
    """Few parts, then many (twenty spheres), then few again: the pair, flag and id buffers grow and every step is right."""
    from rrpy import synth
    frames, inv = seq2
    sc = frames[0]
    rng = np.random.default_rng(5)
    centres = np.stack([rng.uniform(-0.7, 0.7, 20), rng.uniform(0.3, 1.9, 20), rng.uniform(-0.7, 0.7, 20)], 1)

    def many(p, frame=0):
        d = np.full(p.shape[:-1], np.inf)
        for c in centres:
            d = np.minimum(d, np.linalg.norm(p - c - np.array([0.02 * frame, 0.0, 0.0]), axis=-1) - 0.15)
        return d
    seq = [frames[0], synth.rerender(sc, 0, sdf=many), synth.rerender(sc, 1, sdf=many), frames[1]]
    fu = _context(sc, inv)
    outs = _sequence(fu, seq, sc, "grow")
    assert len(outs[2][0]) > len(outs[0][0]) + 5 and (outs[2][4] != oracle_track.NONE).sum() > 5
    fu.close()


def test_cuda_tensor_and_pinned_outputs(seq2):
    import torch
    frames, inv = seq2
    fu = _context(frames[0], inv)
    _fuse(fu, frames[0])
    fu.track_parts()
    _fuse(fu, frames[3])
    host = fu.track_parts()
    n, e = len(host[0]), len(host[6])
    dev = fu.download_part_tracks(n, e, device=True)
    for d, h in zip(dev, host[3:]):
        assert isinstance(d, torch.Tensor) and d.is_cuda and np.array_equal(d.cpu().numpy(), h)
    pinned = [torch.empty(k, dtype=torch.int32).pin_memory() for k in (n, n, n, max(e, 1))]
    assert _status(fu, "rr_download_part_tracks", *[C.c_void_p(t.data_ptr()) for t in pinned]) == 0
    for t, h in zip(pinned, host[3:]):
        assert np.array_equal(t.numpy().view(np.uint32)[:len(h)], h)
    assert e >= 1                                            # the merge ends a track
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_track_equals_single_context(seq2, n):
    from rrpy import capi
    frames, inv = seq2
    sc = frames[0]
    fu = _context(sc, inv)
    want = []
    for fr in frames:
        fu.upload_frames(fr.color, fr.depth)
        fu.fuse_frame()
        want.append(fu.track_parts())
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
    for f, fr in enumerate(frames):
        g.upload_frames(fr.color, fr.depth)
        g.fuse_frame()
        _same(f"group of {n} frame {f}", g.track_parts(), want[f])
    g.reset_part_tracks()
    again = g.track_parts()
    assert np.array_equal(again[3], np.arange(len(again[0]), dtype=np.uint32))
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_track_parts(tmp_path, seq2, devices):
    """fusion_playback --track-parts N over stream files of several frame sets prints Fusion.track_parts(N) of each."""
    import os
    import subprocess
    from test_host_cpp import BIN, write_scene_files
    from rrpy import capi, synth, volume_io
    frames, _ = seq2
    sc = frames[0]
    ks, streams = write_scene_files(str(tmp_path), sc, frames=frames)
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    for i in range(sc.N):
        volume_io.write_volume(str(tmp_path / f"sensor{i}.cv_xyz_inv"), inv[i])
    mv = 20
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    want = []
    for f, fr in enumerate(frames):
        fu.upload_frames(fr.color, fr.depth)
        fu.frame()
        voxels, _, _, ids, prev, ovl, ended = fu.track_parts(mv)
        want += [f"frame {f} part {k} track {ids[k]} voxels {voxels[k]} prev {prev[k]} overlap {ovl[k]}"
                 for k in range(len(voxels)) if ids[k] != oracle_track.NONE]
        want += [f"frame {f} ended {t}" for t in ended]
    fu.close()
    assert any(" ended " in w for w in want)
    args = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
            "--streams", ";".join(streams), "--frames", str(len(frames)), "--voxel", "0.02", "--view", "64", "64",
            "--track-parts", str(mv)] + (["--devices", devices] if devices else [])
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert [l for l in r.stdout.splitlines() if l.startswith("frame ")] == want
