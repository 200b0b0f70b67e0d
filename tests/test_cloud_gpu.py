"""The point-cloud export on the device (rr_extract_points / rr_download_points / rr_group_extract_points) against the oracle's
scalar restatement (oracle/ro_cloud.cpp), bit for bit: counts, positions, normals, colours, quality and pixel ids. The oracle
extracts from its own pre-process where the scene is small, and from the stage images the context holds at full size."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import oracle_cloud
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10
NAMES = ("positions", "normals", "colors", "quality", "pixels")


def _same_cloud(what, got, want, min_points=1):
    for n, g, w in zip(NAMES, got, want):
        g = g.cpu().numpy() if hasattr(g, "cpu") else g
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n == "pixels":
            assert g.dtype == np.uint32 and np.array_equal(g, w), f"{what} pixels differ"
        else:
            assert bits_equal(g, w).all(), mismatch_report(f"{what} {n}", g, w)
    assert len(want[4]) >= min_points, f"{what}: only {len(want[4])} points"


def _oracle_pre(sc, flags=(True, True, True), compress=None):
    import oracle_py as O
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    return O.preprocess(sc, grid, cams, *flags, compress=compress)


def _stages(fu):
    """The stage images the context holds now, as the oracle takes them."""
    return {k: fu.download_stage(k) for k in ("depth_b", "normal", "quality")}


def _context(sc, inv, frame=True, flags=(True, True, True)):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame(*flags)
    return fu


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


@pytest.fixture(scope="module")
def scene2(small_scene):
    from rrpy import synth
    return small_scene, synth.analytic_inverse(small_scene, INV_RES)


@pytest.fixture(scope="module")
def scene8():
    from rrpy import synth
    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("flags", [(f, p, r) for f in (True, False) for p in (True, False) for r in (True, False)])
def test_cloud_matches_oracle_small_scene(scene2, flags):
    sc, inv = scene2
    fu = _context(sc, inv, flags=flags)
    got = fu.extract_points()
    want = oracle_cloud.extract_points_scene(sc, _oracle_pre(sc, flags))
    _same_cloud(f"flags {flags}", got, want, min_points=1000)
    assert set(np.unique(got[4] // (sc.W * sc.H))) == {0, 1}
    fu.close()


def test_cloud_eight_sensors_and_masks(scene8):
    sc, inv = scene8
    fu = _context(sc, inv)
    pre = _oracle_pre(sc)
    full = fu.extract_points()
    _same_cloud("8 sensors", full, oracle_cloud.extract_points_scene(sc, pre), min_points=2000)
    assert len(np.unique(full[4] // (sc.W * sc.H))) == 8
    for sensors in ([3], [7], [0, 2, 5, 7], [1, 6]):
        mask = sum(1 << s for s in sensors)
        _same_cloud(f"sensors {sensors}", fu.extract_points(sensors), oracle_cloud.extract_points_scene(sc, pre, mask), min_points=20)
    empty = fu.extract_points([])
    assert [len(a) for a in empty] == [0] * 5 and empty[0].shape == (0, 3)
    fu.close()


@pytest.mark.parametrize("fmt", ["dxt1", "dxt5", "depth8"])
def test_cloud_frame_formats(fmt):
    import oracle_py as O
    from rrpy import capi, synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=136, cv_res=(32, 32, 64))     # colour size: multiples of 4
    inv = synth.analytic_inverse(sc, INV_RES)
    near_far = np.float32([[0.5, 4.5]] * sc.N)
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    color, depth, flags, compress = sc.color, sc.depth, (True, True, True), None
    if fmt == "dxt1":
        packed = np.stack([synth.encode_dxt1(sc.color[i]) for i in range(sc.N)])
        fu.set_frame_format(dxt1_color=True)
        fu.upload_frames(packed, sc.depth)
        color = np.stack([O.decode_dxt1(packed[i], sc.CW, sc.CH) for i in range(sc.N)])
    elif fmt == "dxt5":
        packed = np.stack([synth.encode_dxt5(sc.color[i], seed=i) for i in range(sc.N)])
        fu.set_frame_format(dxt5_color=True)
        fu.upload_frames(packed, sc.depth)
        color = np.stack([O.decode_dxt5(packed[i], sc.CW, sc.CH) for i in range(sc.N)])
    else:
        d8 = np.stack([synth.encode_depth8(sc.depth[i], 0.5, 4.5) for i in range(sc.N)])
        fu.set_frame_format(depth8=True, near_far=near_far)
        fu.upload_frames(sc.color, d8)
        depth, flags, compress = O.depth8_to_float(d8), (True, False, True), near_far
    fu.frame(*flags)
    got = fu.extract_points()
    osc = dataclasses.replace(sc, color=color, depth=depth)
    want = oracle_cloud.extract_points_scene(osc, _oracle_pre(osc, flags, compress))
    _same_cloud(fmt, got, want, min_points=1000)
    fu.close()


def test_cloud_headline_frame_set():
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs()
    sc = scenes[0]
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    got = fu.extract_points()
    want = oracle_cloud.extract_points_scene(sc, _stages(fu))
    _same_cloud("headline", got, want, min_points=100000)
    fu.close()


@pytest.mark.parametrize("order", ["fuse_frame_replays", "staged_calls"])
def test_cloud_after_call_orders(scene2, order):
    """After rr_fuse_frame graph replays, and after the four calls of the staged per-frame order: the cloud of the last
    frame set's pre-process."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 7)
    fu = _context(sc, inv, frame=False)
    if order == "fuse_frame_replays":
        fu.fuse_frame()
        fu.fuse_frame()
        fu.upload_frames(other.color, other.depth)
        fu.fuse_frame()                       # a replay of the captured graph on other frames
    else:
        fu.frame()
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
        fu.integrate()
    _same_cloud(order, fu.extract_points(), oracle_cloud.extract_points_scene(other, _oracle_pre(other)), min_points=1000)
    fu.close()


def test_cloud_refusals(scene2):
    from rrpy import capi
    sc, inv = scene2
    n = C.c_uint32(7)
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    assert _status(fu, "rr_download_points", None, None, None, None, None) == -1      # nothing extracted yet
    assert _status(fu, "rr_extract_points", 1, C.byref(n)) == -1                      # no calibration
    assert _status(fu, "rr_extract_points", 0, C.byref(n)) == 0 and n.value == 0      # an empty mask needs nothing
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    assert _status(fu, "rr_extract_points", 3, C.byref(n)) == -1                      # before any pre-process
    assert "rr_preprocess" in fu.L.rr_last_error(fu.h).decode()
    fu.preprocess()
    assert _status(fu, "rr_extract_points", 1 << 2, C.byref(n)) == -1                 # sensor 2 of 2
    assert _status(fu, "rr_extract_points", 1 << 31, C.byref(n)) == -1
    assert _status(fu, "rr_extract_points", 3, None) == -1                            # no count pointer
    with pytest.raises(ValueError):
        fu.extract_points([-1])
    with pytest.raises(capi.RRError):
        fu.extract_points([5])
    assert _status(fu, "rr_extract_points", 3, C.byref(n)) == 0 and n.value > 1000
    assert _status(fu, "rr_download_points", None, None, None, None, None) == 0
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)                                       # a slab context has every stage image
    assert _status(fu, "rr_extract_points", 3, C.byref(n)) == 0 and n.value > 1000
    fu.close()
    # a missing calibration for a sensor of the mask
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame()
    fu2 = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    fu2.set_bbox(sc.bbox_min, sc.bbox_max)
    fu2.calib_upload(0, sc.cv_xyz[0], sc.cv_uv[0])
    assert _status(fu2, "rr_extract_points", 2, C.byref(n)) == -1
    assert "calibration" in fu2.L.rr_last_error(fu2.h).decode()
    fu2.close()
    fu.close()


def test_cloud_buffers_grow(scene8):
    """A large cloud, a small one, a large one again: the buffers grow once, shrink never, and every cloud is right."""
    sc, inv = scene8
    fu = _context(sc, inv)
    pre = _oracle_pre(sc)
    for sensors in ([2], None, [5], None, [0, 1]):
        mask = None if sensors is None else sum(1 << s for s in sensors)
        _same_cloud(f"sensors {sensors}", fu.extract_points(sensors), oracle_cloud.extract_points_scene(sc, pre, mask), min_points=100)
    fu.close()


def test_cloud_has_no_side_effects(scene2):
    """The volume, brick lists, last view, rr_fill_colors, mesh, rr_draw_points and the next fused frame (its launches and its
    volume) are the same with and without an extraction in between."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 3)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    runs = []
    for extract in (False, True):
        fu = _context(sc, inv, frame=False)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        mesh = fu.extract_mesh()
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        if extract:
            fu.extract_points()
            fu.extract_points([1])
        r = dict(view=view, fill=fu.fill_colors(), tsdf=fu.download_tsdf(), bricks=fu.download_bricks(),
                 stages=_stages(fu), mesh=fu.download_mesh(len(mesh[0]), len(mesh[3])))
        r["points"] = fu.draw_points(mv, pr, 200, 120, shade_mode=0)
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        r["launches"] = fu.launch_count() - l0
        assert r["launches"] == per_frame
        r["next"] = fu.download_tsdf()
        runs.append(r)
        fu.close()
    a, b = runs
    for k in ("fill", "tsdf", "next"):
        assert bits_equal(a[k], b[k]).all(), k
    for k in ("view", "points", "mesh"):
        for x, y in zip(a[k], b[k]):
            assert bits_equal(x, y).all() if x.dtype == np.float32 else np.array_equal(x, y), k
    for x, y in zip(a["bricks"], b["bricks"]):
        assert np.array_equal(x, y)
    for k in a["stages"]:
        assert bits_equal(a["stages"][k], b["stages"][k]).all(), k
    assert a["launches"] == b["launches"]


def test_cloud_device_outputs(scene2):
    """device=True: CUDA tensors on the context's GPU equal to the host download, usable by sample_points as they are."""
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    host = fu.extract_points()
    dev = fu.extract_points(device=True)
    for n, h, d in zip(NAMES, host, dev):
        assert d.is_cuda and d.device == torch.device("cuda", 0), n
        assert tuple(d.shape) == h.shape, n
    _same_cloud("device", dev, host)
    val_d, nrm_d, rgba_d = fu.sample_points(dev[0])
    assert val_d.is_cuda
    val_h, nrm_h, rgba_h = fu.sample_points(host[0])
    assert bits_equal(val_d.cpu().numpy(), val_h).all() and bits_equal(rgba_d.cpu().numpy(), rgba_h).all()
    assert np.isfinite(val_h).sum() > 0.9 * len(val_h)         # the sensor points lie inside the fused volume
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_cloud_equals_single_context(scene2, n):
    from rrpy import capi
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    want = fu.extract_points()
    want1 = fu.extract_points([1])
    fu.close()
    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    _same_cloud(f"group of {n}", g.extract_points(), want, min_points=1000)
    _same_cloud(f"group of {n}, sensor 1", g.extract_points([1]), want1, min_points=100)
    dev = g.extract_points(device=True)
    _same_cloud(f"group of {n}, device", dev, want)
    g.close()


def _read_ply(path):
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode().split("\n")
    assert header[1] == "format binary_little_endian 1.0"
    assert not any(l.startswith("element face") for l in header)
    nv = int(next(l for l in header if l.startswith("element vertex")).split()[2])
    vt = np.dtype([("p", "<f4", 3), ("n", "<f4", 3), ("c", "u1", 3), ("q", "<f4")])
    assert end + nv * vt.itemsize == len(data)
    return np.frombuffer(data, vt, nv, end)


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_dump_points(tmp_path, small_scene, devices):
    """fusion_playback --dump-points writes the last frame set's cloud as a PLY equal to Fusion.extract_points() of the same
    frames: positions, normals and quality bit for bit, colours by the byte rule of writePly; through rr_group the same bytes."""
    from test_host_cpp import BIN, write_scene_files
    from rrpy import capi, synth, volume_io
    sc = small_scene
    ks, streams = write_scene_files(str(tmp_path), sc)
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    for i in range(sc.N):
        volume_io.write_volume(str(tmp_path / f"sensor{i}.cv_xyz_inv"), inv[i])
    runs = {}
    for dev in (None, devices) if devices else (None,):
        out = str(tmp_path / f"points_{dev}.ply")
        r = subprocess.run([os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
                            "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", "64", "64",
                            "--dump-points", out] + (["--devices", dev] if dev else []), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        assert "points " in r.stdout
        runs[dev] = open(out, "rb").read()
    if devices:
        assert runs[devices] == runs[None], "the multi-device run wrote other bytes"
    v = _read_ply(str(tmp_path / "points_None.ply"))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame()
    pos, nrm, rgb, q, pix = fu.extract_points()
    fu.close()
    assert len(v) == len(pos) > 1000
    assert bits_equal(v["p"], pos).all() and bits_equal(v["n"], nrm).all() and bits_equal(v["q"], q).all()
    c = np.nan_to_num(rgb, nan=0.0)
    want_c = (np.minimum(np.maximum(c, np.float32(0)), np.float32(1)) * np.float32(255) + np.float32(0.5)).astype(np.uint8)
    assert np.array_equal(v["c"], want_c)
