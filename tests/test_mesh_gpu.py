"""Surface extraction on the device (rr_extract_mesh / rr_download_mesh / rr_group_extract_mesh) against the oracle's scalar
marching cubes (oracle/ro_mesh.cpp), bit for bit: counts, positions, normals, colours and triangles. The oracle extracts from
its own pre-process and integrate where the scene is small, and from the volume and stage images the context holds otherwise
(the 512^3 frame set, call orders that leave the brick tables stale)."""
import ctypes as C

import numpy as np
import oracle_mesh
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10


def _same_mesh(what, got, want):
    names = ("positions", "normals", "rgba", "triangles")
    for n, g, w in zip(names, got, want):
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n == "triangles":
            assert np.array_equal(g, w), f"{what} triangles: {(g != w).any(axis=1).sum()} of {len(w)} differ"
        else:
            assert bits_equal(g, w).all(), mismatch_report(f"{what} {n}", g, w)


def _oracle_inputs(sc, use_bricks=True):
    import oracle_py as O
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
    return grid, pre, occ


def _context(sc, inv, use_bricks=True, store_weight=0, frame=True):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame()
    return fu


def _oracle_of_context(fu, sc, inv, limit=LIMIT):
    """The oracle's extraction from what the context holds now: its volume, stage images and limit."""
    import oracle_py as O
    tsdf = fu.download_tsdf()
    pre = dict(depth_b=fu.download_stage("depth_b"), quality=fu.download_stage("quality"))
    return oracle_mesh.extract_mesh(tsdf, fu.volume_res(), limit, inv, sc, pre, sc.bbox_min, sc.bbox_max)


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


@pytest.fixture(scope="module")
def scene2():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("store_weight", [0, 1, 2])
def test_mesh_matches_oracle_bricks(scene2, store_weight):
    import oracle_py as O
    sc, inv = scene2
    grid, pre, occ = _oracle_inputs(sc)
    want_tsdf = O.integrate(inv, pre, grid, LIMIT, True, occ)
    if store_weight == 2:
        want_tsdf = want_tsdf.astype(np.float16).astype(np.float32)
    want = oracle_mesh.extract_mesh(want_tsdf, grid["res"], LIMIT, inv, sc, pre, sc.bbox_min, sc.bbox_max)
    fu = _context(sc, inv, store_weight=store_weight)
    got = fu.extract_mesh()
    _same_mesh(f"format {store_weight}", got, want)
    assert len(got[0]) > 1000 and len(got[3]) > 1000
    assert (got[2][:, 3] == 1.0).any()
    _same_mesh("second call", fu.extract_mesh(), got)
    fu.close()


def test_mesh_dense_mode(scene2):
    import oracle_py as O
    sc, inv = scene2
    grid, pre, occ = _oracle_inputs(sc)
    want_tsdf = O.integrate(inv, pre, grid, LIMIT, False, occ)
    want = oracle_mesh.extract_mesh(want_tsdf, grid["res"], LIMIT, inv, sc, pre, sc.bbox_min, sc.bbox_max)
    fu = _context(sc, inv, use_bricks=False)
    _same_mesh("dense", fu.extract_mesh(), want)
    fu.close()


def test_mesh_eight_sensors():
    import oracle_py as O
    from rrpy import synth
    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    grid, pre, occ = _oracle_inputs(sc)
    want = oracle_mesh.extract_mesh(O.integrate(inv, pre, grid, LIMIT, True, occ), grid["res"], LIMIT, inv, sc, pre, sc.bbox_min, sc.bbox_max)
    fu = _context(sc, inv)
    got = fu.extract_mesh()
    _same_mesh("8 sensors", got, want)
    assert len(got[3]) > 1000
    fu.close()


def test_mesh_headline_frame_set():
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
    got = fu.extract_mesh()
    want = _oracle_of_context(fu, sc, inv, limit=bench.LIMIT)
    _same_mesh("512^3", got, want)
    assert len(got[3]) > 100000
    fu.close()


def test_mesh_of_an_empty_frame_set(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.upload_frames(sc.color, np.zeros_like(sc.depth))
    fu.frame()
    nv, nt = C.c_uint32(7), C.c_uint32(7)
    assert _status(fu, "rr_extract_mesh", C.byref(nv), C.byref(nt)) == 0
    assert nv.value == 0 and nt.value == 0
    pos, nrm, rgba, tri = fu.download_mesh(0, 0)
    assert pos.shape == (0, 3) and tri.shape == (0, 3)
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "bricks_clear", "preprocess_other", "configure_limit"])
def test_mesh_after_call_orders(scene2, order):
    """A call between the integrate and the extraction: the mesh is still marching cubes over the volume the context holds,
    with attributes from the limit and stage images in effect at the call."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 7)
    fu = _context(sc, inv)
    limit = LIMIT
    if order == "bricks_update_other":
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
    elif order == "bricks_clear":
        fu.bricks_clear()
    elif order == "preprocess_other":
        fu.upload_frames(other.color, other.depth)
        fu.preprocess()
    else:
        limit = 0.02
        fu.configure(limit=limit, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    got = fu.extract_mesh()
    want = _oracle_of_context(fu, other if "other" in order else sc, inv, limit=limit)
    _same_mesh(order, got, want)
    assert len(got[3]) > 1000
    fu.close()


def test_mesh_refusals(scene2):
    from rrpy import capi
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    nv, nt = C.c_uint32(), C.c_uint32()
    assert _status(fu, "rr_extract_mesh", C.byref(nv), C.byref(nt)) == -1          # nothing integrated yet
    assert _status(fu, "rr_download_mesh", None, None, None, None) == -1           # nothing extracted yet
    fu.frame()
    assert _status(fu, "rr_download_mesh", None, None, None, None) == -1
    assert _status(fu, "rr_extract_mesh", C.byref(nv), C.byref(nt)) == 0 and nt.value > 0
    assert _status(fu, "rr_download_mesh", None, None, None, None) == 0
    # a new voxel format is a new volume: nothing integrated, nothing extracted
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True, store_weight=capi.VOXELS_HALF2)
    assert _status(fu, "rr_extract_mesh", C.byref(nv), C.byref(nt)) == -1
    assert _status(fu, "rr_download_mesh", None, None, None, None) == -1
    fu.frame()
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_extract_mesh", C.byref(nv), C.byref(nt)) == -1
    assert "rr_group_extract_mesh" in fu.L.rr_last_error(fu.h).decode()
    fu.close()


def test_mesh_buffers_grow(scene2):
    """A small mesh first (a coarse volume), then a larger one (a finer volume, same context): the device buffers grow and
    both meshes are right."""
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.configure(limit=LIMIT, voxel_size=2 * VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.frame()
    small = fu.extract_mesh()
    _same_mesh("small", small, _oracle_of_context(fu, sc, inv))
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.frame()
    large = fu.extract_mesh()
    _same_mesh("large", large, _oracle_of_context(fu, sc, inv))
    assert len(large[0]) > 2 * len(small[0]) > 0 and len(large[3]) > 2 * len(small[3])
    fu.close()


def test_mesh_has_no_side_effects(scene2):
    """A raymarch, the next fused frame's volume and the launches per fused frame are the same with and without an
    extraction in between (captured frame graphs stay valid)."""
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
        if extract:
            fu.extract_mesh()
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        assert fu.launch_count() - l0 == per_frame
        runs.append((view, fu.download_tsdf(), per_frame))
        fu.close()
    (v0, t0, p0), (v1, t1, p1) = runs
    assert bits_equal(v0[0], v1[0]).all() and bits_equal(v0[1], v1[1]).all()
    assert bits_equal(t0, t1).all()
    assert p0 == p1


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_mesh_equals_single_context(scene2, n):
    from rrpy import capi, synth
    sc, inv = scene2
    other = synth.rerender(sc, 5)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    want = fu.extract_mesh()
    want_view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
    want_tsdf = fu.download_tsdf()
    fu.upload_frames(other.color, other.depth)
    fu.fuse_frame()
    want_next = fu.download_tsdf()
    fu.close()

    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    _same_mesh(f"group of {n}", g.extract_mesh(), want)
    view = g.raymarch(mv, pr, 200, 120, shade_mode=1)
    assert bits_equal(view[0], want_view[0]).all() and bits_equal(view[1], want_view[1]).all()
    assert bits_equal(g.download_tsdf(), want_tsdf).all()
    g.upload_frames(other.color, other.depth)
    g.fuse_frame()
    assert bits_equal(g.download_tsdf(), want_next).all()
    g.close()


def _read_ply(path):
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode().split("\n")
    assert header[1] == "format binary_little_endian 1.0"
    nv = int(next(l for l in header if l.startswith("element vertex")).split()[2])
    nt = int(next(l for l in header if l.startswith("element face")).split()[2])
    vt = np.dtype([("p", "<f4", 3), ("n", "<f4", 3), ("c", "u1", 3)])
    ft = np.dtype([("k", "u1"), ("i", "<u4", 3)])
    v = np.frombuffer(data, vt, nv, end)
    f = np.frombuffer(data, ft, nt, end + nv * vt.itemsize)
    assert end + nv * vt.itemsize + nt * ft.itemsize == len(data)
    assert (f["k"] == 3).all()
    return v, f


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_dump_mesh(tmp_path, small_scene, devices):
    """fusion_playback --dump-mesh writes the last frame set's surface as a PLY equal to Fusion.extract_mesh() of the same
    frames: positions and normals bit for bit, colours by the byte rule of writePly; through rr_group the same bytes."""
    import os
    import subprocess
    from test_host_cpp import BIN, write_scene_files
    from rrpy import capi, synth, volume_io
    sc = small_scene
    ks, streams = write_scene_files(str(tmp_path), sc)
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    for i in range(sc.N):
        volume_io.write_volume(str(tmp_path / f"sensor{i}.cv_xyz_inv"), inv[i])
    runs = {}
    for dev in (None, devices) if devices else (None,):
        out = str(tmp_path / f"mesh_{dev}.ply")
        r = subprocess.run([os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
                            "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", "64", "64",
                            "--dump-mesh", out] + (["--devices", dev] if dev else []), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        assert "mesh vertices" in r.stdout
        runs[dev] = open(out, "rb").read()
    if devices:
        assert runs[devices] == runs[None], "the multi-device run wrote other bytes"
    v, f = _read_ply(str(tmp_path / "mesh_None.ply"))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame()
    pos, nrm, rgba, tri = fu.extract_mesh()
    fu.close()
    assert len(v) == len(pos) > 1000 and len(f) == len(tri)
    assert bits_equal(v["p"], pos).all() and bits_equal(v["n"], nrm).all()
    c = np.nan_to_num(rgba[:, :3], nan=0.0)
    want_c = (np.minimum(np.maximum(c, np.float32(0)), np.float32(1)) * np.float32(255) + np.float32(0.5)).astype(np.uint8)
    assert np.array_equal(v["c"], want_c)
    assert np.array_equal(f["i"], tri)
