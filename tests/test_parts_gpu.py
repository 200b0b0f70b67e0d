"""Connected parts on the device (rr_label_parts / rr_download_parts / rr_download_mesh_parts / rr_group_label_parts)
against the oracle (oracle/oracle_parts.py: scipy.ndimage.label), bit for bit: labels, voxel counts, boxes, centroids and
the parts of the mesh's vertices and triangles. The oracle labels the oracle's own integrate where the scene is small, and
the volume the context holds otherwise (the 512^3 frame set, call orders that leave the brick tables stale)."""
import ctypes as C

import numpy as np
import oracle_parts
import pytest

from conftest import bits_equal

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10


def _oracle_tsdf(sc, inv, use_bricks=True, store_weight=0):
    import oracle_py as O
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
    t = O.integrate(inv, pre, grid, LIMIT, use_bricks, occ)
    return t.astype(np.float16).astype(np.float32) if store_weight == 2 else t


def _context(sc, inv, use_bricks=True, store_weight=0, frame=True):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame()
    return fu


def _got(fu):
    voxels, boxes, cen = fu.label_parts()
    return fu.part_labels(), voxels, boxes, cen


def _same_parts(what, got, want):
    names = ("labels", "voxels", "boxes", "centroids")
    for n, g, w in zip(names, got, want):
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n == "centroids":
            assert bits_equal(g, w).all(), f"{what} centroids: {(~bits_equal(g, w)).any(axis=1).sum()} of {len(w)} differ"
        else:
            assert np.array_equal(g, w), f"{what} {n}: {(np.asarray(g) != np.asarray(w)).sum()} entries differ"


def _check_against(fu, tsdf, sc, what, mesh=True):
    """Labels and statistics of the context against the oracle on tsdf; with mesh, also the mesh parts."""
    want = oracle_parts.label_parts(tsdf, sc.bbox_min, sc.bbox_max)
    got = _got(fu)
    _same_parts(what, got, want)
    if mesh:
        pos, _, _, tri = fu.extract_mesh()
        vp, tp = fu.mesh_parts()
        wvp, wtp = oracle_parts.mesh_parts(want[0], tsdf, tri)
        assert len(vp) == len(pos) and np.array_equal(vp, wvp), f"{what}: vertex parts differ"
        assert np.array_equal(tp, wtp), f"{what}: triangle parts differ"
        assert (vp[tri] == tp[:, None]).all(), f"{what}: a triangle spans two parts"
    return got


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


@pytest.fixture(scope="module")
def scene2():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("store_weight", [0, 1, 2])
def test_parts_match_oracle_bricks(scene2, store_weight):
    sc, inv = scene2
    fu = _context(sc, inv, store_weight=store_weight)
    got = _check_against(fu, _oracle_tsdf(sc, inv, store_weight=store_weight), sc, f"format {store_weight}")
    assert len(got[1]) >= 1 and got[1].sum() > 1000
    _same_parts("second call", _got(fu), got)
    fu.close()


def test_parts_dense_mode(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, use_bricks=False)
    _check_against(fu, _oracle_tsdf(sc, inv, use_bricks=False), sc, "dense")
    fu.close()


def _three_objects(p, frame=0):
    a = np.linalg.norm(p - np.array([0.5, 1.1, 0.0]), axis=-1) - 0.25
    b = np.linalg.norm(p - np.array([-0.5, 1.1, 0.0]), axis=-1) - 0.25
    c = np.linalg.norm(p - np.array([0.0, 1.6, 0.0]), axis=-1) - 0.05
    return np.minimum(np.minimum(a, b), c)


def test_three_objects_are_three_parts():
    # depth images of the headline size: at 128x106 the pre-process's filters erase the 5 cm sphere (a few pixels wide), and
    # the one-voxel band of v > 0 behind the big spheres' sparse samples falls apart into patches
    from rrpy import synth
    sc = synth.make_scene(N=4, W=512, H=424, CW=640, CH=540, cv_res=(32, 32, 64), sdf=_three_objects)
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv)
    labels, voxels, boxes, cen = _check_against(fu, _oracle_tsdf(sc, inv), sc, "three objects")
    assert len(voxels) >= 3
    res = fu.volume_res()
    bmin, bmax = np.asarray(sc.bbox_min, np.float64), np.asarray(sc.bbox_max, np.float64)
    owners = set()
    for centre in ((0.5, 1.1, 0.0), (-0.5, 1.1, 0.0), (0.0, 1.6, 0.0)):
        v = np.floor((np.asarray(centre) - bmin) / (bmax - bmin) * res).astype(int)
        inside = [k for k in range(len(voxels)) if all(boxes[k, 2 * a] <= v[a] < boxes[k, 2 * a + 1] for a in range(3))]
        assert inside, f"no part's box holds {centre}"
        owners.add(inside[0] if len(inside) == 1 else max(inside, key=lambda k: voxels[k]))
    assert len(owners) == 3
    fu.close()


def test_wall_spans_many_bricks():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), sdf=synth.wall_sdf)
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv)
    labels, voxels, boxes, _ = _check_against(fu, _oracle_tsdf(sc, inv), sc, "wall")
    big = int(np.argmax(voxels))
    assert all(boxes[big, 2 * a + 1] - boxes[big, 2 * a] > 2 * BRICK / VOXEL for a in (1,))
    fu.close()


def test_parts_eight_sensors():
    from rrpy import synth
    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv)
    _check_against(fu, _oracle_tsdf(sc, inv), sc, "8 sensors")
    fu.close()


def test_parts_headline_frame_set():
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
    got = _check_against(fu, fu.download_tsdf(), sc, "512^3")
    assert got[1].sum() > 100000
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "configure_limit"])
def test_parts_with_stale_brick_tables(scene2, order):
    """The brick tables no longer describe the volume: the whole volume is labelled, as the oracle does on the download."""
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    if order == "bricks_update_other":
        other = synth.rerender(sc, 7)
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
    else:
        fu.configure(limit=0.02, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    got = _check_against(fu, fu.download_tsdf(), sc, order)
    assert got[1].sum() > 1000
    fu.close()


def test_parts_of_an_empty_frame_set(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.upload_frames(sc.color, np.zeros_like(sc.depth))
    fu.frame()
    n = C.c_uint32(7)
    assert _status(fu, "rr_label_parts", C.byref(n)) == 0 and n.value == 0
    assert (fu.part_labels() == 0xFFFFFFFF).all()
    voxels, boxes, cen = fu.download_parts(0)
    assert voxels.shape == (0,) and boxes.shape == (0, 6) and cen.shape == (0, 3)
    fu.close()


def test_parts_refusals(scene2):
    from rrpy import capi, synth
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    n = C.c_uint32()
    assert _status(fu, "rr_label_parts", C.byref(n)) == -1                       # nothing integrated yet
    assert _status(fu, "rr_download_parts", None, None, None, None) == -1        # nothing labelled yet
    fu.frame()
    assert _status(fu, "rr_label_parts", None) == -1                             # null count pointer
    assert _status(fu, "rr_download_parts", None, None, None, None) == -1
    assert _status(fu, "rr_label_parts", C.byref(n)) == 0 and n.value > 0
    assert _status(fu, "rr_download_parts", None, None, None, None) == 0
    assert _status(fu, "rr_download_mesh_parts", None, None) == -1               # no mesh
    fu.extract_mesh()
    assert _status(fu, "rr_download_mesh_parts", None, None) == 0
    # a mesh and a labelling of different fused frame sets
    other = synth.rerender(sc, 9)
    fu.upload_frames(other.color, other.depth)
    fu.frame()
    assert _status(fu, "rr_download_mesh_parts", None, None) == 0                # both still of the frame set before
    assert _status(fu, "rr_label_parts", C.byref(n)) == 0
    assert _status(fu, "rr_download_mesh_parts", None, None) == -1               # the mesh is of the frame set before
    fu.extract_mesh()
    assert _status(fu, "rr_download_mesh_parts", None, None) == 0
    fu.frame()
    fu.extract_mesh()
    assert _status(fu, "rr_download_mesh_parts", None, None) == -1               # the labelling is of the frame set before
    # a new voxel format is a new volume: nothing integrated, nothing labelled
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True, store_weight=capi.VOXELS_HALF2)
    assert _status(fu, "rr_label_parts", C.byref(n)) == -1
    assert _status(fu, "rr_download_parts", None, None, None, None) == -1
    fu.frame()
    fu.set_slab(0, int(fu.volume_res()[2]) // 2)
    assert _status(fu, "rr_label_parts", C.byref(n)) == -1
    assert "rr_group_label_parts" in fu.L.rr_last_error(fu.h).decode()
    fu.close()


def _noise_field(sc, seed):
    """Twenty spheres of 15 cm: a frame set with many parts (smaller ones do not survive the pre-process at 128x106)."""
    rng = np.random.default_rng(seed)
    centres = np.stack([rng.uniform(-0.7, 0.7, 20), rng.uniform(0.3, 1.9, 20), rng.uniform(-0.7, 0.7, 20)], 1)

    def sdf(p, frame=0):
        d = np.full(p.shape[:-1], np.inf)
        for c in centres:
            d = np.minimum(d, np.linalg.norm(p - c, axis=-1) - 0.15)
        return d
    return sdf


def test_parts_buffers_grow(scene2):
    """A frame set with few parts, then one with many (same context): the part buffers grow and both labellings are right."""
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    few = _check_against(fu, fu.download_tsdf(), sc, "few", mesh=False)
    many_sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), sdf=_noise_field(sc, 3))
    fu.upload_frames(many_sc.color, many_sc.depth)
    fu.frame()
    many = _check_against(fu, fu.download_tsdf(), sc, "many")
    assert len(many[1]) > len(few[1]) + 5
    fu.close()


def test_parts_have_no_side_effects(scene2):
    """Against a twin context that never labels: volume, brick tables, view, fill_colors, mesh and cloud; after the next
    fused frame the volume, the launches per frame and rr_integrator_last."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 3)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    runs = []
    for label in (False, True):
        fu = _context(sc, inv, frame=False)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        mesh = fu.extract_mesh()
        cloud = fu.extract_points()
        if label:
            fu.label_parts()
            fu.mesh_parts()
        out = dict(view=view, tsdf=fu.download_tsdf(), bricks=fu.download_bricks(), fill=fu.fill_colors(),
                   mesh=fu.download_mesh(len(mesh[0]), len(mesh[3])), cloud=fu.download_points(len(cloud[0])))
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        out["per_frame"], out["next_frame"] = (per_frame, fu.launch_count() - l0), fu.download_tsdf()
        out["last"] = fu.integrator_last()
        runs.append(out)
        fu.close()
    a, b = runs
    for key in ("view", "mesh", "cloud", "bricks"):
        for x, y in zip(a[key], b[key]):
            assert (bits_equal(x, y).all() if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y)), key
    for key in ("tsdf", "next_frame", "fill"):
        assert bits_equal(a[key], b[key]).all(), key
    assert a["per_frame"] == b["per_frame"] and b["per_frame"][0] == b["per_frame"][1]
    assert a["last"] == b["last"]


def test_cuda_tensor_outputs_equal_host_outputs(scene2):
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    fu.label_parts()
    fu.extract_mesh()
    host_labels, host_vp = fu.part_labels(), fu.mesh_parts()
    dev_labels, dev_vp = fu.part_labels(device=True), fu.mesh_parts(device=True)
    assert isinstance(dev_labels, torch.Tensor) and dev_labels.is_cuda
    assert np.array_equal(dev_labels.cpu().numpy(), host_labels)
    for d, h in zip(dev_vp, host_vp):
        assert d.is_cuda and np.array_equal(d.cpu().numpy(), h)
    # pinned host memory
    n = int(fu.label_parts_count())
    pinned = torch.empty(tuple(int(v) for v in fu.volume_res()[::-1]), dtype=torch.int32).pin_memory()
    assert _status(fu, "rr_download_parts", None, None, None, C.c_void_p(pinned.data_ptr())) == 0
    assert np.array_equal(pinned.numpy().view(np.uint32), host_labels) and n > 0
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_parts_equal_single_context(scene2, n):
    from rrpy import capi
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    want = _got(fu)
    want_mesh = fu.extract_mesh()
    want_mp = fu.mesh_parts()
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
    voxels, boxes, cen = g.label_parts()
    _same_parts(f"group of {n}", (g.part_labels(), voxels, boxes, cen), want)
    if n > 1:
        bounds = g.slabs()
        assert any(boxes[k, 4] < b < boxes[k, 5] for k in range(len(voxels)) for b in bounds[1:-1]), "no part crosses a slab boundary"
    g.extract_mesh()
    for x, y in zip(g.mesh_parts(), want_mp):
        assert np.array_equal(x, y)
    assert len(want_mp[0]) == len(want_mesh[0])
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_parts(tmp_path, small_scene, devices):
    """fusion_playback --parts prints Fusion.label_parts() of the same frames; --min-part-voxels N with --dump-mesh writes the
    triangles of the parts of at least N voxels and the vertices they use, re-indexed in their original order."""
    import os
    import subprocess
    from test_host_cpp import BIN, write_scene_files
    from test_mesh_gpu import _read_ply
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
    voxels, boxes, cen = fu.label_parts()
    pos, nrm, rgba, tri = fu.extract_mesh()
    vp, tp = fu.mesh_parts()
    fu.close()
    assert len(voxels) > 0
    threshold = int(np.sort(voxels)[-1])                 # keeps the largest part only
    out = str(tmp_path / "mesh.ply")
    args = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
            "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", "64", "64", "--parts",
            "--dump-mesh", out, "--min-part-voxels", str(threshold)] + (["--devices", devices] if devices else [])
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("part ")]
    want = [f"part {k} voxels {voxels[k]} box {' '.join(str(int(b)) for b in boxes[k])} centroid "
            + " ".join("%.9g" % float(c) for c in cen[k]) for k in range(len(voxels))]
    assert lines == want
    keep_t = voxels[tp] >= threshold
    used = np.zeros(len(pos), bool)
    used[tri[keep_t].ravel()] = True
    index = np.cumsum(used) - 1
    v, f = _read_ply(out)
    assert len(v) == used.sum() and len(f) == keep_t.sum() > 0
    assert bits_equal(v["p"], pos[used]).all() and bits_equal(v["n"], nrm[used]).all()
    assert np.array_equal(f["i"], index[tri[keep_t]].astype(np.uint32))
