"""Mesh simplification on the device (rr_simplify_mesh / rr_download_simplified_mesh / rr_group_simplify_mesh) against the
oracle (oracle/oracle_simplify.py), bit for bit: positions, normals, colours, triangles and sources. The oracle simplifies
the oracle's own mesh of the oracle's own integrate where the scene is small, and the mesh of the volume and stage images
the context holds otherwise (the 512^3 frame set, call orders that leave the brick tables stale)."""
import ctypes as C

import numpy as np
import oracle_mesh
import oracle_simplify
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.02, (40, 44, 40), 0.01, 0.1, 10
SIZES = (1, 2, 3, 5)
NAMES = ("positions", "normals", "rgba", "triangles", "sources")


def _same(what, got, want):
    for n, g, w in zip(NAMES, got, want):
        g = g.cpu().numpy() if hasattr(g, "cpu") else np.asarray(g)
        assert g.shape == w.shape, f"{what} {n}: shape {g.shape} != {w.shape}"
        if n in ("triangles", "sources"):
            assert np.array_equal(g, w), f"{what} {n}: {(g != w).reshape(len(w), -1).any(axis=1).sum()} of {len(w)} differ"
        else:
            assert bits_equal(g, w).all(), mismatch_report(f"{what} {n}", g, w)


def _context(sc, inv, use_bricks=True, store_weight=0, frame=True):
    from rrpy import capi
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=use_bricks, store_weight=store_weight)
    fu.upload_frames(sc.color, sc.depth)
    if frame:
        fu.frame()
    return fu


class _Oracle:
    """The oracle's mesh of a volume and its simplifications: from the oracle's own pre-process and integrate, or (of_context)
    from the volume, stage images and limit a context holds now."""

    def __init__(self, tsdf, sc, inv, pre, limit=LIMIT):
        self.tsdf, self.sc, self.inv, self.pre, self.limit = tsdf, sc, inv, pre, limit
        Z, Y, X = tsdf.shape
        self.mesh = oracle_mesh.extract_mesh(tsdf, (X, Y, Z), limit, inv, sc, pre, sc.bbox_min, sc.bbox_max)

    @classmethod
    def integrated(cls, sc, inv, use_bricks=True, store_weight=0):
        import oracle_py as O
        grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
        cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
        pre = O.preprocess(sc, grid, cams)
        occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
        t = O.integrate(inv, pre, grid, LIMIT, use_bricks, occ)
        return cls(t.astype(np.float16).astype(np.float32) if store_weight == 2 else t, sc, inv, pre)

    @classmethod
    def of_context(cls, fu, sc, inv, limit=LIMIT):
        pre = dict(depth_b=fu.download_stage("depth_b"), quality=fu.download_stage("quality"))
        return cls(fu.download_tsdf(), sc, inv, pre, limit)

    def simplify(self, c):
        pos, _, _, tri = self.mesh
        return oracle_simplify.simplify_mesh(self.tsdf, pos, tri, c, self.limit, self.sc.bbox_min, self.sc.bbox_max,
                                             self.inv, self.sc, self.pre)


def _check(fu, oracle, what, sizes=SIZES):
    """The context's mesh equals the oracle's, and each simplification equals the oracle's; returns them by size."""
    got_mesh = fu.extract_mesh()
    for n, g, w in zip(NAMES, got_mesh, oracle.mesh):
        assert (np.array_equal(g, w) if n == "triangles" else bits_equal(g, w).all()), f"{what}: mesh {n} differs"
    out = {}
    for c in sizes:
        got = fu.simplify_mesh(c)
        _same(f"{what} c={c}", got, oracle.simplify(c))
        out[c] = got
    return out


def _status(fu, fn, *args):
    return getattr(fu.L, fn)(fu.h, *args)


@pytest.fixture(scope="module")
def scene2():
    from rrpy import synth
    sc = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
    return sc, synth.analytic_inverse(sc, INV_RES)


@pytest.mark.parametrize("mode", ["f32", "f32_weight", "half2", "dense"])
def test_simplify_matches_oracle(scene2, mode):
    sc, inv = scene2
    store_weight = dict(f32=0, f32_weight=1, half2=2, dense=0)[mode]
    use_bricks = mode != "dense"
    fu = _context(sc, inv, use_bricks=use_bricks, store_weight=store_weight)
    out = _check(fu, _Oracle.integrated(sc, inv, use_bricks, store_weight), mode)
    nv = [len(out[c][0]) for c in SIZES]
    assert nv[0] > 1000 and all(a > b for a, b in zip(nv, nv[1:])), nv
    assert all(len(out[c][3]) > 0 for c in SIZES)
    assert (out[2][2][:, 3] == 1.0).any()
    fu.close()


def test_simplify_eight_sensors():
    from rrpy import synth
    sc = synth.make_scene(8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    fu = _context(sc, inv)
    _check(fu, _Oracle.integrated(sc, inv), "8 sensors", sizes=(2, 3))
    fu.close()


def test_simplify_headline_frame_set():
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
    out = _check(fu, _Oracle.of_context(fu, sc, inv, limit=bench.LIMIT), "512^3", sizes=(2, 4))
    assert len(out[2][3]) > 10000
    fu.close()


@pytest.mark.parametrize("order", ["bricks_update_other", "configure_limit"])
def test_simplify_with_stale_brick_tables(scene2, order):
    """The brick tables no longer describe the volume: the mesh is of the whole volume, and normals and colours come from
    the limit and stage images in effect at the call."""
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv)
    limit = LIMIT
    other = synth.rerender(sc, 7)
    if order == "bricks_update_other":
        fu.upload_frames(other.color, other.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
    else:
        limit = 0.02
        fu.configure(limit=limit, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    _check(fu, _Oracle.of_context(fu, other if "other" in order else sc, inv, limit=limit), order, sizes=(2,))
    fu.close()


def test_simplify_an_empty_frame_set(scene2):
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.upload_frames(sc.color, np.zeros_like(sc.depth))
    fu.frame()
    assert fu.extract_mesh_counts() == (0, 0)
    nv, nt = C.c_uint32(7), C.c_uint32(7)
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == 0 and nv.value == 0 and nt.value == 0
    got = fu.download_simplified_mesh(0, 0)
    assert [g.shape for g in got] == [(0, 3), (0, 3), (0, 4), (0, 3), (0,)]
    fu.close()


def test_normals_and_colours_are_point_samples(scene2):
    sc, inv = scene2
    fu = _context(sc, inv)
    fu.extract_mesh()
    for c in (1, 3):
        pos, nrm, rgba, _, _ = fu.simplify_mesh(c)
        _, snrm, srgba = fu.sample_points(pos, "world")
        assert bits_equal(nrm, snrm).all() and bits_equal(rgba, srgba).all()
    # a context restricted to a slab still samples the whole volume
    fu.set_slab(0, int(fu.volume_res()[2]) // 3)
    got = fu.simplify_mesh(3)
    fu.set_slab(0, int(fu.volume_res()[2]))
    _, snrm, srgba = fu.sample_points(got[0], "world")
    assert bits_equal(got[1], snrm).all() and bits_equal(got[2], srgba).all()
    fu.close()


def test_sources_carry_the_mesh_parts(scene2):
    sc, inv = scene2
    fu = _context(sc, inv)
    _, _, _, tri = fu.extract_mesh()
    voxels, _, _ = fu.label_parts()
    vp, tp = fu.mesh_parts()
    _, _, _, stri, src = fu.simplify_mesh(2)
    assert len(src) > 0 and (tp[src] < len(voxels)).all()
    assert np.array_equal(tp[src], vp[tri[src, 0]])
    # mesh_parts is still the full mesh's after the simplification
    for x, y in zip(fu.mesh_parts(), (vp, tp)):
        assert np.array_equal(x, y)
    fu.close()


def test_simplify_refusals(scene2):
    from rrpy import capi, synth
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    nv, nt = C.c_uint32(), C.c_uint32()
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == -1                     # no mesh
    assert _status(fu, "rr_download_simplified_mesh", None, None, None, None, None) == -1         # nothing simplified
    fu.frame()
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == -1                     # still no mesh
    fu.extract_mesh()
    assert _status(fu, "rr_simplify_mesh", 0, C.byref(nv), C.byref(nt)) == -1                     # c = 0
    assert _status(fu, "rr_simplify_mesh", 2, None, C.byref(nt)) == -1                             # null count pointers
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), None) == -1
    assert _status(fu, "rr_download_simplified_mesh", None, None, None, None, None) == -1
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == 0 and nt.value > 0
    assert _status(fu, "rr_download_simplified_mesh", None, None, None, None, None) == 0
    # a later fused frame: the mesh is of an older volume state; the last simplification can still be read
    other = synth.rerender(sc, 9)
    fu.upload_frames(other.color, other.depth)
    fu.fuse_frame()
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == -1
    assert "rr_extract_mesh" in fu.L.rr_last_error(fu.h).decode()
    assert _status(fu, "rr_download_simplified_mesh", None, None, None, None, None) == 0
    fu.extract_mesh()
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == 0
    fu.frame()
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == -1
    # a new voxel format is a new volume: nothing to simplify, nothing to download
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True, store_weight=capi.VOXELS_HALF2)
    assert _status(fu, "rr_simplify_mesh", 2, C.byref(nv), C.byref(nt)) == -1
    assert _status(fu, "rr_download_simplified_mesh", None, None, None, None, None) == -1
    fu.close()


def test_simplify_has_no_side_effects(scene2):
    """Against a twin context that never simplifies: the full mesh, mesh parts, volume, view, fill_colors, cloud, parts and
    a query after the call; after the next fused frame the volume, the launches per frame and rr_integrator_last."""
    from rrpy import synth
    sc, inv = scene2
    other = synth.rerender(sc, 3)
    mv, pr = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0)), synth.perspective(50.0, 200 / 120, 0.1, 10.0)
    pts = np.random.default_rng(5).uniform(sc.bbox_min, sc.bbox_max, (500, 3)).astype(np.float32)
    runs = []
    for simplify in (False, True):
        fu = _context(sc, inv, frame=False)
        fu.fuse_frame()
        fu.fuse_frame()                      # the captured graph
        l0 = fu.launch_count()
        fu.fuse_frame()
        per_frame = fu.launch_count() - l0
        view = fu.raymarch(mv, pr, 200, 120, shade_mode=1)
        mesh = fu.extract_mesh()
        cloud = fu.extract_points()
        parts = fu.label_parts()
        q0 = fu.sample_points(pts[:100])
        if simplify:
            for c in (2, 5):
                fu.simplify_mesh(c)
        out = dict(view=view, tsdf=fu.download_tsdf(), bricks=fu.download_bricks(), fill=fu.fill_colors(),
                   mesh=fu.download_mesh(len(mesh[0]), len(mesh[3])), mesh_parts=fu.mesh_parts(),
                   cloud=fu.download_points(len(cloud[0])), parts=fu.download_parts(len(parts[0])),
                   query=fu.sample_points(pts), q0=q0)
        fu.upload_frames(other.color, other.depth)
        l0 = fu.launch_count()
        fu.fuse_frame()
        out["per_frame"], out["next_frame"] = (per_frame, fu.launch_count() - l0), fu.download_tsdf()
        out["last"] = fu.integrator_last()
        runs.append(out)
        fu.close()
    a, b = runs
    for key in ("view", "mesh", "mesh_parts", "cloud", "parts", "query", "q0", "bricks"):
        for x, y in zip(a[key], b[key]):
            assert (bits_equal(x, y).all() if np.asarray(x).dtype.kind == "f" else np.array_equal(x, y)), key
    for key in ("tsdf", "next_frame", "fill"):
        assert bits_equal(a[key], b[key]).all(), key
    assert a["per_frame"] == b["per_frame"] and b["per_frame"][0] == b["per_frame"][1]
    assert a["last"] == b["last"]


def _noise_field(seed):
    """Twenty spheres of 15 cm: a larger mesh than the default scene's."""
    rng = np.random.default_rng(seed)
    centres = np.stack([rng.uniform(-0.7, 0.7, 20), rng.uniform(0.3, 1.9, 20), rng.uniform(-0.7, 0.7, 20)], 1)

    def sdf(p, frame=0):
        d = np.full(p.shape[:-1], np.inf)
        for c in centres:
            d = np.minimum(d, np.linalg.norm(p - c, axis=-1) - 0.15)
        return d
    return sdf


def test_simplify_buffers_grow_and_repeat(scene2):
    """A small mesh (a coarse volume), then a larger one (a finer volume, then a busier scene), same context: the buffers
    grow, every result equals the oracle's, and a repeated call gives the same bits."""
    from rrpy import synth
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.configure(limit=LIMIT, voxel_size=2 * VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.frame()
    small = _check(fu, _Oracle.of_context(fu, sc, inv), "coarse", sizes=(2,))
    fu.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    fu.frame()
    big = _check(fu, _Oracle.of_context(fu, sc, inv), "fine", sizes=(1, 2))
    assert len(big[1][3]) > 2 * len(small[2][3])
    busy = synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), sdf=_noise_field(3))
    fu.upload_frames(busy.color, busy.depth)
    fu.frame()
    again = _check(fu, _Oracle.of_context(fu, busy, inv), "busy", sizes=(1, 2))
    for c in (1, 2):
        _same(f"repeat c={c}", fu.simplify_mesh(c), tuple(x for x in again[c]))
    fu.close()


def test_cuda_tensor_and_pinned_outputs(scene2):
    import torch
    sc, inv = scene2
    fu = _context(sc, inv)
    fu.extract_mesh()
    host = fu.simplify_mesh(2)
    dev = fu.simplify_mesh(2, device=True)
    for d, h in zip(dev, host):
        assert isinstance(d, torch.Tensor) and d.is_cuda
    _same("device", dev, host)
    nv, nt = len(host[0]), len(host[3])
    pinned = [torch.empty(s, dtype=t).pin_memory() for s, t in (((nv, 3), torch.float32), ((nv, 3), torch.float32),
                                                                 ((nv, 4), torch.float32), ((nt, 3), torch.int32), ((nt,), torch.int32))]
    assert _status(fu, "rr_download_simplified_mesh", *[C.c_void_p(p.data_ptr()) for p in pinned]) == 0
    _same("pinned", [p.numpy().view(np.uint32) if p.dtype == torch.int32 else p.numpy() for p in pinned], host)
    fu.close()


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % max(1, have) for i in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3])
def test_group_simplify_equals_single_context(scene2, n):
    from rrpy import capi
    sc, inv = scene2
    fu = _context(sc, inv, frame=False)
    fu.fuse_frame()
    fu.extract_mesh()
    want = {c: fu.simplify_mesh(c) for c in (2, 3)}
    fu.close()

    g = capi.Group(_devices(n), sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=LIMIT, voxel_size=VOXEL, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
    if n > 1:
        Z = int(g.member(0).volume_res()[2])       # slab boundaries through the middle of the scene, where the surface is
        g.set_slabs([0] + [int(b) for b in np.linspace(Z // 2 - 5, Z // 2 + 5, n - 1)] + [Z])
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    nv, nt = C.c_uint32(), C.c_uint32()
    assert g.L.rr_group_simplify_mesh(g.h, 2, C.byref(nv), C.byref(nt)) != 0    # no mesh yet
    g.extract_mesh()
    for c in (2, 3):
        _same(f"group of {n} c={c}", g.simplify_mesh(c), want[c])
    if n > 1:                                      # the simplified surface lies on both sides of every slab boundary
        zs = (want[2][0][:, 2] - sc.bbox_min[2]) / (sc.bbox_max[2] - sc.bbox_min[2]) * Z
        assert all((zs < b).any() and (zs > b).any() for b in g.slabs()[1:-1])
    g.close()


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_fusion_playback_simplify(tmp_path, small_scene, devices):
    """fusion_playback --dump-mesh --simplify 2 writes Fusion.simplify_mesh(2) of the same frames; with --min-part-voxels N
    it keeps the simplified triangles whose source triangle's part has at least N voxels, and the vertices they use,
    re-indexed in their order."""
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
    fu.extract_mesh()
    voxels, _, _ = fu.label_parts()
    _, tp = fu.mesh_parts()
    pos, nrm, rgba, tri, src = fu.simplify_mesh(2)
    fu.close()
    assert len(tri) > 100
    threshold = int(np.sort(voxels)[-1])                 # keeps the largest part only
    for min_part in (None, threshold):
        out = str(tmp_path / f"simple_{min_part}.ply")
        args = [os.path.join(BIN, "fusion_playback"), ks, "--depth", str(sc.W), str(sc.H), "--color", str(sc.CW), str(sc.CH),
                "--streams", ";".join(streams), "--frames", "2", "--voxel", "0.02", "--view", "64", "64",
                "--dump-mesh", out, "--simplify", "2"]
        args += (["--min-part-voxels", str(min_part)] if min_part is not None else []) + (["--devices", devices] if devices else [])
        r = subprocess.run(args, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        keep_t = np.ones(len(tri), bool) if min_part is None else voxels[tp[src]] >= min_part
        used = np.zeros(len(pos), bool)
        used[tri[keep_t].ravel()] = True
        index = np.cumsum(used) - 1
        v, f = _read_ply(out)
        assert len(v) == used.sum() and len(f) == keep_t.sum() > 0
        assert bits_equal(v["p"], pos[used]).all() and bits_equal(v["n"], nrm[used]).all()
        c = np.nan_to_num(rgba[used, :3], nan=0.0)
        want_c = (np.minimum(np.maximum(c, np.float32(0)), np.float32(1)) * np.float32(255) + np.float32(0.5)).astype(np.uint8)
        assert np.array_equal(v["c"], want_c)
        assert np.array_equal(f["i"], index[tri[keep_t]].astype(np.uint32))
        if min_part is None:
            assert used.all()
