"""GPU parity: CUDA path through the C ABI vs the scalar oracle on the same seeded synthetic frames.

Bars (BASELINE.json north_star): brick counters / occupied lists bit-exact; TSDF, weights, normals within
1e-5 * limit — in practice the pinned arithmetic makes every stage bit-identical, and that is what is asserted.
"""
import numpy as np
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu


def _run_both(scene, voxel_size, inv_res, use_bricks, flags=(True, True, True), store_weight=False, limit=0.01):
    import oracle_py as O
    from rrpy import capi, synth
    inv = synth.analytic_inverse(scene, inv_res)
    fu = capi.Fusion(scene.N, scene.W, scene.H, scene.CW, scene.CH)
    capi.load_scene(fu, scene, inv)
    fu.configure(limit=limit, voxel_size=voxel_size, brick_size=0.1, min_voxels=10, use_bricks=use_bricks, store_weight=store_weight)
    fu.upload_frames(scene.color, scene.depth)
    n_occ, ratio = fu.frame(*flags, sync_bricks=True)
    got = {k: fu.download_stage(k) for k in capi.STAGES}
    got["counters"], got["occupied"] = fu.download_bricks()
    got["tsdf"] = fu.download_tsdf()
    if store_weight:
        got["weight"] = fu.download_weight()
    got["n_occ"], got["ratio"] = n_occ, ratio
    got["cams"] = fu.camera_positions()
    got["res"] = fu.volume_res()
    got["brick_info"] = fu.brick_info()
    got["ranges"] = fu.brick_ranges()
    got["last"] = fu.integrator_last()
    fu.close()

    grid = O.brick_grid(scene.bbox_min, scene.bbox_max, voxel_size, 0.1)
    cams = [O.frustum(scene.cv_xyz[i])[1] for i in range(scene.N)]
    pre = O.preprocess(scene, grid, cams, *flags)
    occ = O.occupied_bricks(pre["bricks"], 10)
    ts = O.integrate(inv, pre, grid, limit, use_bricks, occ, want_weight=store_weight)
    want = dict(pre)
    want["counters"], want["occupied"] = pre["bricks"], occ
    if store_weight:
        want["tsdf"], want["weight"] = ts
    else:
        want["tsdf"] = ts
    want["grid"], want["cams"] = grid, np.array(cams)
    return got, want


def _assert_frame(got, want, stages=("morph", "depth", "lab", "depth_b", "sil", "normal", "quality")):
    g = want["grid"]
    assert np.array_equal(got["res"], g["res"])
    assert got["brick_info"]["num_bricks"] == g["num_bricks"]
    assert np.array_equal(got["brick_info"]["res_bricks"], g["res_bricks"])
    assert np.float32(got["brick_info"]["brick_size"]).tobytes() == np.float32(g["brick_size"]).tobytes()
    assert np.array_equal(got["ranges"], g["ranges"])
    assert bits_equal(got["cams"], want["cams"]).all(), mismatch_report("camera positions", got["cams"], want["cams"])
    for k in stages:
        assert bits_equal(got[k], want[k]).all(), mismatch_report(k, got[k], want[k])
    assert np.array_equal(got["counters"], want["counters"]), "brick counters differ"
    assert np.array_equal(got["occupied"], want["occupied"]), "occupied brick list differs"
    assert got["n_occ"] == len(want["occupied"])
    assert bits_equal(got["tsdf"], want["tsdf"]).all(), mismatch_report("tsdf", got["tsdf"], want["tsdf"])
    if "weight" in want:
        assert bits_equal(got["weight"], want["weight"]).all(), mismatch_report("weight", got["weight"], want["weight"])


@pytest.mark.parametrize("fused", ["1", "0"])
def test_frame_bricks_small(small_scene, fused):
    # tunable fused: the staged / fused clear+integrate kernels (1) vs k_fill + k_integrate_bricks (0)
    from rrpy import capi
    capi.set_tunable("fused", int(fused))
    try:
        got, want = _run_both(small_scene, 0.02, (50, 55, 50), use_bricks=True)
    finally:
        capi.set_tunable("fused", 1)
    assert got["last"]["path"] == ("staged" if fused == "1" else "two_kernel"), got["last"]
    assert len(want["occupied"]) > 20, "synthetic scene should occupy bricks"
    assert ((want["tsdf"] > -0.01) & (want["tsdf"] < 0.01)).sum() > 1000, "scene should produce a TSDF band"
    _assert_frame(got, want)


def test_frame_dense_small_with_weight(small_scene):
    got, want = _run_both(small_scene, 0.02, (50, 55, 50), use_bricks=False, store_weight=True)
    _assert_frame(got, want)


@pytest.mark.parametrize("flags", [(False, True, True), (True, False, True), (True, True, False)])
def test_frame_flag_variants(small_scene, flags):
    got, want = _run_both(small_scene, 0.025, (40, 44, 40), use_bricks=True, flags=flags)
    _assert_frame(got, want)


@pytest.mark.parametrize("voxel", [0.03, 0.025])
def test_frame_bricks_with_weight_odd_sizes(small_scene, voxel):
    # 0.03 -> 67x74x67 voxels (row length not a multiple of 4: scalar fill path, 1-voxel brick overlaps); weight volume on
    got, want = _run_both(small_scene, voxel, (50, 55, 50), use_bricks=True, store_weight=True)
    _assert_frame(got, want)


def test_frame_inverse_finer_than_volume(small_scene):
    # reference default: 1 cm voxels over a 7 mm inverse volume (coarse cells smaller than voxels)
    got, want = _run_both(small_scene, 0.03, (96, 100, 90), use_bricks=False)
    _assert_frame(got, want)


def test_staged_ingest_double_buffer(small_scene):
    """rr_stage_frames / rr_swap_frames (the double PBO of double_pixel_buffer.cpp): a staged frame set must not be
    visible before the swap, and a pipelined sequence must give the same volumes as plain uploads."""
    import torch
    from rrpy import capi, synth
    scene = small_scene
    scene2 = synth.rerender(scene, 11)
    inv = synth.analytic_inverse(scene, (40, 44, 40))

    def tsdf_plain(sc):
        fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
        capi.load_scene(fu, scene, inv)
        fu.configure(limit=0.01, voxel_size=0.025, brick_size=0.1, min_voxels=10, use_bricks=True)
        fu.upload_frames(sc.color, sc.depth)
        fu.frame(sync_bricks=True)
        out = fu.download_tsdf()
        fu.close()
        return out

    want1, want2 = tsdf_plain(scene), tsdf_plain(scene2)
    assert not np.array_equal(want1.view(np.uint32), want2.view(np.uint32))

    hc = [torch.from_numpy(s.color).pin_memory() for s in (scene, scene2)]
    hd = [torch.from_numpy(s.depth).pin_memory() for s in (scene, scene2)]
    cb, db = hc[0].numel(), hd[0].numel() * 4
    fu = capi.Fusion(scene.N, scene.W, scene.H, scene.CW, scene.CH)
    capi.load_scene(fu, scene, inv)
    fu.configure(limit=0.01, voxel_size=0.025, brick_size=0.1, min_voxels=10, use_bricks=True)
    with pytest.raises(capi.RRError):
        fu.swap_frames()                      # nothing staged yet
    fu.stage_frames_ptr(hc[0].data_ptr(), cb, hd[0].data_ptr(), db)
    for i in range(4):
        fu.swap_frames()                                                  # frame set i becomes current
        nxt = (i + 1) % 2
        fu.stage_frames_ptr(hc[nxt].data_ptr(), cb, hd[nxt].data_ptr(), db)   # set i+1 copies while set i is fused
        fu.frame(sync_bricks=True)
        got = fu.download_tsdf()
        want = want1 if i % 2 == 0 else want2
        assert bits_equal(got, want).all(), mismatch_report(f"tsdf of pipelined frame {i}", got, want)
    fu.stage_sync()
    fu.close()


def _half_round(a):
    """The value a half2 voxel holds: binary32 -> nearest-even binary16 -> binary32 (numpy's float16 cast is IEEE RN)."""
    with np.errstate(over="ignore"):
        return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


@pytest.mark.parametrize("use_bricks,fused", [(True, "1"), (True, "0"), (False, "1")])
def test_half2_voxels_are_the_rounded_oracle(small_scene, use_bricks, fused, monkeypatch):
    """BASELINE config 5 voxel format: (tsdf, weight) as half2. The arithmetic stays fp32; only the store rounds, so the
    volume must equal the fp16-rounded oracle bit for bit (SURVEY.md 8d: 'report against an fp16-rounded oracle')."""
    import oracle_py as O
    from rrpy import capi, synth
    capi.set_tunable("fused", int(fused))
    try:
        sc = small_scene
        inv = synth.analytic_inverse(sc, (50, 55, 50))
        fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
        capi.load_scene(fu, sc, inv)
        fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=use_bricks, store_weight=capi.VOXELS_HALF2)
        fu.upload_frames(sc.color, sc.depth)
        fu.frame(sync_bricks=True)
        tsdf, weight = fu.download_tsdf(), fu.download_weight()
        fu.close()
    finally:
        capi.set_tunable("fused", 1)
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.02, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], 10)
    wt, ww = O.integrate(inv, pre, grid, 0.01, use_bricks, occ, want_weight=True)
    wt, ww = _half_round(wt), _half_round(ww)
    assert (np.abs(wt) > 0).any() and (ww > 0).any()
    assert bits_equal(tsdf, wt).all(), mismatch_report("half2 tsdf", tsdf, wt)
    assert bits_equal(weight, ww).all(), mismatch_report("half2 weight", weight, ww)
    # the stated fp16 tolerance (SURVEY.md 8d): 11-bit mantissa on |v| <= limit -> within 2^-11 * limit of the fp32 oracle
    full = O.integrate(inv, pre, grid, 0.01, use_bricks, occ)
    ok = np.isfinite(full)
    assert np.abs(tsdf[ok] - full[ok]).max() <= 0.01 * 2.0 ** -11


def test_frame_eight_sensors(monkeypatch):
    """BASELINE config 5 sensor count: 8 sensors on the ring (the reference's uniform arrays stop at 5; the kernels are
    instantiated up to 8). Bricks + dense, bit-identical to the oracle."""
    from rrpy import synth
    sc = synth.make_scene(N=8, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    for use_bricks in (True, False):
        got, want = _run_both(sc, 0.025, (40, 44, 40), use_bricks=use_bricks, store_weight=True)
        _assert_frame(got, want)
    assert len(want["occupied"]) > 10


def test_fuse_frame_graph_replay(small_scene):
    """rr_fuse_frame: one call per frame set, captured as a CUDA graph per frame slot and replayed. Alternating frame sets
    through the double-buffered ingest, a tunable change and a reconfiguration must all keep the volume bit-identical to
    the oracle (and to the call-by-call path)."""
    import oracle_py as O
    from rrpy import capi, synth
    sc = small_scene
    scenes = [sc, synth.rerender(sc, 9)]
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)

    def oracle(scene, voxel):
        grid = O.brick_grid(scene.bbox_min, scene.bbox_max, voxel, 0.1)
        cams = [O.frustum(scene.cv_xyz[i])[1] for i in range(scene.N)]
        pre = O.preprocess(scene, grid, cams)
        occ = O.occupied_bricks(pre["bricks"], 10)
        return O.integrate(inv, pre, grid, 0.01, True, occ), pre["bricks"], occ

    try:
        for voxel in (0.02, 0.025):
            fu.configure(limit=0.01, voxel_size=voxel, brick_size=0.1, min_voxels=10, use_bricks=True)
            want = [oracle(s_, voxel) for s_ in scenes]
            fu.upload_frames(scenes[0].color, scenes[0].depth)
            fu.frame()                                           # builds the z table (an extra launch, and an allocation)
            l0 = fu.launch_count()
            per_frame = None
            for i in range(7):                                   # capture slot A, capture slot B, replays, re-capture ...
                k = i % 2
                fu.upload_frames(scenes[k].color, scenes[k].depth)      # stage + swap: the frame slot alternates
                l1 = fu.launch_count()
                if i == 4:
                    capi.set_tunable("zchunk", 7)                # new launch shape: the captured graphs must not be reused
                fu.fuse_frame()
                n = fu.launch_count() - l1
                per_frame = per_frame or n
                assert n == per_frame, "a replayed frame must account for the same kernel launches as a direct one"
                tsdf = fu.download_tsdf()
                counters, occupied = fu.download_bricks()
                assert np.array_equal(counters, want[k][1]) and np.array_equal(occupied, want[k][2])
                assert fu.bricks_count()[0] == len(want[k][2])
                assert bits_equal(tsdf, want[k][0]).all(), mismatch_report(f"tsdf frame {i} voxel {voxel}", tsdf, want[k][0])
            assert fu.launch_count() > l0
            capi.set_tunable("zchunk", 13)
        # the call-by-call path gives the same volume
        fu.upload_frames(scenes[0].color, scenes[0].depth)
        fu.frame(sync_bricks=True)
        assert bits_equal(fu.download_tsdf(), want[0][0]).all()
    finally:
        capi.set_tunable("zchunk", 13)
        fu.close()



def test_configure_refuses_volumes_beyond_32_bit_voxel_indices(small_scene):
    """rr_configure: 2^31 voxels or more would wrap the kernels' 32-bit voxel offsets (the allocation itself would fit HBM),
    so the configuration is refused with RR_ERR_UNSUPPORTED before anything is allocated."""
    from rrpy import capi
    sc = small_scene[0] if isinstance(small_scene, tuple) else small_scene
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    fu.set_bbox(sc.bbox_min, sc.bbox_max)
    ext = float(np.max(np.asarray(sc.bbox_max) - np.asarray(sc.bbox_min)))
    with pytest.raises(capi.RRError, match="2\\^31"):
        fu.configure(limit=0.01, voxel_size=ext / 1400.0, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.close()


@pytest.mark.parametrize("n_sensors", [2, 5])
def test_staged_integrator_paths_are_bit_identical(n_sensors):
    """The TMA-staged integrator (csrc/rr_integrate_staged.cu) under launch shapes that exercise every path: tiny tiles
    (most footprints exceed them: items evaluated from global memory beside staged ones), small y / z chunks (many items,
    the slot ring wraps), both consumer-warp variants, no run-ahead cap, unthrottled clear. Tunables must never change
    results: every volume equals the oracle's bit for bit, the kernel stays selected and raises no consistency flag."""
    import oracle_py as O
    from rrpy import capi, synth
    sc = synth.make_scene(N=n_sensors, W=128, H=106, CW=160, CH=136, cv_res=(32, 32, 64))
    inv = synth.analytic_inverse(sc, (40, 44, 40))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.0125, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], 10)
    want = O.integrate(inv, pre, grid, 0.01, True, occ)
    assert len(occ) > 20
    defaults = dict(stage_tile=0, stage_zchunk=13, stage_ychunk=0, stage_cwarps=0, stage_tail_cap=2, stage_fill_depth=0, stage_bulk_fill=4, stage_fill_rows=16)
    variants = [dict(), dict(stage_tile=8), dict(stage_tile=14, stage_zchunk=4), dict(stage_ychunk=2, stage_zchunk=3), dict(stage_cwarps=11),
                dict(stage_tail_cap=0, stage_fill_depth=-1, stage_bulk_fill=16), dict(stage_fill_rows=5, stage_tail_cap=1),
                dict(stage_ychunk=3), dict(stage_ychunk=7, stage_cwarps=11)]
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.0125, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    seen_oversize = False
    try:
        for v in variants:
            for k, val in {**defaults, **v}.items():
                capi.set_tunable(k, val)
            fu.fuse_frame()
            fu.frame()                               # the call-by-call form too (a second integrate of the same frame set)
            got = fu.download_tsdf()
            info = fu.integrator_info()
            assert info["staged"] == 1 and info["flags"] == 0, (v, info)
            seen_oversize = seen_oversize or info["oversize_pairs"] > 0
            assert bits_equal(got, want).all(), mismatch_report(f"tsdf with {v}", got, want)
        fu.integrate()                               # a repeated integrate without a brick update in between
        assert bits_equal(fu.download_tsdf(), want).all()
    finally:
        for k, val in defaults.items():
            capi.set_tunable(k, val)
        fu.close()
    assert seen_oversize
