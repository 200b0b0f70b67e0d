"""Parity at BASELINE.json's full size (4 sensors, 512x424 depth, 512^3 volume) through size-independent properties —
the scalar oracle would need minutes per frame here, so it checks a sample of bricks and the rest is covered by
identities between independent GPU paths:
  * the TMA-staged clear+integrate kernel == k_fill + k_integrate_bricks (two different kernels), bit for bit;
  * dense integration == brick integration inside occupied bricks; outside them the brick path holds exactly -limit;
  * 2 z-slabs + composite == single volume (integration slices and the 1280x720 raymarched image);
  * the oracle, run on a random sample of occupied bricks only, agrees bit for bit with the volume."""
import os

import numpy as np
import pytest

from conftest import bits_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full():
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs()
    return dict(bench=bench, capi=capi, scene=scenes[0], inv=inv, voxel=voxel)


def _ctx(full, use_bricks=True):
    b, capi, sc = full["bench"], full["capi"], full["scene"]
    fu = capi.Fusion(b.N_SENSORS, b.W, b.H, b.CW, b.CH)
    capi.load_scene(fu, sc, full["inv"])
    fu.configure(limit=b.LIMIT, voxel_size=full["voxel"], brick_size=b.BRICK, min_voxels=b.MIN_VOX, use_bricks=use_bricks)
    fu.upload_frames(sc.color, sc.depth)
    return fu


def test_fullsize_paths_agree(full):
    import oracle_py as O
    b, capi, sc = full["bench"], full["capi"], full["scene"]
    fu = _ctx(full)
    assert tuple(fu.volume_res()) == (512, 512, 512)
    n_occ, ratio = fu.frame(sync_bricks=True)
    assert fu.integrator_last()["path"] == "staged", fu.integrator_last()
    fused = fu.download_tsdf()
    counters, occ = fu.download_bricks()
    ranges = fu.brick_ranges()
    assert 100 < n_occ < 2000 and len(occ) == n_occ
    # (1) the two-kernel path
    capi.set_tunable("fused", 0)
    try:
        fu.frame(sync_bricks=True)
        assert fu.integrator_last()["path"] == "two_kernel", fu.integrator_last()
        unfused = fu.download_tsdf()
    finally:
        capi.set_tunable("fused", 1)
    assert bits_equal(fused, unfused).all(), f"{(~bits_equal(fused, unfused)).sum()} voxels differ between fused and two-kernel paths"
    del unfused
    # (2) dense vs bricks
    mask = np.zeros(fused.shape, bool)
    for r in ranges[occ]:
        mask[r[4]:r[5], r[2]:r[3], r[0]:r[1]] = True
    assert (fused[~mask] == np.float32(-b.LIMIT)).all()
    fu.configure(limit=b.LIMIT, voxel_size=full["voxel"], brick_size=b.BRICK, min_voxels=b.MIN_VOX, use_bricks=False)
    fu.frame(sync_bricks=True)
    dense = fu.download_tsdf()
    assert bits_equal(dense[mask], fused[mask]).all()
    band = (fused > -b.LIMIT) & (fused < b.LIMIT)
    assert band.sum() > 100000
    del dense
    # (4) oracle on a sample of occupied bricks (same pre-processing outputs, taken from the GPU stages it already matches
    #     bit for bit at small sizes): integrate only those bricks on the CPU
    pre = {k: fu.download_stage(k) for k in ("sil", "depth_b", "quality")}
    fu.close()
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, full["voxel"], b.BRICK)
    assert np.array_equal(grid["ranges"], ranges)
    rng = np.random.default_rng(3)
    sample = np.sort(rng.choice(occ, size=24, replace=False)).astype(np.uint32)
    want = O.integrate(full["inv"], pre, grid, b.LIMIT, True, sample)
    for r in ranges[sample]:
        sl = (slice(r[4], r[5]), slice(r[2], r[3]), slice(r[0], r[1]))
        assert bits_equal(fused[sl], want[sl]).all()


def test_fullsize_whole_frame_matches_the_oracle(full):
    """BASELINE's headline configuration against the oracle IN FULL: all seven stage images of the 4 x 512 x 424 pre-processing,
    the brick counters, the occupied list and every voxel of the 512^3 volume, bit for bit (the oracle needs ~0.5 s for the
    whole chain on the host cores), then the 1280x720 raymarch of config 2 on that volume."""
    import oracle_py as O
    from rrpy import capi, synth
    b, sc = full["bench"], full["scene"]
    fu = _ctx(full)
    n_occ, _ = fu.frame(sync_bricks=True)
    info = fu.integrator_info()
    assert info["staged"] == 1 and info["flags"] == 0, info          # the TMA-staged integrator is the one that ran, and it is healthy
    got = {k: fu.download_stage(k) for k in capi.STAGES}
    counters, occupied = fu.download_bricks()
    tsdf = fu.download_tsdf()
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, full["voxel"], b.BRICK)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], b.MIN_VOX)
    for k in ("morph", "depth", "lab", "depth_b", "sil", "normal", "quality"):
        assert bits_equal(got[k], pre[k]).all(), f"stage {k}: {(~bits_equal(got[k], pre[k])).sum()} values differ"
    assert np.array_equal(counters, pre["bricks"]), "brick counters differ"
    assert np.array_equal(occupied, occ) and n_occ == len(occ), "occupied brick list differs"
    want = O.integrate(full["inv"], pre, grid, b.LIMIT, True, occ)
    assert bits_equal(tsdf, want).all(), f"{(~bits_equal(tsdf, want)).sum()} of 512^3 voxels differ from the oracle"
    assert ((want > -b.LIMIT) & (want < b.LIMIT)).sum() > 100000
    # config 2's view size on this volume
    VW, VH = 1280, 720
    mv, pr = synth.look_at((1.7, 1.6, 2.3), (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
    for shade_mode in (0, 1):
        rgba, depth = fu.raymarch(mv, pr, VW, VH, shade_mode=shade_mode)
        ns = fu.download_num_samples(VW, VH)
        w = O.raymarch(want, b.LIMIT, full["inv"], sc, pre, grid, occ, mv, pr, VW, VH, shade_mode, skip_space=True)
        assert (w["depth"] < 1.0).sum() > 20000
        assert bits_equal(depth, w["depth"]).all() and bits_equal(rgba, w["rgba"]).all() and bits_equal(ns, w["samples"]).all()
    fu.close()


def test_fullsize_slabs_agree(full):
    import torch
    from rrpy import multigpu as M, synth
    b = full["bench"]
    VW, VH = 1280, 720
    mv, pr = synth.look_at((1.7, 1.6, 2.3), (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
    one = _ctx(full)
    one.frame(sync_bricks=True)
    want_rgba, want_depth = one.raymarch(mv, pr, VW, VH, shade_mode=1)
    want = one.download_tsdf()
    one.close()
    assert (want_depth < 1).sum() > 20000
    records = torch.empty((2, VW * VH, M.RECORD_FLOATS), dtype=torch.float32, device="cuda")
    parts = []
    for r in range(2):
        fu = _ctx(full)
        z0, z1 = M.slab_range(r, 2, 512)
        fu.set_slab(z0, z1)
        fu.frame(sync_bricks=True)
        got = fu.download_tsdf()
        h = M.halo(b.LIMIT, 512)
        lo, hi = max(0, z0 - h), min(512, z1 + h)
        assert bits_equal(got[lo:hi], want[lo:hi]).all()
        del got
        fu.raymarch_partial(mv, pr, VW, VH, records[r].data_ptr(), shade_mode=1)
        fu.synchronize()
        parts.append(fu)
    rgba, depth = parts[0].composite(records.data_ptr(), 2, VW, VH)
    for fu in parts:
        fu.close()
    assert bits_equal(depth, want_depth).all() and bits_equal(rgba, want_rgba).all()
