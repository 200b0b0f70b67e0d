"""GPU vs the reference's own shaders, directly (no oracle in between). Runs last in the suite (file name) so that its
looser, formulation-dependent bars can never mask a result of the bit-exact parity tests.

The shaders run live where oracle/_ref/libref_glsl.so was built from the reference tree; everywhere else the kernels are
compared with what those shaders computed for tools/make_golden.py::glsl_scene (tests/golden/ref_glsl_*.npz)."""
import hashlib

import numpy as np
import pytest

from conftest import assert_points, assert_raymarch, assert_trigrid, bits_equal, gold

pytestmark = pytest.mark.gpu

GOLDEN_VIEW = dict(eye=(1.2, 1.4, 1.6), at=(0.0, 1.1, 0.0), fovy=50.0, w=160, h=90)      # tools/make_golden.py::RM_VIEW


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _golden_frame(use_bricks=True, skip_space=False):
    """One fused frame of tools/make_golden.py::glsl_scene on the GPU, with the golden's voxel size and inverse volume."""
    from rrpy import capi, synth
    g = gold("ref_glsl_stages.npz")
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, g["inv"])
    fu.configure(limit=0.01, voxel_size=float(g["voxel"]), brick_size=0.1, min_voxels=10, use_bricks=use_bricks, skip_space=skip_space)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame(sync_bricks=True)
    return fu, g


def _golden_view():
    from rrpy import synth
    V = GOLDEN_VIEW
    return synth.look_at(V["eye"], V["at"]), synth.perspective(V["fovy"], V["w"] / V["h"], 0.1, 10.0)


def test_kernels_against_the_reference_shader_outputs():
    """The CUDA path's full chain against the reference shaders' full chain as committed (ref_glsl_stages.npz, every stage fed
    by the shaders' own previous stage), bricked and dense: the stages with the bars of the live comparison below, the volume
    with the oracle's bar on the same golden. The bricked volume is also the oracle's, bit for bit (the raymarch golden's hash)."""
    for use_bricks, key in ((True, "tsdf_bricks"), (False, "tsdf_dense")):
        fu, g = _golden_frame(use_bricks)
        got = {k: fu.download_stage(k) for k in ("morph", "depth", "lab", "depth_b", "sil", "normal", "quality")}
        counters, occupied = fu.download_bricks()
        tsdf = fu.download_tsdf()
        fu.close()
        if use_bricks:
            assert np.array_equal(counters, g["pre_bricks"]) and np.array_equal(occupied, g["occupied"]) and len(occupied) > 10
            assert _sha(tsdf) == str(gold("ref_glsl_raymarch.npz")["tsdf_sha"]), "the kernels' volume differs from the oracle's"
        assert bits_equal(got["morph"], g["pre_morph"]).all() and bits_equal(got["sil"], g["pre_sil"]).all()
        for k, tol in dict(depth=2e-6, lab=2e-4, depth_b=2e-6, normal=2e-4, quality=4e-5).items():
            want = g["pre_" + k]
            assert ((got[k] != got[k]) == (want != want)).all(), k
            ok = np.isfinite(got[k]) & np.isfinite(want)
            assert np.abs(got[k][ok] - want[ok]).max() <= tol, f"{k}: {np.abs(got[k][ok] - want[ok]).max()}"
        want = g[key]
        assert (np.abs(want) < 0.0099).sum() > 200, "the golden volume must hold in-band voxels"
        assert (np.isnan(tsdf) == np.isnan(want)).all(), key
        ok = np.isfinite(tsdf) & np.isfinite(want)
        # the oracle's bar on the same golden (test_oracle_against_reference_shader_goldens): the kernels match the oracle bit for bit
        assert np.abs(tsdf[ok].astype(np.float64) - want[ok]).max() <= 2e-5 * 0.01, key


def test_raymarch_kernel_against_the_reference_shader_outputs():
    """rr_raymarch against tsdf_raymarch.fs + shading.glsl as committed (ref_glsl_raymarch.npz: the shader run on the oracle's
    volume, which the kernels reproduce bit for bit), every shade mode with the cube-proxy march, and the skipSpace branch fed
    the reference's rasterised brick depth peels against the kernels' brick hull."""
    g = gold("ref_glsl_raymarch.npz")
    mv, pr = _golden_view()
    W, H = GOLDEN_VIEW["w"], GOLDEN_VIEW["h"]
    fu, _ = _golden_frame(skip_space=False)
    assert _sha(fu.download_tsdf()) == str(g["tsdf_sha"]), "the kernels' volume differs from the golden's input volume"
    for mode in range(4):
        rgba, depth = fu.raymarch(mv, pr, W, H, shade_mode=mode)
        got = dict(rgba=rgba, depth=depth, samples=fu.download_num_samples(W, H))
        assert_raymarch(got, g[f"rgba{mode}"], g["depth"], g["samples"], g["hit"], f"mode {mode}", np.asarray(pr))
    fu.close()
    fu, _ = _golden_frame(skip_space=True)
    rgba, depth = fu.raymarch(mv, pr, W, H, shade_mode=1)
    got = dict(rgba=rgba, depth=depth, samples=fu.download_num_samples(W, H))
    fu.close()
    assert_raymarch(got, g["skip_rgba"], g["skip_depth"], g["skip_samples"], g["skip_hit"], "skipSpace", np.asarray(pr), sample_flips=0.01)


def test_point_and_trigrid_kernels_against_the_reference_shader_outputs():
    """rr_draw_points, rr_draw_calibs and rr_draw_trigrid against points.{vs,gs,fs}, calib_vis.{vs,fs} and trigrid_accum.{vs,gs,fs}
    + trigrid_normalize.fs as committed (ref_glsl_points.npz, ref_glsl_trigrid.npz: the shaders run on the oracle's maps and
    volume, which the kernels reproduce bit for bit), every shade mode, the triangle mesh also from inside the volume."""
    gp, gt = gold("ref_glsl_points.npz"), gold("ref_glsl_trigrid.npz")
    from rrpy import synth
    mv, pr = _golden_view()
    W, H = GOLDEN_VIEW["w"], GOLDEN_VIEW["h"]
    fu, _ = _golden_frame()
    assert _sha(fu.download_stage("quality")) == str(gt["quality_sha"]), "the kernels' maps differ from the golden's input maps"
    assert _sha(fu.download_tsdf()) == str(gp["tsdf_sha"]), "the kernels' volume differs from the golden's input volume"
    for mode in range(4):
        assert_points(fu.draw_points(mv, pr, W, H, shade_mode=mode), (gp[f"points_rgba{mode}"], gp[f"points_depth{mode}"]), f"points mode {mode}")
    assert_points(fu.draw_calibs(mv, pr, W, H, active_kinect=0, limit=0.01), (gp["calibs_rgba"], gp["calibs_depth"]), "calibs")
    for tag, eye in (("", GOLDEN_VIEW["eye"]), ("in_", tuple(float(x) for x in gt["eye_in"]))):
        mv = synth.look_at(eye, GOLDEN_VIEW["at"])
        for mode in range(4):
            assert_trigrid(fu.draw_trigrid(mv, pr, W, H, shade_mode=mode, min_length=float(gt["min_length"])),
                           (gt[f"{tag}rgba{mode}"], gt[f"{tag}depth{mode}"]), f"trigrid {tag}mode {mode}")
    fu.close()


def test_kernels_against_the_reference_shaders_directly(small_scene):
    """The CUDA path against the reference's OWN shaders run on the CPU (oracle/_ref/libref_glsl.so: glsl/pre_*.fs,
    inc_*.glsl, tsdf_integration.vs compiled as C++, see oracle/glsl_host/), full chain on both sides, no oracle in between.
    The shader host environment uses a different float formulation (mix() without fma, libm pow), so the bars are BASELINE's:
    brick counters and occupied list bit-exact, silhouettes identical, normals within 2e-4 absolute (unit vectors),
    TSDF within 3e-5 of the truncation distance over the whole chained pipeline (1e-5 on identical inputs is the CPU test)."""
    import oracle_py as O
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import capi, synth
    sc = small_scene
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame(sync_bricks=True)
    got = {k: fu.download_stage(k) for k in ("morph", "depth", "lab", "depth_b", "sil", "normal", "quality")}
    counters, occupied = fu.download_bricks()
    tsdf = fu.download_tsdf()
    fu.close()

    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.02, 0.1)       # host geometry (pinned against volume_sampler.cpp)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    ref = G.preprocess(sc, grid, cams)
    ref_occ = O.occupied_bricks(ref["bricks"], 10)
    ref_tsdf = G.integrate(inv, ref, grid, 0.01, True, ref_occ)
    assert np.array_equal(counters, ref["bricks"]) and np.array_equal(occupied, ref_occ) and len(ref_occ) > 50
    assert bits_equal(got["morph"], ref["morph"]).all() and bits_equal(got["sil"], ref["sil"]).all()
    for k, tol in dict(depth=2e-6, lab=2e-4, depth_b=2e-6, normal=2e-4, quality=4e-5).items():
        assert ((got[k] != got[k]) == (ref[k] != ref[k])).all(), k
        ok = np.isfinite(got[k]) & np.isfinite(ref[k])
        assert np.abs(got[k][ok] - ref[k][ok]).max() <= tol, f"{k}: {np.abs(got[k][ok] - ref[k][ok]).max()}"
    assert (np.isnan(tsdf) == np.isnan(ref_tsdf)).all()
    ok = np.isfinite(tsdf) & np.isfinite(ref_tsdf)
    assert np.abs(tsdf[ok].astype(np.float64) - ref_tsdf[ok]).max() <= 3e-5 * 0.01    # measured 1.2e-5 (CPU dry run)


@pytest.mark.parametrize("eye,mode", [((-2.0, 1.0, 1.2), 0), ((1.6, 1.5, 2.2), 1)])
def test_raymarch_kernel_against_the_reference_shader_directly(small_scene, eye, mode):
    """rr_raymarch (cube-proxy march, space skipping off) against glsl/tsdf_raymarch.fs + shading.glsl run on the CPU on the
    volume the kernels integrated: same fragments, same sample counts, window depth within 1e-5 (BASELINE: 1 mm), colours
    within 2e-3."""
    import oracle_py as O
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import capi, synth
    sc = small_scene
    VW, VH = 320, 180
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True, skip_space=False)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame(sync_bricks=True)
    tsdf = fu.download_tsdf()
    pre = {k: fu.download_stage(k) for k in ("depth_b", "quality", "normal")}
    mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
    rgba, depth = fu.raymarch(mv, pr, VW, VH, shade_mode=mode)
    samples = fu.download_num_samples(VW, VH)
    fu.close()
    want = G.raymarch(tsdf, 0.01, inv, sc, pre, mv, pr, VW, VH, mode)
    hit = depth < 1.0
    assert np.array_equal(hit, want["hit"] > 0) and hit.sum() > 1000
    assert np.array_equal(samples, want["samples"])
    assert np.abs(depth - want["depth"]).max() <= 1e-5
    assert (np.isnan(rgba) == np.isnan(want["rgba"])).all()
    ok = np.isfinite(rgba) & np.isfinite(want["rgba"])
    assert np.abs(rgba[ok] - want["rgba"][ok]).max() <= 2e-3


@pytest.mark.parametrize("eye", [(1.6, 1.5, 2.2), (0.2, 1.2, 0.3)])
def test_trigrid_and_points_kernels_against_the_reference_shaders_directly(small_scene, eye):
    """rr_draw_trigrid and rr_draw_points on the maps the kernels pre-processed, against glsl/trigrid_accum.{vs,gs,fs} +
    trigrid_normalize.fs and glsl/points.{vs,gs,fs} run on the CPU on the same maps (oracle/_ref/libref_glsl.so), no oracle in
    between: same coverage up to a handful of threshold pixels, window depth within 2e-5, colours within 5e-5 (trigrid) /
    2e-5 (points) - the bars of the oracle's own pin in tests/test_oracle_cpu.py."""
    import ref_glsl_py as G
    if not G.available() or not hasattr(G.lib(), "rg_draw_trigrid"):
        pytest.skip("oracle/_ref/libref_glsl.so not built with the trigrid shaders (needs the reference tree at build time)")
    from rrpy import capi, synth
    sc = small_scene
    VW, VH = 200, 112
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, synth.analytic_inverse(sc, (40, 44, 40)))
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.frame(sync_bricks=True)
    pre = {k: fu.download_stage(k) for k in ("depth_b", "quality", "normal")}
    mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
    for mode in (0, 1, 3):
        rgba, depth = fu.draw_trigrid(mv, pr, VW, VH, shade_mode=mode, min_length=0.06)
        w_rgba, w_depth = G.draw_trigrid(sc, pre, mv, pr, VW, VH, mode, 0.06)
        cov, w_cov = depth < 1.0, w_depth < 1.0
        assert w_cov.sum() > 100 and (cov != w_cov).sum() <= max(2, int(0.002 * w_cov.sum())), f"trigrid mode {mode}: coverage"
        both = cov & w_cov
        assert np.abs(depth - w_depth)[both].max() <= 2e-5
        d = np.abs(rgba - w_rgba)[both]
        assert (d > 5e-5).any(axis=-1).sum() <= max(2, int(0.002 * both.sum())), f"trigrid mode {mode}: colour differs by up to {d.max()}"
        rgba, depth = fu.draw_points(mv, pr, VW, VH, shade_mode=mode)
        w_rgba, w_depth = G.draw_points(sc, pre, mv, pr, VW, VH, mode)
        cov, w_cov = depth < 1.0, w_depth < 1.0
        assert w_cov.sum() > 50 and (cov != w_cov).sum() <= max(2, int(0.002 * w_cov.sum())), f"points mode {mode}: coverage"
        same = cov & w_cov & (np.abs(depth - w_depth) <= 2e-7)
        assert same.sum() >= 0.995 * (cov & w_cov).sum()
        assert np.abs(rgba - w_rgba)[same].max() <= 2e-5
    fu.close()


def test_empty_frame_set_on_the_gpu():
    """Edge case: a frame set without a single depth return. No brick marks, an empty occupied list, a volume that is -limit
    everywhere, a raymarch without samples - bit-identical to the oracle (whose empty-frame behaviour is checked against the
    reference's shaders in tests/test_oracle_cpu.py::test_empty_frame_set_oracle_and_reference_shaders)."""
    import dataclasses
    import oracle_py as O
    from rrpy import capi, synth
    sc = synth.make_scene(N=2, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48), seed=3)
    sc = dataclasses.replace(sc, depth=np.zeros_like(sc.depth))
    inv = synth.analytic_inverse(sc, (30, 33, 30))
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=0.01, voxel_size=0.04, brick_size=0.1, min_voxels=10, use_bricks=True, skip_space=True)
    fu.upload_frames(sc.color, sc.depth)
    n_occ, ratio = fu.frame(sync_bricks=True)
    got = {k: fu.download_stage(k) for k in ("morph", "depth", "lab", "depth_b", "sil", "normal", "quality")}
    counters, occupied = fu.download_bricks()
    tsdf = fu.download_tsdf()
    mv, pr = synth.look_at((1.6, 1.5, 2.2), (0.0, 1.1, 0.0)), synth.perspective(50.0, 16 / 9, 0.1, 10.0)
    rgba, depth = fu.raymarch(mv, pr, 96, 54, shade_mode=1)
    samples = fu.download_num_samples(96, 54)
    fu.fuse_frame(); fu.fuse_frame()                      # the graph path on an empty occupied list
    assert fu.bricks_count()[0] == 0
    tsdf2 = fu.download_tsdf()
    fu.close()
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.04, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    assert n_occ == 0 and ratio == 0.0 and len(occupied) == 0 and not counters.any()
    for k in got:
        assert bits_equal(got[k], pre[k]).all(), k
    assert (tsdf == np.float32(-0.01)).all() and (tsdf2 == np.float32(-0.01)).all()
    assert (depth == 1.0).all() and not samples.any() and not rgba.any()
