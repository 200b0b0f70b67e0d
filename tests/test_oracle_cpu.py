"""CPU tests (no GPU): the oracle (scalar restatement) against
  * golden vectors produced by REAL reference code (tests/golden/ref_*.npz, made by tools/make_golden.py from oracle/_ref),
  * the live oracle/_ref library when it is present (build container only),
  * known answers of the arithmetic pins (GL filtering equations, deterministic pow),
  * the reference's OWN shaders (pre-processing, integration, raymarch + shading, colour fill), compiled as C++ and run on
    the CPU (oracle/_ref/libref_glsl.so, oracle/glsl_host/) - live where built, and as tests/golden/ref_glsl_*.npz elsewhere,
  * self-regression pins of the restatement (the reference ships no tests of its own).
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLD, assert_points, assert_raymarch, assert_trigrid, bits_equal, gold


@pytest.fixture(scope="module")
def O():
    import oracle_py
    return oracle_py


# ------------------------------------------------------------------------------------------------ reference goldens

def test_frustum_matches_reference_golden(O):
    g = gold("ref_calib_invert.npz")
    planes, cam = O.frustum(g["cv_xyz"])
    assert bits_equal(planes, g["planes"]).all()
    assert bits_equal(cam, g["cam"]).all()
    L = O.lib()
    inside = np.array([L.ro_frustum_inside(np.ascontiguousarray(planes), np.ascontiguousarray(p)) for p in g["points"]], np.int32)
    assert np.array_equal(inside, g["inside"])
    assert 0.02 < inside.mean() < 0.9, "the sample should straddle the frustum"


@pytest.mark.parametrize("brute", [False, True])
def test_calib_invert_matches_reference_golden(O, brute):
    g = gold("ref_calib_invert.npz")
    inv = O.calib_invert(g["cv_xyz"], g["bbox_min"], g["bbox_max"], g["out_res"], brute=brute)
    assert inv.shape == g["inv"].shape
    valid = g["inv"][..., 3] > 0
    assert 0.3 < valid.mean() < 1.0
    assert (g["inv"][~valid] == -1.0).all()
    assert bits_equal(inv, g["inv"]).all(), f"{(~bits_equal(inv, g['inv'])).sum()} values differ from calibration_inverter.cpp"


def test_calib_invert_roundtrip_property(O):
    """cv_xyz(cv_xyz_inv(p)) ~ p: what the reference checks visually (calib_vis.vs:26-37)."""
    g = gold("ref_calib_invert.npz")
    xyz, inv = g["cv_xyz"], g["inv"]
    Z, Y, X, _ = xyz.shape
    oz, oy, ox, _ = inv.shape
    bmin, bmax = g["bbox_min"], g["bbox_max"]
    L = O.lib()
    errs = []
    out = np.zeros(4, np.float32)
    for (z, y, x) in np.argwhere(inv[..., 3] > 0)[::37]:
        uvd = inv[z, y, x, :3]
        if (uvd < 1.5 / np.array([X, Y, Z])).any() or (uvd > 1 - 1.5 / np.array([X, Y, Z])).any():
            continue   # IDW of 8 neighbours is biased at the volume border
        L.ro_kat_tex3d(np.ascontiguousarray(xyz), 3, X, Y, Z, uvd[0], uvd[1], uvd[2], out)
        p = bmin + (np.array([x, y, z]) + 0.5) / np.array([ox, oy, oz]) * (bmax - bmin)
        errs.append(np.linalg.norm(out[:3] - p))
    assert len(errs) > 50
    assert np.median(errs) < 0.05, "inverse lookup should land within a fraction of a calibration cell (cells are ~0.15 m here)"


def test_volume_file_format_matches_reference_golden():
    """CalibrationVolume<T> layout: uint32 res[3]; float limits[2]; T data[] (calibration_volume.hpp:18-27)."""
    g = gold("ref_volume_file.npz")
    data = g["data"]
    Z, Y, X, ch = data.shape
    want = np.array([X, Y, Z], np.uint32).tobytes() + np.array([0.5, 4.5], np.float32).tobytes() + data.tobytes()
    assert g["raw"].tobytes() == want
    assert np.array_equal(g["back"], data)
    from rrpy import volume_io
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "v.cv_xyz_inv")
        volume_io.write_volume(p, data, (0.5, 4.5))
        assert open(p, "rb").read() == want
        back, lim = volume_io.read_volume(p, ch)
        assert np.array_equal(back, data) and tuple(lim) == (0.5, 4.5)


def test_brick_ranges_match_reference_contained_voxels(O):
    """divideBox + VolumeSampler::containedVoxels: per-brick voxel lists, order y -> x -> z (volume_sampler.cpp:50-62)."""
    g = gold("ref_bricks.npz")
    for ci in range(4):
        dims = g[f"c{ci}_dims"].astype(int)
        voxel, brick = g[f"c{ci}_voxel_brick"]
        bmax = g[f"c{ci}_bmax"]
        grid = O.brick_grid(np.zeros(3, np.float32), bmax, voxel, brick)
        assert np.array_equal(grid["res"], dims.astype(np.uint32))
        _, raw = O.divide_box_args(np.zeros(3, np.float32), bmax, grid["brick_size"], grid["res"], want_raw=True)
        assert (raw[:, 1::2] <= dims).all(), "index lists must not run past the volume (aliasing is defined as dropped)"
        off = 0
        for b, n in zip(g[f"c{ci}_sel"], g[f"c{ci}_counts"]):
            r = grid["ranges"][b]
            want = g[f"c{ci}_indices"][off:off + n]
            off += n
            ys, xs, zs = np.meshgrid(np.arange(r[2], r[3]), np.arange(r[0], r[1]), np.arange(r[4], r[5]), indexing="ij")
            mine = (zs * dims[0] * dims[1] + ys * dims[0] + xs).reshape(-1).astype(np.uint32)
            assert np.array_equal(mine, want), f"case {ci} brick {b}"
    # voxel centres (volume_sampler.cpp:33-48)
    pos = g["positions_7_5_3"]
    z, y, x = np.meshgrid(np.arange(3), np.arange(5), np.arange(7), indexing="ij")
    for a, (idx, n) in enumerate(((x, 7), (y, 5), (z, 3))):
        mine = (idx.astype(np.float32) + np.float32(0.5)) * (np.float32(1.0) / np.float32(n))
        assert bits_equal(mine, pos[..., a]).all()
    # glm::round as used by setBrickSize (recon_integration.cpp:475)
    L = O.lib()
    mine = np.array([L.ro_adjust_brick_size(np.float32(1.0), v) for v in g["round_in"]], np.float32)
    assert bits_equal(mine, g["round_out"]).all()


def test_draw_uniforms_match_reference_golden(O):
    """recon_integration.cpp:183-206 evaluated with gloost / glm in float vs the oracle's double-then-round inverses."""
    g = gold("ref_draw_uniforms.npz")
    for v in g["views"]:
        mv, pr, i2e, nm, cam = v[:16], v[16:32], v[32:48], v[48:64], v[64:67]
        u = O.raymarch_uniforms(mv, pr, g["bbox_min"], g["bbox_max"], 320, 180)
        np.testing.assert_allclose(u[:16], i2e, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(u[64:80], nm, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(u[80:83], cam, rtol=2e-5, atol=2e-6)


def test_trilinear_agrees_with_reference_get_trilinear(O):
    """DataTypes.cpp getTrilinear (voxel-unit coordinates, weights w*a + (1-w)*b) vs the GL LINEAR restatement
    (normalised coordinates, fma form): same value up to rounding."""
    g = gold("ref_trilinear.npz")
    xyz = gold("ref_calib_invert.npz")["cv_xyz"]
    Z, Y, X, _ = xyz.shape
    L = O.lib()
    out = np.zeros(4, np.float32)
    for c, want in zip(g["coords"], g["values"]):
        s, t, r = (c[0] + 0.5) / X, (c[1] + 0.5) / Y, (c[2] + 0.5) / Z
        L.ro_kat_tex3d(np.ascontiguousarray(xyz), 3, X, Y, Z, s, t, r, out)
        np.testing.assert_allclose(out[:3], want, rtol=0, atol=3e-5)


# ------------------------------------------------------------------------------------------------ live oracle/_ref

def _ref():
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    return ref_py


def test_live_reference_inverter_and_frustum(O):
    R = _ref()
    from rrpy import synth
    sc = synth.make_scene(N=2, W=64, H=53, CW=80, CH=68, cv_res=(12, 14, 24), seed=4321)
    for i in range(2):
        p, c = R.frustum(sc.cv_xyz[i])
        po, co = O.frustum(sc.cv_xyz[i])
        assert bits_equal(p, po).all() and bits_equal(c, co).all()
        a = R.calib_invert(sc.cv_xyz[i], sc.bbox_min, sc.bbox_max, (17, 19, 15))
        b = O.calib_invert(sc.cv_xyz[i], sc.bbox_min, sc.bbox_max, (17, 19, 15))
        assert bits_equal(a, b).all()


def test_goldens_are_current():
    """tests/golden was generated by tools/make_golden.py from the reference present in this container."""
    R = _ref()
    g = gold("ref_calib_invert.npz")
    inv = R.calib_invert(g["cv_xyz"], g["bbox_min"], g["bbox_max"], g["out_res"])
    assert bits_equal(inv, g["inv"]).all()
    import ref_glsl_py as G
    if G.available():
        import oracle_py as O_
        from rrpy import synth
        gs = gold("ref_glsl_stages.npz")
        sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)
        grid = O_.brick_grid(sc.bbox_min, sc.bbox_max, float(gs["voxel"]), 0.1)
        pre = G.preprocess(sc, grid, [O_.frustum(sc.cv_xyz[0])[1]])
        for k, v in pre.items():
            assert bits_equal(v, gs["pre_" + k]).all() if v.dtype == np.float32 else np.array_equal(v, gs["pre_" + k]), k


# ------------------------------------------------------------------------------------------------ the reference's shaders, run
# oracle/_ref/libref_glsl.so = the reference's own glsl/pre_*.fs, inc_*.glsl and tsdf_integration.vs compiled as C++ against a
# GLSL host environment (oracle/glsl_host/) that evaluates filtering and built-ins in a DIFFERENT formulation than the
# oracle (mix() without fma, libm pow, plain dot products). Agreement is therefore to rounding, not to the bit; the bars:
STAGE_TOL = dict(morph=0.0, depth=5e-7, lab=5e-5, depth_b=5e-7, sil=0.0, normal=5e-5, quality=1e-5)


def _assert_stage(name, got, want, tol, max_flips=0):
    """|got - want| <= tol except for at most max_flips elements (discrete decisions on a rounding-sized margin)."""
    assert ((got != got) == (want != want)).all(), f"{name}: NaN pattern differs"
    ok = np.isfinite(got.astype(np.float64)) & np.isfinite(want.astype(np.float64))
    assert ((got == want) | ok | ((got != got) & (want != want))).all(), f"{name}: infinities differ"
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))[ok]
    bad = int((d > tol).sum())
    assert bad <= max_flips, f"{name}: {bad} elements differ by more than {tol} (max {d.max():.3e})"


def _glsl_stagewise(O, G, sc, voxel, inv_res):
    """Each shader stage of the reference against the oracle ON THE SAME INPUTS (the oracle's previous stage)."""
    import dataclasses
    from rrpy import synth
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    L = G.lib()
    N, H, W = sc.depth.shape
    X, Y, Z = sc.cv_res
    bmin, bmax = np.ascontiguousarray(sc.bbox_min, np.float32), np.ascontiguousarray(sc.bbox_max, np.float32)
    bricks = np.zeros(grid["num_bricks"], np.uint32)
    for i in range(N):
        out = np.zeros((H, W), np.float32)
        L.rg_pre_morph(np.ascontiguousarray(sc.depth[i]), W, H, out)
        assert bits_equal(out, pre["morph"][i]).all(), "pre_morph.fs: the hole fill must match bit for bit"
        d2, lab = np.zeros((H, W, 2), np.float32), np.zeros((H, W, 3), np.float32)
        L.rg_pre_depth(pre["morph"][i], W, H, sc.cv_xyz[i], sc.cv_uv[i], X, Y, Z, sc.color[i], sc.CW, sc.CH, bmin, bmax, 0.5, 4.5,
                       1, 0, 0.0, 0.0, 0.0, d2, lab)
        _assert_stage("pre_depth.fs depth", d2, pre["depth"][i], STAGE_TOL["depth"])
        _assert_stage("pre_depth.fs lab", lab, pre["lab"][i], STAGE_TOL["lab"])
        db, sil = np.zeros((H, W, 2), np.float32), np.zeros((H, W), np.float32)
        L.rg_pre_boundary(pre["depth"][i], pre["lab"][i], W, H, 1, db, sil)
        assert bits_equal(sil, pre["sil"][i]).all(), "pre_boundary.fs: silhouettes must be identical"
        assert bits_equal(db, pre["depth_b"][i]).all(), "pre_boundary.fs only selects and flags: identical on identical inputs"
        nrm = np.zeros((H, W, 3), np.float32)
        L.rg_pre_normal(pre["depth_b"][i], W, H, sc.cv_xyz[i], X, Y, Z, bmin, grid["brick_size"], grid["res_bricks"],
                        grid["num_bricks"], bricks, nrm)
        _assert_stage("pre_normal.fs", nrm, pre["normal"][i], STAGE_TOL["normal"])
        q = np.zeros((H, W), np.float32)
        L.rg_pre_quality(pre["depth_b"][i], pre["normal"][i], pre["lab"][i], W, H, sc.cv_xyz[i], X, Y, Z,
                         np.ascontiguousarray(cams[i], np.float32), q)
        _assert_stage("pre_quality.fs", q, pre["quality"][i], STAGE_TOL["quality"])
    assert np.array_equal(bricks, pre["bricks"]), "inc_bricks.glsl mark_brick: brick counters must be bit-exact"
    inv = synth.analytic_inverse(sc, inv_res)
    occ = O.occupied_bricks(pre["bricks"], 10)
    worst = 0.0
    for use_bricks in (True, False):
        want = O.integrate(inv, pre, grid, 0.01, use_bricks, occ)
        got = G.integrate(inv, pre, grid, 0.01, use_bricks, occ)
        _assert_stage("tsdf_integration.vs", got, want, 1e-5 * 0.01)       # BASELINE bar: within 1e-5 of the truncation distance
        ok = np.isfinite(want)
        worst = max(worst, float(np.abs(got[ok].astype(np.float64) - want[ok]).max()))
    return len(occ), worst


def test_oracle_matches_the_reference_shaders_run_on_cpu(O):
    """The pin of the GLSL stages: the reference's shader sources executed on the CPU vs the oracle's restatement."""
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    n_occ, worst = _glsl_stagewise(O, G, synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64)), 0.02, (50, 55, 50))
    assert n_occ > 50
    n_occ, worst2 = _glsl_stagewise(O, G, synth.make_scene(N=3, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48), seed=99), 0.025, (40, 44, 40))
    assert n_occ > 20 and max(worst, worst2) < 1e-7


@pytest.mark.parametrize("flags,depth8", [((False, True, True), False), ((True, False, True), False), ((True, True, False), False),
                                          ((True, False, True), True)])
def test_oracle_matches_the_reference_shaders_flag_variants(O, flags, depth8):
    """filterTextures / useProcessedDepths / refineBoundary off, and the 8-bit sqrt-compressed depth stream (pre_depth.fs
    `uncompress`, NetKinectArray.cpp:345-351): the oracle's chain vs the reference shaders' chain, stage by stage, each stage
    fed the oracle's previous stage."""
    import dataclasses
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=136, cv_res=(24, 24, 48), seed=5)
    compress = None
    if depth8:
        d8 = synth.encode_depth8(sc.depth[0], 0.5, 4.5)
        sc = dataclasses.replace(sc, depth=O.depth8_to_float(d8[None]))
        compress = np.float32([[0.5, 4.5]])
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.04, 0.1)
    cams = [O.frustum(sc.cv_xyz[0])[1]]
    a = O.preprocess(sc, grid, cams, *flags, compress=compress)
    # the shaders' chain from the same raw frame; then every stage again on the oracle's inputs
    b = G.preprocess(sc, grid, cams, *flags, compress=compress)
    assert bits_equal(a["morph"], b["morph"]).all() and np.array_equal(a["bricks"], b["bricks"])
    assert bits_equal(a["sil"], b["sil"]).all()
    for k in ("depth", "lab", "depth_b", "normal", "quality"):
        _assert_stage(k, a[k], b[k], 4 * STAGE_TOL[k])
    assert (a["sil"] > 0).sum() > 200, "the variant must keep a surface"


def test_oracle_integration_matches_the_reference_shader_with_five_sensors(O):
    """`uniform sampler3D[5] cv_xyz_inv`: the reference's sensor limit, running mean over five sensors in order."""
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    sc = synth.make_scene(N=5, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48), seed=21)
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.03, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    inv = synth.analytic_inverse(sc, (40, 44, 40))
    occ = O.occupied_bricks(pre["bricks"], 10)
    want, weight = O.integrate(inv, pre, grid, 0.01, True, occ, want_weight=True)
    got = G.integrate(inv, pre, grid, 0.01, True, occ)
    assert len(occ) > 20 and (weight > 0).sum() > 1000
    _assert_stage("tsdf_integration.vs, 5 sensors", got, want, 1e-5 * 0.01, max_flips=2)


def test_empty_frame_set_oracle_and_reference_shaders(O):
    """No depth returns at all: no silhouette, no brick marks, an empty occupied list, a volume that is -limit everywhere
    (bricks mode only clears), and a raymarch without a single sample - in the oracle and in the reference's shaders."""
    import dataclasses
    import ref_glsl_py as G
    from rrpy import synth
    sc = synth.make_scene(N=2, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48), seed=3)
    sc = dataclasses.replace(sc, depth=np.zeros_like(sc.depth))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.04, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    assert not pre["sil"].any() and not pre["bricks"].any() and not pre["quality"].any() and not pre["normal"].any()
    occ = O.occupied_bricks(pre["bricks"], 10)
    assert len(occ) == 0
    inv = synth.analytic_inverse(sc, (30, 33, 30))
    tsdf = O.integrate(inv, pre, grid, 0.01, True, occ)
    assert (tsdf == np.float32(-0.01)).all()
    mv, pr = synth.look_at((1.6, 1.5, 2.2), (0.0, 1.1, 0.0)), synth.perspective(50.0, 16 / 9, 0.1, 10.0)
    rm = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, 96, 54, 1, skip_space=True)
    assert (rm["depth"] == 1.0).all() and not rm["samples"].any() and not rm["rgba"].any()
    if G.available():
        ref = G.preprocess(sc, grid, cams)
        for k in ("morph", "depth", "lab", "depth_b", "sil", "normal", "quality"):
            _assert_stage(k, pre[k], ref[k], 4 * STAGE_TOL.get(k, 0.0))
        assert not ref["bricks"].any()
        assert bits_equal(G.integrate(inv, ref, grid, 0.01, True, occ), tsdf).all()


def test_oracle_against_reference_shader_goldens(O):
    """Same pin for machines without oracle/_ref: tests/golden/ref_glsl_stages.npz holds what the reference's shaders computed
    (full chain, every stage fed by the shaders' own previous stage). The oracle's own chain must stay within rounding:
    discrete outputs identical, the volume within 2e-5 of the truncation distance (1e-5 per the stagewise test above, plus
    the drift the chained float stages add)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(GOLD), "..", "tools"))
    from rrpy import synth
    g = gold("ref_glsl_stages.npz")
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)    # tools/make_golden.py::glsl_scene
    voxel = float(g["voxel"])
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    assert bits_equal(pre["morph"], g["pre_morph"]).all() and bits_equal(pre["sil"], g["pre_sil"]).all()
    assert np.array_equal(pre["bricks"], g["pre_bricks"])
    for k in ("depth", "lab", "depth_b", "normal", "quality"):
        _assert_stage(k, pre[k], g["pre_" + k], 4 * STAGE_TOL[k])
    occ = O.occupied_bricks(pre["bricks"], 10)
    assert np.array_equal(occ, g["occupied"]) and len(occ) > 10
    for use_bricks, key in ((True, "tsdf_bricks"), (False, "tsdf_dense")):
        got = O.integrate(g["inv"], pre, grid, 0.01, use_bricks, occ)
        assert (np.abs(g[key]) < 0.0099).sum() > 200, "the golden volume must hold in-band voxels"
        _assert_stage(key, got, g[key], 2e-5 * 0.01)


def test_oracle_raymarch_matches_the_reference_shader_run_on_cpu(O, small_scene, small_frame):
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    sc = small_scene
    grid, pre, occ, inv, tsdf = (small_frame[k] for k in ("grid", "pre", "occ", "inv", "tsdf"))
    VW, VH = 160, 90
    for eye in ((1.6, 1.5, 2.2), (0.7, 1.3, 0.75)):                    # outside the volume, and inside it
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        for mode in range(4):
            want = G.raymarch(tsdf, 0.01, inv, sc, pre, mv, pr, VW, VH, mode)
            got = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, VW, VH, mode, skip_space=False)
            assert_raymarch(got, want["rgba"], want["depth"], want["samples"], want["hit"], f"eye {eye} mode {mode}", np.asarray(pr))


def test_oracle_point_renderers_match_the_reference_shaders_run_on_cpu(O, small_scene, small_frame):
    """ReconPoints::draw and ReconCalibs::draw (SURVEY.md 8f-4): the oracle's restatement (oracle/ro_points.cpp) against the
    reference's own points.vs / points.gs / points.fs and calib_vis.vs / calib_vis.fs run on the CPU through the fixed-function
    point pipeline of OpenGL 4.4 (oracle/glsl_host/glsl_harness.cpp), every shade mode, camera outside and inside the volume."""
    import ref_glsl_py as G
    if not G.available() or not hasattr(G.lib(), "rg_draw_points"):
        pytest.skip("oracle/_ref/libref_glsl.so not built with the point shaders (needs the reference tree at build time)")
    from rrpy import synth
    sc = small_scene
    pre, inv, tsdf = (small_frame[k] for k in ("pre", "inv", "tsdf"))
    VW, VH = 200, 112
    for eye in ((1.6, 1.5, 2.2), (0.7, 1.3, 0.75)):
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        for mode in range(4):
            assert_points(O.draw_points(sc, pre, mv, pr, VW, VH, mode), G.draw_points(sc, pre, mv, pr, VW, VH, mode), f"points eye {eye} mode {mode}")
        IZ, IY, IX = inv.shape[1:4]
        for limit in (0.01, 0.005):
            assert_points(O.draw_calibs(tsdf, (IX, IY, IZ), limit, sc.bbox_min, sc.bbox_max, mv, pr, VW, VH),
                          G.draw_calibs(tsdf, inv, sc, 1, limit, mv, pr, VW, VH), f"calibs eye {eye} limit {limit}")


def test_oracle_point_renderers_against_the_committed_shader_outputs(O):
    """The same pin on machines without the reference tree: tests/golden/ref_glsl_points.npz holds what the reference's shaders
    drew for the golden scene (tools/make_golden.py::golden_glsl_points); the oracle regenerates stages and volume bit for bit."""
    from rrpy import synth
    g = gold("ref_glsl_points.npz")
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)    # tools/make_golden.py::glsl_scene
    voxel = float(g["voxel"])
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    inv = synth.analytic_inverse(sc, (20, 22, 20))
    tsdf = O.integrate(inv, pre, grid, 0.01, True, O.occupied_bricks(pre["bricks"], 10))
    assert hashlib.sha256(np.ascontiguousarray(tsdf).tobytes()).hexdigest() == str(g["tsdf_sha"]), "the golden's input volume changed"
    V = dict(eye=(1.2, 1.4, 1.6), at=(0.0, 1.1, 0.0), fovy=50.0, w=160, h=90)                  # make_golden.py::RM_VIEW
    mv, pr = synth.look_at(V["eye"], V["at"]), synth.perspective(V["fovy"], V["w"] / V["h"], 0.1, 10.0)
    for mode in range(4):
        assert_points(O.draw_points(sc, pre, mv, pr, V["w"], V["h"], mode), (g[f"points_rgba{mode}"], g[f"points_depth{mode}"]), f"points mode {mode}")
    assert_points(O.draw_calibs(tsdf, (20, 22, 20), 0.01, sc.bbox_min, sc.bbox_max, mv, pr, V["w"], V["h"]), (g["calibs_rgba"], g["calibs_depth"]), "calibs")


def test_oracle_trigrid_matches_the_reference_shaders_run_on_cpu(O, small_scene, small_frame):
    """ReconTrigrid::draw (SURVEY.md 8f-4): the oracle's restatement (oracle/ro_trigrid.cpp) against the reference's own
    trigrid_accum.vs / .gs / .fs and trigrid_normalize.fs run on the CPU through the same fixed-function stages
    (oracle/ro_raster.h), every shade mode, camera outside and inside the volume."""
    import ref_glsl_py as G
    if not G.available() or not hasattr(G.lib(), "rg_draw_trigrid"):
        pytest.skip("oracle/_ref/libref_glsl.so not built with the trigrid shaders (needs the reference tree at build time)")
    from rrpy import synth
    sc, pre = small_scene, small_frame["pre"]
    VW, VH = 200, 112
    for eye in ((1.6, 1.5, 2.2), (0.2, 1.2, 0.3)):
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        for mode in range(4):
            assert_trigrid(O.draw_trigrid(sc, pre, mv, pr, VW, VH, mode, min_length=0.06), G.draw_trigrid(sc, pre, mv, pr, VW, VH, mode, min_length=0.06),
                           f"trigrid eye {eye} mode {mode}")


def test_oracle_trigrid_against_the_committed_shader_outputs(O):
    """The same pin on machines without the reference tree: tests/golden/ref_glsl_trigrid.npz holds what the reference's shaders
    drew for the golden scene (tools/make_golden.py::golden_glsl_trigrid)."""
    from rrpy import synth
    g = gold("ref_glsl_trigrid.npz")
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)    # tools/make_golden.py::glsl_scene
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, float(g["voxel"]), 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    assert hashlib.sha256(np.ascontiguousarray(pre["quality"]).tobytes()).hexdigest() == str(g["quality_sha"]), "the golden's input maps changed"
    V = dict(eye=(1.2, 1.4, 1.6), at=(0.0, 1.1, 0.0), fovy=50.0, w=160, h=90)                  # make_golden.py::RM_VIEW
    pr = synth.perspective(V["fovy"], V["w"] / V["h"], 0.1, 10.0)
    for tag, eye in (("", V["eye"]), ("in_", tuple(float(x) for x in g["eye_in"]))):
        mv = synth.look_at(eye, V["at"])
        for mode in range(4):
            assert_trigrid(O.draw_trigrid(sc, pre, mv, pr, V["w"], V["h"], mode, min_length=float(g["min_length"])),
                           (g[f"{tag}rgba{mode}"], g[f"{tag}depth{mode}"]), f"trigrid {tag}mode {mode}")


def test_the_rasteriser_partitions_a_shared_edge(O):
    """The fixed-function stages' claim (oracle/ro_raster.h): two triangles that share an edge never both cover a pixel centre and
    never leave one out - checked on the accumulation target: with one sensor, shade mode 3 and a fragment pass that keeps
    everything within epsilon, the summed quality of a pixel is that of ONE fragment, i.e. rgb / alpha is the pure camera colour
    and the alpha equals the interpolated quality, never twice it."""
    from rrpy import synth
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.035, 0.1)
    pre = O.preprocess(sc, grid, [O.frustum(sc.cv_xyz[0])[1]])
    mv, pr = synth.look_at((1.2, 1.4, 1.6), (0.0, 1.1, 0.0)), synth.perspective(50.0, 320 / 180, 0.1, 10.0)
    rgba, depth, accum, depth1 = O.draw_trigrid(sc, pre, mv, pr, 320, 180, 3, min_length=0.06, want_passes=True)
    cov = depth < 1.0
    assert cov.sum() > 500
    # every covered pixel holds the quality of one fragment: bounded by the map's maximum (two fragments would exceed it on
    # the many pixels whose quality is above half of it)
    qmax = float(pre["quality"].max())
    assert accum[..., 3][cov].max() <= qmax * (1 + 1e-6)
    hi = cov & (accum[..., 3] > 0.5 * qmax)
    assert hi.sum() > 20
    # and pass 1 covers exactly what pass 2 covers from the front surface (no seam holes inside the silhouette): a covered pixel's
    # four neighbours are covered unless the pixel is on the silhouette; count isolated single-pixel holes
    pad = np.pad(cov, 1)
    holes = (~cov) & pad[:-2, 1:-1] & pad[2:, 1:-1] & pad[1:-1, :-2] & pad[1:-1, 2:]
    assert holes.sum() <= 2, f"{holes.sum()} one-pixel holes inside the mesh"


def test_depth_peels_from_the_reference_brick_shaders_and_a_rasteriser(O, small_scene, small_frame):
    """drawDepthLimits with the reference's bricks.vs / bricks.gs / bricks.fs and a rasteriser (glsl_harness.cpp::rg_depth_peels;
    the cube strip is read from unit_cube.cpp) against the ray-cast statement ref_glsl_py.depth_peels: same coverage, nearest and
    farthest face depth to rounding; the nearest BACK face differs where bricks.gs dropped faces between occupied bricks, which
    never changes getStartPos' `r >= b` decision."""
    import ref_glsl_py as G
    if not G.available() or G.reference_cube_strip() is None:
        pytest.skip("needs oracle/_ref/libref_glsl.so and the reference tree (unit-cube strip)")
    from rrpy import synth
    sc = small_scene
    grid, pre, occ = (small_frame[k] for k in ("grid", "pre", "occ"))
    VW, VH = 240, 135
    for eye in ((1.6, 1.5, 2.2), (-2.0, 1.0, 1.2), (0.7, 1.3, 0.75)):
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        cast = G.depth_peels(sc, grid, occ, mv, pr, VW, VH, 0.01)
        rast = G.depth_peels_rasterised(sc, grid, pre["bricks"], occ, mv, pr, VW, VH)
        cov = cast[..., 0] < 1.0
        assert np.array_equal(cov, rast[..., 0] < 1.0) and cov.sum() > 1000
        assert np.abs(cast[..., 0] - rast[..., 0]).max() <= 5e-7 and np.abs(cast[..., 1] - rast[..., 1]).max() <= 5e-7
        assert (rast[..., 2] >= cast[..., 2] - 5e-7).all(), "dropping internal faces can only move the nearest back face away"
        assert np.array_equal(cast[..., 0] >= cast[..., 2], rast[..., 0] >= rast[..., 2]), "getStartPos' front-face-culled decision"


def test_oracle_space_skipping_matches_the_reference_shader_on_rasterised_peels(O, small_scene, small_frame):
    """The skipSpace branch of tsdf_raymarch.fs (getStartPos, screenToVol) fed the depth peels drawDepthLimits' rasteriser
    would leave (ref_glsl_py.depth_peels: pixel-centre ray / brick-cube intersections in window space, float64) against the
    oracle's analytic hull: same fragments, surface within 0.1 mm, colours within 2e-3; ceil() of the march length may flip
    the sample count of a few pixels."""
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    sc = small_scene
    grid, pre, occ, inv, tsdf = (small_frame[k] for k in ("grid", "pre", "occ", "inv", "tsdf"))
    VW, VH = 240, 135
    for eye in ((1.6, 1.5, 2.2), (-2.0, 1.0, 1.2), (0.7, 1.3, 0.75)):   # the last one sits inside the volume
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        # the reference's own brick shaders + rasteriser where its cube strip can be read, the ray-cast statement otherwise
        peels = (G.depth_peels_rasterised(sc, grid, pre["bricks"], occ, mv, pr, VW, VH) if G.reference_cube_strip() is not None
                 else G.depth_peels(sc, grid, occ, mv, pr, VW, VH, 0.01))
        want = G.raymarch(tsdf, 0.01, inv, sc, pre, mv, pr, VW, VH, 1, depth_peels=peels)
        got = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, VW, VH, 1, skip_space=True)
        assert_raymarch(got, want["rgba"], want["depth"], want["samples"], want["hit"], f"skipSpace eye {eye}", np.asarray(pr), sample_flips=0.01)


def test_reference_cube_proxy_faces_are_front_facing_outward():
    """ref_glsl_py.depth_peels takes a brick's entry face as gl_FrontFacing and its exit face as back-facing (bricks.fs keeps the
    nearest BACK face in .b). That holds iff the reference's unit-cube triangle strip (unit_cube.cpp:21-30, 53-62) is wound
    counter-clockwise seen from outside; checked on the reference's own numbers where the tree is present."""
    import re
    path = "/root/reference/framework/rendering/unit_cube.cpp"
    if not os.path.exists(path):
        pytest.skip("reference tree not present")
    src = open(path).read()
    verts = re.search(r"std::vector<float> vertices\{(.*?)\};", src, re.S).group(1)
    V = np.array([float(x.rstrip("f")) for x in re.findall(r"[-0-9.]+f", verts)], np.float64).reshape(-1, 3)
    body = src[src.index("void UnitCube::drawInstanced"):]
    idx = [int(x) for x in re.search(r"indices \{(.*?)\};", body, re.S).group(1).replace("\n", " ").split(",")]
    assert V.shape == (8, 3) and len(idx) == 14
    faces = 0
    for i in range(len(idx) - 2):
        a, b, c = (idx[i], idx[i + 1], idx[i + 2]) if i % 2 == 0 else (idx[i + 1], idx[i], idx[i + 2])   # strip winding rule
        n = np.cross(V[b] - V[a], V[c] - V[a])
        assert np.abs(n).sum() > 0, "degenerate strip triangle"
        assert np.dot(n, (V[a] + V[b] + V[c]) / 3.0 - 0.5) > 0, "triangle wound clockwise seen from outside"
        faces += 1
    assert faces == 12


def test_oracle_raymarch_against_reference_shader_golden(O):
    """tests/golden/ref_glsl_raymarch.npz: the reference's raymarch shader on the oracle's volume of the golden scene."""
    from rrpy import synth
    g = gold("ref_glsl_raymarch.npz")
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(24, 24, 48), seed=77)    # tools/make_golden.py::glsl_scene
    voxel = float(g["voxel"])
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    pre = O.preprocess(sc, grid, cams)
    inv = synth.analytic_inverse(sc, (20, 22, 20))
    occ = O.occupied_bricks(pre["bricks"], 10)
    tsdf = O.integrate(inv, pre, grid, 0.01, True, occ)
    assert hashlib.sha256(np.ascontiguousarray(tsdf).tobytes()).hexdigest() == str(g["tsdf_sha"]), "the golden's input volume changed"
    mv, pr = synth.look_at((1.2, 1.4, 1.6), (0.0, 1.1, 0.0)), synth.perspective(50.0, 160 / 90, 0.1, 10.0)   # make_golden.py::RM_VIEW
    for mode in range(4):
        got = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, 160, 90, mode, skip_space=False)
        assert_raymarch(got, g[f"rgba{mode}"], g["depth"], g["samples"], g["hit"], f"golden mode {mode}", np.asarray(pr))
    got = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, 160, 90, 1, skip_space=True)
    assert_raymarch(got, g["skip_rgba"], g["skip_depth"], g["skip_samples"], g["skip_hit"], "golden skipSpace", np.asarray(pr), sample_flips=0.01)


def _assert_colorfill(O, rgba, depth, want_filled, want_atlas_c, want_atlas_d, what):
    got, ac, ad = O.fill_colors(rgba, depth, want_atlas=True)
    assert bits_equal(ac, want_atlas_c).all() and bits_equal(ad, want_atlas_d).all(), f"{what}: the mip atlas (transfer + inpaint passes) must be identical"
    assert (np.isnan(got) == np.isnan(want_filled)).all()
    ok = np.isfinite(got) & np.isfinite(want_filled)
    assert np.abs(got[ok] - want_filled[ok]).max() <= 5e-7, f"{what}: filled colours (two bilinear fetches blended)"
    assert (got != rgba).any(axis=-1).sum() > 50, f"{what}: the fill must change pixels"


def test_oracle_colorfill_matches_the_reference_shaders_run_on_cpu(O, small_scene, small_frame):
    """fillColors: framebuffer_transfer.fs, tsdf_inpaint.fs and tsdf_colorfill.fs of the reference run on the CPU under a harness
    that plays ViewLod / ReconIntegration::fillColors (oracle/glsl_host/glsl_harness.cpp) vs ro_colorfill.cpp."""
    import ref_glsl_py as G
    if not G.available():
        pytest.skip("oracle/_ref/libref_glsl.so not built (needs the reference tree at build time)")
    from rrpy import synth
    sc = small_scene
    grid, pre, occ, inv, tsdf = (small_frame[k] for k in ("grid", "pre", "occ", "inv", "tsdf"))
    for VW, VH in ((320, 180), (161, 97)):                             # odd sizes: truncated lod resolutions
        mv, pr = synth.look_at((1.6, 1.5, 2.2), (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        rm = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, VW, VH, 0, skip_space=True)
        want, ac, ad = G.fill_colors(rm["rgba"], rm["depth"], want_atlas=True)
        _assert_colorfill(O, rm["rgba"], rm["depth"], want, ac, ad, f"{VW}x{VH}")


def test_oracle_colorfill_against_reference_shader_golden(O):
    g = gold("ref_glsl_colorfill.npz")
    _assert_colorfill(O, g["rgba"], g["depth"], g["filled"], g["atlas_color"], g["atlas_depth"], "golden")


def test_space_skipping_hull_agrees_with_the_cube_march(O, small_scene, small_frame):
    """The space-skipping start (analytic ray / occupied-brick hull here, rasterised depth peels in the reference) is the one
    part of the raymarch no reference code pins. It changes the sampling phase, so hits are not identical to the pinned cube
    march; they must agree statistically: > 95 % of the cube march's hits are found, median distance between the two
    surface points < 0.5 mm."""
    from rrpy import synth
    sc = small_scene
    grid, pre, occ, inv, tsdf = (small_frame[k] for k in ("grid", "pre", "occ", "inv", "tsdf"))
    VW, VH = 320, 180
    dims = (sc.bbox_max - sc.bbox_min).astype(np.float64)
    for eye in ((1.6, 1.5, 2.2), (0.7, 1.3, 0.75), (-2.0, 1.0, 1.2)):
        mv, pr = synth.look_at(eye, (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        a = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, VW, VH, 0, skip_space=True)
        b = O.raymarch(tsdf, 0.01, inv, sc, pre, grid, occ, mv, pr, VW, VH, 0, skip_space=False)
        ha, hb = a["depth"] < 1.0, b["depth"] < 1.0
        both = ha & hb
        assert hb.sum() > 1000 and both.sum() >= 0.95 * hb.sum() and (ha & ~hb).sum() <= 0.01 * hb.sum()
        dmm = np.linalg.norm((a["pos"].astype(np.float64) - b["pos"]) * dims, axis=-1)[both] * 1000.0
        assert np.median(dmm) < 0.5


# ------------------------------------------------------------------------------------------------ arithmetic pins

def test_gl_sampling_known_answers(O):
    L = O.lib()
    img = np.arange(12, dtype=np.float32).reshape(3, 4)          # H=3, W=4, value = 4*y + x
    # texel centres reproduce texels exactly; NEAREST picks floor(s*W)
    for y in range(3):
        for x in range(4):
            s, t = (x + 0.5) / 4, (y + 0.5) / 3
            assert L.ro_kat_tex2d(img, 4, 3, s, t, 0) == img[y, x]
            assert L.ro_kat_tex2d(img, 4, 3, s, t, 1) == img[y, x]
    assert L.ro_kat_tex2d(img, 4, 3, 0.5, 0.5, 0) == pytest.approx(5.5)      # midway between four texels
    assert L.ro_kat_tex2d(img, 4, 3, -3.0, -1.0, 0) == 0.0                   # CLAMP_TO_EDGE
    assert L.ro_kat_tex2d(img, 4, 3, 7.0, 9.0, 0) == 11.0
    assert L.ro_kat_tex2d(img, 4, 3, 0.49999, 0.0, 1) == 1.0 and L.ro_kat_tex2d(img, 4, 3, 0.5, 0.0, 1) == 2.0
    vol = np.zeros((2, 2, 2, 4), np.float32)
    vol[1, :, :, 0] = 1.0; vol[:, 1, :, 1] = 1.0; vol[:, :, 1, 2] = 1.0      # channels = z, y, x ramps
    out = np.zeros(4, np.float32)
    L.ro_kat_tex3d(vol, 4, 2, 2, 2, 0.5, 0.25, 0.75, out)
    assert out[2] == pytest.approx(0.5) and out[1] == 0.0 and out[0] == 1.0
    L.ro_kat_tex3d(vol, 4, 2, 2, 2, 0.4, 0.6, 0.5, out)
    np.testing.assert_allclose(out[:3], [0.5, 0.7, 0.3], atol=1e-6)


def test_deterministic_pow_accuracy(O):
    """pow(x,y) = exp2(y*log2 x): a few ulp from libm over the ranges the shaders use; NaN for x < 0 (NVIDIA GL)."""
    L = O.lib()
    xs = np.concatenate([np.linspace(1e-4, 1.0, 400), np.linspace(1.0, 120.0, 200)]).astype(np.float32)
    for y in (2.0, 6.0, 2.4, 1.0 / 3.0, 20.0):
        got = np.array([L.ro_kat_pow(x, np.float32(y)) for x in xs], np.float64)
        want = np.power(xs.astype(np.float64), np.float64(np.float32(y)))
        ok = (want > 1e-30) & (want < 1e30)
        rel = np.abs(got - want)[ok] / want[ok]
        assert ok.sum() > 400 and rel.max() < 1e-5, (y, rel.max())
    assert L.ro_kat_pow(np.float32(0.0), np.float32(6.0)) == 0.0
    assert L.ro_kat_pow(np.float32(1.0), np.float32(20.0)) == 1.0
    assert np.isnan(L.ro_kat_pow(np.float32(-0.5), np.float32(2.0)))
    assert L.ro_kat_exp2(np.float32(10.0)) == 1024.0 and L.ro_kat_log2(np.float32(0.125)) == -3.0


def test_rgb_to_lab_known_answers(O):
    """inc_color.glsl divides by 255 once more than needed, so inputs in [0,1] land near black: L is tiny but monotone."""
    L = O.lib()
    lab = np.zeros(3, np.float32)
    L.ro_kat_rgb_to_lab(np.zeros(3, np.float32), lab)
    assert np.allclose(lab, 0.0, atol=1e-6)
    prev = -1.0
    for v in (0.1, 0.5, 1.0):
        L.ro_kat_rgb_to_lab(np.full(3, v, np.float32), lab)
        assert lab[0] > prev and abs(lab[1]) < 1e-3 and abs(lab[2]) < 1e-3      # grey: a = b = 0
        prev = lab[0]
    # closed form for the linear branch: n/12.92*100, Y/100 <= eps -> L = 903.3*Y/100 ... (kappa branch)
    L.ro_kat_rgb_to_lab(np.ones(3, np.float32), lab)
    Y = (1.0 / 255.0) / 12.92 * 100.0 * (0.2126 + 0.7152 + 0.0722) / 100.0
    assert lab[0] == pytest.approx(116.0 * ((903.3 * Y + 16.0) / 116.0) - 16.0, rel=1e-4)


# ------------------------------------------------------------------------------------------------ shader restatement

@pytest.fixture(scope="module")
def small_frame(O, small_scene):
    from rrpy import synth
    inv = synth.analytic_inverse(small_scene, (50, 55, 50))
    grid = O.brick_grid(small_scene.bbox_min, small_scene.bbox_max, 0.02, 0.1)
    cams = [O.frustum(small_scene.cv_xyz[i])[1] for i in range(small_scene.N)]
    pre = O.preprocess(small_scene, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], 10)
    tsdf = O.integrate(inv, pre, grid, 0.01, True, occ)
    return dict(inv=inv, grid=grid, pre=pre, occ=occ, tsdf=tsdf)


def test_oracle_self_regression_pins(O, small_scene, small_frame):
    from rrpy import synth
    g = gold("oracle_frame_pins.npz")
    pins = dict(zip(g["names"], g["sha256"]))
    f = small_frame
    mv, pr = synth.look_at((1.6, 1.5, 2.2), (0.0, 1.1, 0.0)), synth.perspective(50.0, 16 / 9, 0.1, 10.0)
    rm = O.raymarch(f["tsdf"], 0.01, f["inv"], small_scene, f["pre"], f["grid"], f["occ"], mv, pr, 160, 90, 1, True)
    got = dict(f["pre"])
    got.update(occupied=f["occ"], tsdf=f["tsdf"], rgba=rm["rgba"], depth=rm["depth"], samples=rm["samples"])
    for k, want in pins.items():
        assert hashlib.sha256(np.ascontiguousarray(got[k]).tobytes()).hexdigest() == want, f"oracle output '{k}' changed"
    assert len(f["occ"]) == int(g["n_occupied"]) and int((rm["depth"] < 1).sum()) == int(g["hits"])


def test_oracle_stage_invariants(small_scene, small_frame):
    """Properties the shaders guarantee by construction (SURVEY.md appendix A.0)."""
    pre, sc = small_frame["pre"], small_scene
    raw = sc.depth
    valid_raw = (raw > 0.5) & (raw < 4.5)
    assert np.array_equal(pre["morph"][valid_raw], raw[valid_raw]), "dilate keeps valid pixels"
    assert ((pre["morph"] > 0) & ~valid_raw).sum() > 0, "dilate fills some holes"
    d, db, sil, q, n = pre["depth"], pre["depth_b"], pre["sil"], pre["quality"], pre["normal"]
    assert set(np.unique(sil)) <= {0.0, 1.0}
    assert ((d[..., 1] >= 0) & (d[..., 1] <= 1.0 + 1e-6)).all(), "mean range weight is a fraction of 169 taps"
    assert (sil[db[..., 0] <= 0] == 0).all() and (db[..., 1][sil == 1] == 0).all()
    assert set(np.unique(db[..., 0][db[..., 0] < 0])) <= {-1.0}
    inside = (db[..., 0] > 0) & (db[..., 0] < 1)
    nn = np.linalg.norm(n, axis=-1)
    assert np.allclose(nn[inside & np.isfinite(nn)], 1.0, atol=1e-4) and (nn[~inside] == 0).all()
    assert (q[~inside] == 0).all() and (q[inside & np.isfinite(q)] >= 0).all()
    assert pre["bricks"].sum() >= inside.sum(), "every valid pixel marks its own brick (+ at most one neighbour)"
    assert pre["bricks"].sum() <= 2 * inside.sum()


def test_oracle_integration_invariants(O, small_scene, small_frame):
    f = small_frame
    tsdf, grid = f["tsdf"], f["grid"]
    limit = np.float32(0.01)
    fin = tsdf[np.isfinite(tsdf)]
    assert fin.min() >= -limit and fin.max() <= limit
    # voxels outside every occupied brick keep the cleared value
    mask = np.zeros(tsdf.shape, bool)
    for b in f["occ"]:
        r = grid["ranges"][b]
        mask[r[4]:r[5], r[2]:r[3], r[0]:r[1]] = True
    assert (tsdf[~mask] == -limit).all()
    assert ((tsdf > -limit) & (tsdf < limit)).sum() > 1000
    # dense integration agrees with the brick path inside occupied bricks
    dense = O.integrate(f["inv"], f["pre"], grid, 0.01, False, f["occ"])
    assert bits_equal(dense[mask], tsdf[mask]).all()
    # weight channel: zero where nothing was fused
    t2, w = O.integrate(f["inv"], f["pre"], grid, 0.01, True, f["occ"], want_weight=True)
    assert bits_equal(t2, tsdf).all() and (w >= 0).all() and (w[~mask] == 0).all() and (w > 0).sum() > 1000


def test_planar_wall_gives_linear_ramp(O):
    """Analytic scene (SURVEY.md §4): a wall perpendicular to sensor 0 => along the optical axis the fused TSDF is the
    clamped linear ramp (voxel depth - wall depth) in normalised depth units."""
    from rrpy import synth
    sc = synth.make_scene(N=1, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64), sdf=synth.wall_sdf)
    sc.depth[:] = np.where(sc.depth > 0, 2.0, 0.0).astype(np.float32)       # exact wall, no noise
    inv = synth.analytic_inverse(sc, (50, 55, 50))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.02, 0.1)
    cams = [O.frustum(sc.cv_xyz[0])[1]]
    pre = O.preprocess(sc, grid, cams)
    tsdf = O.integrate(inv, pre, grid, 0.04, False, np.zeros(0, np.uint32))
    s = sc.sensors[0]
    Z, Y, X = tsdf.shape
    zz, yy, xx = np.meshgrid(np.arange(Z), np.arange(Y), np.arange(X), indexing="ij")
    P = sc.bbox_min + (np.stack([xx, yy, zz], -1) + 0.5) / np.array([X, Y, Z]) * (sc.bbox_max - sc.bbox_min)
    depth_m = (P - s.pos) @ s.fwd
    want = (depth_m - 2.0) / 4.0
    band = (np.abs(want) < 0.03) & (tsdf > -0.04) & (tsdf < 0.04)
    assert band.sum() > 2000
    assert np.abs(tsdf[band] - want[band]).max() < 2e-3, "ramp slope/offset (trilinear lookup of an affine field is exact up to the 2 mm distortion)"


def test_colorfill_oracle_properties(O):
    """Stage invariants of the colour hole filling restatement (oracle/ro_colorfill.cpp): only surface pixels change,
    every hole ends up with a blended colour of alpha 1 when valid neighbours exist, the atlas layout follows ViewLod."""
    rng = np.random.default_rng(7)
    H, W = 90, 160
    yy, xx = np.mgrid[0:H, 0:W]
    hit = ((xx - 80) ** 2 + (yy - 45) ** 2) < 38 ** 2
    rgba = np.zeros((H, W, 4), np.float32)
    depth = np.ones((H, W), np.float32)
    rgba[hit, :3] = rng.random((int(hit.sum()), 3), dtype=np.float32)
    holes = hit & (rng.random((H, W)) < 0.25)
    rgba[hit, 3] = 1.0
    rgba[holes, 3] = -1.0
    depth[hit] = (0.5 + 0.3 * rng.random(int(hit.sum()))).astype(np.float32)
    out, atlas_c, atlas_d = O.fill_colors(rgba, depth, want_atlas=True)
    assert O.lib().ro_fill_num_lods(W, H) == 1 + int(np.floor(np.log2(min(W, H))))
    assert atlas_c.shape == (H, int(W * 1.5), 4)
    # lod 0 of the atlas is the raymarch result (cleared where nothing was drawn)
    assert np.array_equal(atlas_c[:, :W][hit], rgba[hit])
    assert np.array_equal(atlas_c[:, :W][~hit], np.broadcast_to(np.float32([0, 1, 0, 0]), (int((~hit).sum()), 4)))
    assert np.array_equal(atlas_d[:, :W][~hit], np.ones(int((~hit).sum()), np.float32))
    # lod 1 sits right of column W in the top rows and holds averaged colours of alpha 1 inside the blob
    lod1 = atlas_c[H - H // 2:, W:W + W // 2]
    assert (lod1[..., 3] == 1.0).sum() > 0.3 * lod1.shape[0] * lod1.shape[1]
    # background untouched, holes filled with alpha-1 blends in the colour range of their neighbours
    assert np.array_equal(out[~hit], rgba[~hit])
    filled = out[holes]
    assert np.isfinite(filled).all() and (filled[:, 3] > 0).mean() > 0.95
    assert filled[:, :3].min() >= 0.0 and filled[:, :3].max() <= 1.0
    # idempotent on an image without holes apart from the texel-fetch rounding of the shader's px / W * W
    clean = rgba.copy()
    clean[holes, 3] = 1.0
    out2 = O.fill_colors(clean, depth)
    assert np.isin(out2[hit].reshape(-1, 4).view(np.uint32), clean.view(np.uint32)).all()


def test_dxt5_decoder_against_reference_squish(O):
    """DXT5 colour ingest (compress_rgb == 5): the oracle's decoder against blocks compressed AND decoded by the reference's
    own codec external/squish (tests/golden/ref_dxt5.npz), including arbitrary block bytes (both endpoint orders: a BC3
    colour block stays in four-colour mode)."""
    g = gold("ref_dxt5.npz")
    H, W = g["image"].shape[:2]
    assert np.array_equal(O.decode_dxt5(g["blocks"], W, H), g["decoded"][..., :3])
    assert np.array_equal(O.decode_dxt5(g["random_blocks"], W, H), g["random_decoded"][..., :3])
    import ref_py as R
    if R.available() and hasattr(R.lib(), "ref_squish_storage_dxt5"):
        assert np.array_equal(R.squish_decompress_dxt5(g["blocks"], W, H), g["decoded"])


def test_dxt1_decoder_against_reference_squish(O):
    """DXT1 colour ingest: the oracle's BC1 decoder against blocks compressed AND decoded by the reference's own codec
    external/squish (tests/golden/ref_dxt1.npz, made by tools/make_golden.py through oracle/_ref), including arbitrary
    block bytes that hit the three-colour (endpoint0 <= endpoint1) mode."""
    g = gold("ref_dxt1.npz")
    H, W, _ = g["image"].shape
    assert np.array_equal(O.decode_dxt1(g["blocks"], W, H), g["decoded"][..., :3])
    assert np.array_equal(O.decode_dxt1(g["random_blocks"], W, H), g["random_decoded"][..., :3])
    assert (g["random_decoded"][..., 3] == 0).sum() > 0            # the fixture does contain three-colour blocks
    import ref_py as R
    if R.available():
        assert np.array_equal(R.squish_decompress_dxt1(g["blocks"], W, H), g["decoded"])
    # 8-bit depth: normalised fixed point, then pre_depth.fs uncompress (through the synthetic sender's inverse)
    from rrpy import synth
    d = np.float32([0.0, 0.6, 1.0, 2.0, 3.9, 4.4])
    f = O.depth8_to_float(synth.encode_depth8(d, 0.5, 4.5))
    assert np.array_equal(f, (synth.encode_depth8(d, 0.5, 4.5).astype(np.float32) / np.float32(255.0)))
