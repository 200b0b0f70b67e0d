"""Every integrator instantiation, the row-width limits of the staged kernel and the API's call orders, against the scalar
oracle bit for bit.

The integrator has four kernels (TMA-staged, fused clear + integrate, k_fill + k_integrate_bricks, dense), three voxel
formats (F32, F32 + weight, half2) and instantiations for 1..8 sensors. rr_integrator_last reports which kernel a call
launched, so every cell asserts the path it asked for as well as the volume: a cell whose path cannot be selected fails.

rr_integrate uses the configuration in effect at the call, the stage images of the last rr_preprocess and the occupied
list of the last rr_bricks_update (empty when rr_configure rebuilt the brick grid since). Settings changes and tunables
between the stages of a frame must honour that; tunables never change results.
"""
import contextlib

import numpy as np
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, LIMIT, BRICK, MIN_VOX = 0.025, (40, 44, 40), 0.01, 0.1, 10
FORMATS = dict(f32=0, f32w=1, half2=2)
# process-wide integrator tunables the tests change, with their defaults (restored after every use)
TUNABLE_DEFAULTS = dict(fused=1, staged=1, stage_cwarps=0, stage_tile=0)


def _half_round(a):
    """The value a half2 voxel holds: binary32 -> nearest-even binary16 -> binary32 (numpy's float16 cast is IEEE RN)."""
    with np.errstate(over="ignore"):
        return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


@contextlib.contextmanager
def tunables(**kw):
    from rrpy import capi
    try:
        for k, v in kw.items():
            capi.set_tunable(k, v)
        yield
    finally:
        for k in kw:
            capi.set_tunable(k, TUNABLE_DEFAULTS[k])


def _oracle_pre(O, sc, grid):
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    return O.preprocess(sc, grid, cams)


def _expect(ts_w, fmt):
    """(tsdf, weight or None) a volume of format `fmt` must hold, from the oracle's fp32 (tsdf, weight)."""
    ts, w = ts_w
    if fmt == "half2":
        return _half_round(ts), _half_round(w)
    return ts, (w if fmt == "f32w" else None)


def _assert_volume(fu, fmt, want, what):
    wt, ww = want
    got = fu.download_tsdf()
    assert bits_equal(got, wt).all(), mismatch_report(f"{what}: tsdf", got, wt)
    if ww is not None:
        gw = fu.download_weight()
        assert bits_equal(gw, ww).all(), mismatch_report(f"{what}: weight", gw, ww)


def _context(d, use_bricks=True, store_weight=0, **cfg):
    from rrpy import capi
    sc = d["scene"]
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, d["inv"])
    fu.configure(limit=cfg.get("limit", LIMIT), voxel_size=d["voxel"], brick_size=BRICK, min_voxels=cfg.get("min_voxels", MIN_VOX),
                 use_bricks=use_bricks, store_weight=store_weight)
    return fu


# ---------------------------------------------------------------------------------------------- instantiation matrix
@pytest.fixture(scope="module")
def matrix():
    """Per sensor count: scene, inverse volumes and the oracle's (tsdf, weight) for bricks and dense, computed once."""
    import oracle_py as O
    from rrpy import synth
    cache = {}

    def get(n):
        if n not in cache:
            sc = synth.make_scene(n, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
            inv = synth.analytic_inverse(sc, INV_RES)
            grid = O.brick_grid(sc.bbox_min, sc.bbox_max, VOXEL, BRICK)
            assert tuple(grid["res"]) == (80, 88, 80)
            pre = _oracle_pre(O, sc, grid)
            occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
            assert len(occ) > 10
            cache[n] = dict(scene=sc, inv=inv, voxel=VOXEL, grid=grid, pre=pre, occ=occ,
                            bricks=O.integrate(inv, pre, grid, LIMIT, True, occ, want_weight=True),
                            dense=O.integrate(inv, pre, grid, LIMIT, False, occ, want_weight=True))
        return cache[n]
    return get


# path -> (use_bricks, tunables, the path rr_integrator_last must report)
PATHS = dict(staged=(True, {}, "staged"), staged11=(True, dict(stage_cwarps=11), "staged"), fused=(True, dict(staged=0), "fused"),
             two_kernel=(True, dict(fused=0), "two_kernel"), dense=(False, {}, "dense"))
CELLS = [pytest.param(n, fmt, path, id=f"N{n}-{fmt}-{path}")
         for n in range(1, 9) for fmt in FORMATS for path in PATHS if not (path == "staged11" and n < 4)]


def _run_cell(d, fmt, path, **extra):
    use_bricks, tun, want_path = PATHS[path]
    fu = _context(d, use_bricks=use_bricks, store_weight=FORMATS[fmt])
    try:
        sc = d["scene"]
        fu.upload_frames(sc.color, sc.depth)
        with tunables(**tun, **extra):
            n_occ, _ = fu.frame(sync_bricks=True)
            last = fu.integrator_last()
            info = fu.integrator_info()
        assert n_occ == len(d["occ"])
        assert last["path"] == want_path, (path, last)
        assert (last["sensors"], last["voxel_mode"], last["repairs"]) == (sc.N, FORMATS[fmt], 0), last
        if want_path == "staged":
            assert info["staged"] == 1 and info["flags"] == 0, info
            assert last["threads"] == (11 if tun.get("stage_cwarps") == 11 else (22 if sc.N <= 4 else 16)), last
        _assert_volume(fu, fmt, _expect(d["bricks" if use_bricks else "dense"], fmt), f"N={sc.N} {fmt} {path}")
        return info
    finally:
        fu.close()


@pytest.mark.parametrize("n,fmt,path", CELLS)
def test_instantiation_matches_oracle(matrix, n, fmt, path):
    _run_cell(matrix(n), fmt, path)


def test_eight_sensor_half2_oversize_footprints(matrix):
    """k_integrate_staged<8, 2, 16> with 8-pixel tiles: most footprints exceed the tile, so the spilling global-memory
    evaluation of that instantiation runs beside the staged one."""
    info = _run_cell(matrix(8), "half2", "staged", stage_tile=8)
    assert info["tile"] == 8 and info["oversize_pairs"] > 0, info


# ------------------------------------------------------------------------------------------------- row-width edge
ROW_WIDTHS = {1020: "staged", 1023: "fused", 1024: "staged", 1028: "fused"}   # X % 4 != 0 or X > 1024: the staged kernel declines


@pytest.fixture(scope="module")
def thin():
    """A 2 m x 0.2 m x 0.24 m slab through the scene: rows of about 1024 voxels at a few hundred thousand voxels a plane."""
    import oracle_py as O
    from rrpy import synth
    sc = synth.make_scene(4, W=256, H=212, CW=160, CH=136, cv_res=(32, 32, 64), bbox=((-1.0, 1.0, -0.12), (1.0, 1.2, 0.12)))
    inv = synth.analytic_inverse(sc, INV_RES)
    cache = {}

    def get(x):
        if x not in cache:
            voxel = 2.0 / x
            grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, BRICK)
            assert grid["res"][0] == x and 100 <= grid["res"][1] <= 106 and 120 <= grid["res"][2] <= 126, grid["res"]
            pre = _oracle_pre(O, sc, grid)
            occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
            assert len(occ) > 10
            cache[x] = dict(scene=sc, inv=inv, voxel=voxel, occ=occ, bricks=O.integrate(inv, pre, grid, LIMIT, True, occ, want_weight=True))
        return cache[x]
    return get


@pytest.mark.parametrize("x", sorted(ROW_WIDTHS))
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_row_width_edge(thin, x, fmt):
    """The staged kernel takes rows up to 1024 voxels that are a multiple of 4 (a row mask of at most 32 words, a row of
    the 4 KB clear buffer). At X = 1024 it sits on both limits; at 1023 and 1028 the fused kernel takes over. Both give the
    oracle's volume."""
    d = thin(x)
    fu = _context(d, store_weight=FORMATS[fmt])
    try:
        assert fu.volume_res()[0] == x
        fu.upload_frames(d["scene"].color, d["scene"].depth)
        n_occ, _ = fu.frame(sync_bricks=True)
        last = fu.integrator_last()
        assert n_occ == len(d["occ"])
        assert last["path"] == ROW_WIDTHS[x], (x, fmt, last)
        if last["path"] == "staged":
            assert fu.integrator_info()["flags"] == 0
        _assert_volume(fu, fmt, _expect(d["bricks"], fmt), f"X={x} {fmt}")
    finally:
        fu.close()


# --------------------------------------------------------------------------------------------------- call orders
MIN_VOX_2 = 40


@pytest.fixture(scope="module")
def orders(matrix):
    """Frame set A (the one integrated) and B (fused first, so stale buffers hold plausible but wrong data) of the
    three-sensor matrix scene, with a cache of oracle volumes keyed by what the integrate call should use."""
    import oracle_py as O
    from rrpy import synth
    d = dict(matrix(3))
    d["other"] = synth.rerender(d["scene"], 9)
    pres = dict(A=d["pre"], B=_oracle_pre(O, d["other"], d["grid"]))
    cache = {}

    def want(fmt, limit=LIMIT, use_bricks=True, min_voxels=MIN_VOX, stages="A", occupancy="A"):
        key = (limit, use_bricks, min_voxels, stages, occupancy)
        if key not in cache:
            occ = O.occupied_bricks(pres[occupancy]["bricks"], min_voxels)
            cache[key] = O.integrate(d["inv"], pres[stages], d["grid"], limit, use_bricks, occ, want_weight=True)
        return _expect(cache[key], fmt)

    d["want"] = want
    assert len(O.occupied_bricks(pres["A"]["bricks"], MIN_VOX_2)) < len(d["occ"])
    assert not bits_equal(want("f32")[0], want("f32", stages="B", occupancy="B")[0]).all()
    return d


def _base_cfg(**kw):
    return dict(dict(limit=LIMIT, min_voxels=MIN_VOX, use_bricks=True, store_weight=0), **kw)


def _configure(fu, d, cfg):
    fu.configure(limit=cfg["limit"], voxel_size=d["voxel"], brick_size=BRICK, min_voxels=cfg["min_voxels"], use_bricks=cfg["use_bricks"],
                 store_weight=cfg["store_weight"])


def _fmt(cfg):
    return {v: k for k, v in FORMATS.items()}[cfg["store_weight"]]


# name -> base configuration / tunables of the context, then the configuration / tunables / action of the mutation
MUTATIONS = dict(
    configure_same=dict(cfg={}),
    limit=dict(cfg=dict(limit=0.015)),
    use_bricks_off=dict(cfg=dict(use_bricks=False)),
    use_bricks_on=dict(base=dict(use_bricks=False), cfg=dict(use_bricks=True)),
    f32_to_half2=dict(cfg=dict(store_weight=2)),
    min_voxels=dict(cfg=dict(min_voxels=MIN_VOX_2)),
    staged_off=dict(tun=dict(staged=0)),
    staged_on=dict(base_tun=dict(staged=0), tun=dict(staged=1)),
    fused_off=dict(tun=dict(fused=0)),
    stage_tile=dict(tun=dict(stage_tile=8)),
    reupload_inverse=dict(act="reupload"),
    integrator_info=dict(act="info"),
    bricks_clear=dict(act="clear"),
)
ORDER_CASES = [pytest.param(m, where, id=f"{m}-after-{where}") for m in MUTATIONS for where in ("preprocess", "update")
               if not (m == "bricks_clear" and where == "preprocess")]


@pytest.mark.parametrize("mutation,where", ORDER_CASES)
def test_mutation_between_stages(orders, mutation, where):
    """bricks_clear -> preprocess -> [mutation] -> bricks_update -> [mutation] -> integrate on a context that has fused
    frame set B before: the volume is the oracle's for the configuration at the integrate call, the stage images of the
    preprocess and the occupied list of the update."""
    from rrpy import capi
    d, m = orders, MUTATIONS[mutation]
    sc = d["scene"]
    base = _base_cfg(**m.get("base", {}))
    after = dict(base, **m.get("cfg", {}))
    base_tun = m.get("base_tun", {})
    with tunables(**base_tun, **{k: TUNABLE_DEFAULTS[k] for k in m.get("tun", {}) if k not in base_tun}):
        fu = _context(d, **base)
        try:
            fu.upload_frames(d["other"].color, d["other"].depth)
            fu.frame()
            fu.upload_frames(sc.color, sc.depth)
            fu.bricks_clear()
            fu.preprocess()

            def mutate():
                if "cfg" in m:
                    _configure(fu, d, after)
                for k, v in m.get("tun", {}).items():
                    capi.set_tunable(k, v)
                if m.get("act") == "reupload":
                    for i in range(sc.N):
                        fu.calib_upload_inv(i, d["inv"][i])
                elif m.get("act") == "info":
                    fu.integrator_info()
                elif m.get("act") == "clear":
                    fu.bricks_clear()

            if where == "preprocess":
                mutate()
            fu.bricks_update()
            if where == "update":
                mutate()
            fu.integrate()
            last = fu.integrator_last()
            want = d["want"](_fmt(after), limit=after["limit"], use_bricks=after["use_bricks"],
                             min_voxels=after["min_voxels"] if where == "preprocess" else base["min_voxels"])
            _assert_volume(fu, _fmt(after), want, f"{mutation} after {where} (integrate ran {last})")
        finally:
            fu.close()


def test_stage_images_of_the_last_preprocess(orders):
    """preprocess A -> bricks_update -> preprocess B -> integrate: B's stage images with A's occupied list."""
    d = orders
    fu = _context(d)
    try:
        fu.upload_frames(d["scene"].color, d["scene"].depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
        fu.upload_frames(d["other"].color, d["other"].depth)
        fu.preprocess()
        fu.integrate()
        _assert_volume(fu, "f32", d["want"]("f32", stages="B", occupancy="A"), f"B's stages, A's bricks ({fu.integrator_last()})")
    finally:
        fu.close()


@pytest.mark.parametrize("use_bricks", [True, False])
def test_setter_then_integrate(orders, use_bricks):
    """kinect_client's shape: a whole frame, then a ReconIntegration setter (setUseBricks) and integrate() alone."""
    d = orders
    fu = _context(d, use_bricks=use_bricks)
    try:
        fu.upload_frames(d["other"].color, d["other"].depth)
        fu.frame()
        fu.upload_frames(d["scene"].color, d["scene"].depth)
        fu.frame()
        _configure(fu, d, _base_cfg(use_bricks=not use_bricks))
        fu.integrate()
        _assert_volume(fu, "f32", d["want"]("f32", use_bricks=not use_bricks), f"use_bricks {use_bricks} -> {not use_bricks}")
    finally:
        fu.close()


def test_integrate_twice(orders):
    d = orders
    fu = _context(d)
    try:
        fu.upload_frames(d["other"].color, d["other"].depth)
        fu.frame()
        fu.upload_frames(d["scene"].color, d["scene"].depth)
        fu.frame()
        first = fu.integrator_last()
        fu.integrate()
        assert fu.integrator_last() == first
        _assert_volume(fu, "f32", d["want"]("f32"), "second integrate")
    finally:
        fu.close()


def test_configure_between_graph_replays(orders):
    """rr_fuse_frame replays a captured graph; every configure drops it, and the next capture must follow the settings."""
    d = orders
    fu = _context(d)
    try:
        fu.upload_frames(d["other"].color, d["other"].depth)
        fu.frame()                                        # builds the z table: the next fuse_frame captures
        fu.upload_frames(d["scene"].color, d["scene"].depth)
        for cfg in (_base_cfg(), _base_cfg(limit=0.015), _base_cfg(use_bricks=False), _base_cfg(store_weight=2), _base_cfg(),
                    _base_cfg(min_voxels=MIN_VOX_2)):
            _configure(fu, d, cfg)
            for rep in range(2):
                fu.fuse_frame()
                _assert_volume(fu, _fmt(cfg), d["want"](_fmt(cfg), limit=cfg["limit"], use_bricks=cfg["use_bricks"], min_voxels=cfg["min_voxels"]),
                               f"fuse_frame {rep} after configure {cfg} ({fu.integrator_last()})")
    finally:
        fu.close()


def test_group_setter_between_update_and_integrate(orders):
    """The ReconIntegration path through a one-device group: a setter between updateOccupiedBricks and integrate."""
    from rrpy import capi
    d = orders
    sc = d["scene"]
    g = capi.Group([0], sc.N, sc.W, sc.H, sc.CW, sc.CH)
    try:
        capi.load_scene(g, sc, d["inv"])
        g.configure(limit=LIMIT, voxel_size=d["voxel"], brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
        g.upload_frames(d["other"].color, d["other"].depth)
        g.frame()
        g.upload_frames(sc.color, sc.depth)
        g.bricks_clear()
        g.preprocess()
        n_occ, _ = g.bricks_update()
        assert n_occ == len(d["occ"])
        g.configure(limit=LIMIT, voxel_size=d["voxel"], brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=True)
        g.integrate()
        got, want = g.download_tsdf(), d["want"]("f32")[0]
        assert bits_equal(got, want).all(), mismatch_report(f"group tsdf ({g.member(0).integrator_last()})", got, want)
    finally:
        g.close()
