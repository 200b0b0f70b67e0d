"""The staged integrator's incremental clear: after every integrate the volume must be bit-identical to what a context
that fuses the same frame set once (a whole-slab clear) holds, whatever ran before it.

The incremental clear only resets the bricks that left the occupied set since the last integrate, so these tests run
long sequences with changing occupancy (including frames with no occupied brick at all) through rr_fuse_frame (graph
replay) and through the separate calls, put every setting change that invalidates the record of what the last integrate
wrote between frames, and check with rr_integrator_last / rr_integrator_cleared that the incremental path is the one
that actually ran.
"""
import contextlib

import numpy as np
import pytest

from conftest import bits_equal, mismatch_report

pytestmark = pytest.mark.gpu

VOXEL, INV_RES, BRICK = 0.025, (40, 44, 40), 0.1
BASE = dict(limit=0.01, voxel_size=VOXEL, brick_size=BRICK, min_voxels=10, use_bricks=True, store_weight=0)


@contextlib.contextmanager
def tunable(name, value, default):
    from rrpy import capi
    try:
        capi.set_tunable(name, value)
        yield
    finally:
        capi.set_tunable(name, default)


@pytest.fixture(scope="module")
def rig():
    """Scene, inverse volumes and four frame sets: three renders of the moving scene and one without any depth."""
    from rrpy import synth
    sc = synth.make_scene(2, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    inv = synth.analytic_inverse(sc, INV_RES)
    empty = synth.rerender(sc, 0)
    empty.depth[...] = 0.0
    frames = dict(a=sc, b=synth.rerender(sc, 3), c=synth.rerender(sc, 6), empty=empty)
    return dict(scene=sc, inv=inv, frames=frames, cache={})


def _context(r, **cfg):
    from rrpy import capi
    sc = r["scene"]
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH)
    capi.load_scene(fu, sc, r["inv"])
    fu.configure(**{**BASE, **cfg})
    return fu


def _volume(fu, cfg):
    t = fu.download_tsdf()
    return t, (fu.download_weight() if cfg.get("store_weight") == 1 else None)


def _fresh(r, name, slab=None, **cfg):
    """The volume a new context holds after fusing frame set `name` once with configuration `cfg`."""
    key = (name, slab, tuple(sorted(cfg.items())))
    if key not in r["cache"]:
        fu = _context(r, **cfg)
        if slab is not None:
            fu.set_slab(*slab)
        f = r["frames"][name]
        fu.upload_frames(f.color, f.depth)
        fu.frame()
        assert fu.integrator_last()["clear"] in ("full", "none"), fu.integrator_last()
        r["cache"][key] = _volume(fu, {**BASE, **cfg})
        fu.close()
    return r["cache"][key]


def _check(fu, r, name, what, slab=None, rows=None, **cfg):
    got = _volume(fu, {**BASE, **cfg})
    want = _fresh(r, name, slab=slab, **cfg)
    for g, w, label in zip(got, want, ("tsdf", "weight")):
        if w is None:
            continue
        if rows is not None:
            g, w = g[rows[0]:rows[1]], w[rows[0]:rows[1]]
        assert bits_equal(g, w).all(), mismatch_report(f"{what}: {label}", g, w)


SEQUENCE = ["a", "b", "a", "empty", "c", "b", "b", "empty", "empty", "a", "c"]


@pytest.mark.parametrize("fmt", [0, 1, 2])
@pytest.mark.parametrize("via", ["fuse_frame", "calls"])
def test_sequence_matches_a_fresh_context(rig, via, fmt):
    r = rig
    fu = _context(r, store_weight=fmt)
    clears, cleared = [], []
    try:
        for i, name in enumerate(SEQUENCE + SEQUENCE[:4]):
            cfg = dict(store_weight=fmt)
            if i >= len(SEQUENCE):
                # a min_voxels change moves occupancy without touching the record of what was written
                cfg["min_voxels"] = 30
                if i == len(SEQUENCE):
                    fu.configure(**{**BASE, **cfg})
            f = r["frames"][name]
            fu.upload_frames(f.color, f.depth)
            if via == "fuse_frame":
                fu.fuse_frame()
            else:
                fu.frame()
            last = fu.integrator_last()
            assert last["path"] == "staged", last
            clears.append(last["clear"])
            cleared.append(fu.integrator_cleared())
            _check(fu, r, name, f"step {i} ({name}, {via}, format {fmt})", **cfg)
    finally:
        fu.close()
    assert clears[0] == "full" and all(c == "incremental" for c in clears[1:]), clears
    # bricks leave the occupied set on the way to the empty frame set, none are left to clear after a repeated one
    assert cleared[SEQUENCE.index("empty")] > 0 and cleared[SEQUENCE.index("empty") + 5] == 0, cleared


def _frame(fu, r, name, via="calls"):
    f = r["frames"][name]
    fu.upload_frames(f.color, f.depth)
    if via == "calls":
        fu.frame()
    else:
        fu.fuse_frame()


# (label, action(fu, r) -> configuration in effect afterwards, whether the next integrate must clear the whole slab)
def _set(**cfg):
    def act(fu, r):
        fu.configure(**{**BASE, **cfg})
        return cfg
    return act


def _reupload_inverse(fu, r):
    for s in range(r["scene"].N):
        fu.calib_upload_inv(s, r["inv"][s])
    return {}


def _slab_there_and_back(fu, r):
    fu.set_slab(10, 50)
    _frame(fu, r, "c")
    fu.set_slab(0, 80)
    return {}


INVALIDATIONS = [
    ("limit", _set(limit=0.02), True),
    ("store_weight 0 -> 1", _set(store_weight=1), True),
    ("store_weight 0 -> half2", _set(store_weight=2), True),
    ("brick size", _set(brick_size=0.15), True),
    ("min_voxels", _set(min_voxels=25), False),
    ("inverse re-upload", _reupload_inverse, False),
    ("set_slab there and back", _slab_there_and_back, True),
]


@pytest.mark.parametrize("via", ["calls", "fuse_frame"])
@pytest.mark.parametrize("label,action,full", INVALIDATIONS, ids=[x[0] for x in INVALIDATIONS])
def test_invalidation_between_frames(rig, label, action, full, via):
    r = rig
    fu = _context(r)
    try:
        for name in ("a", "b", "a"):
            _frame(fu, r, name, via)
        cfg = action(fu, r)
        _frame(fu, r, "c", via)
        assert fu.integrator_last()["clear"] == ("full" if full else "incremental"), (label, fu.integrator_last())
        _check(fu, r, "c", f"after {label}", **cfg)
        for name in ("b", "empty", "a"):
            _frame(fu, r, name, via)
            assert fu.integrator_last()["clear"] == "incremental", (label, name, fu.integrator_last())
            _check(fu, r, name, f"{name} after {label}", **cfg)
    finally:
        fu.close()


def test_store_weight_transitions(rig):
    r = rig
    fu = _context(r)
    try:
        _frame(fu, r, "a")
        for fmt, name in ((1, "b"), (2, "a"), (0, "c"), (2, "b"), (1, "c"), (0, "a")):
            fu.configure(**{**BASE, "store_weight": fmt})
            _frame(fu, r, name)
            assert fu.integrator_last()["clear"] == "full"
            _check(fu, r, name, f"store_weight -> {fmt}", store_weight=fmt)
            _frame(fu, r, "empty")
            assert fu.integrator_last()["clear"] == "incremental"
            _check(fu, r, "empty", f"empty after store_weight -> {fmt}", store_weight=fmt)
    finally:
        fu.close()


def test_other_paths_between_frames(rig):
    """Dense mode and the direct kernels keep no record of what they wrote: the next staged integrate clears everything."""
    r = rig
    fu = _context(r)
    try:
        _frame(fu, r, "a")
        _frame(fu, r, "b")
        fu.configure(**{**BASE, "use_bricks": False})
        _frame(fu, r, "c")
        assert fu.integrator_last()["clear"] == "none"
        fu.configure(**BASE)
        _frame(fu, r, "a")
        assert fu.integrator_last()["clear"] == "full"
        _check(fu, r, "a", "dense -> bricks")
        for knob, value, default in (("staged", 0, 1), ("fused", 0, 1)):
            with tunable(knob, value, default):
                _frame(fu, r, "empty", "fuse_frame")
                assert fu.integrator_last()["path"] != "staged"
                _check(fu, r, "empty", f"{knob}=0")
            _frame(fu, r, "b", "fuse_frame")
            assert fu.integrator_last()["clear"] == "full", knob
            _check(fu, r, "b", f"{knob} back on")
            _frame(fu, r, "c", "fuse_frame")
            assert fu.integrator_last()["clear"] == "incremental", knob
            _check(fu, r, "c", f"{knob} back on, next frame")
    finally:
        fu.close()


def test_call_orders(rig):
    """bricks_clear / a second bricks_update before integrate, and integrate twice, under the incremental clear."""
    r = rig
    fu = _context(r)
    try:
        _frame(fu, r, "a")
        _frame(fu, r, "b")
        # two bricks_update calls before the integrate
        f = r["frames"]["c"]
        fu.upload_frames(f.color, f.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
        fu.bricks_update()
        fu.integrate()
        _check(fu, r, "c", "double bricks_update")
        fu.integrate()
        assert fu.integrator_last()["clear"] == "incremental" and fu.integrator_cleared() == 0
        _check(fu, r, "c", "integrate twice")
        f = r["frames"]["a"]
        fu.upload_frames(f.color, f.depth)
        fu.bricks_clear()
        fu.preprocess()
        fu.bricks_update()
        fu.bricks_clear()            # the counters go, the occupied list and masks of a stay
        fu.integrate()
        _check(fu, r, "a", "bricks_clear before integrate")
    finally:
        fu.close()


def test_graph_replay_takes_the_incremental_path(rig):
    r = rig
    fu = _context(r)
    try:
        for name in ("a", "b"):
            _frame(fu, r, name, "fuse_frame")
        seen = []
        for name in ("a", "b", "a", "b", "empty", "a"):
            _frame(fu, r, name, "fuse_frame")
            seen.append((fu.integrator_last()["clear"], fu.integrator_cleared()))
            _check(fu, r, name, f"replay {name}")
        assert all(c == "incremental" for c, _ in seen), seen
        assert any(n > 0 for _, n in seen), seen
    finally:
        fu.close()


def test_slab_owner_sequence(rig):
    r = rig
    fu = _context(r)
    try:
        fu.set_slab(20, 60)
        for i, name in enumerate(["a", "b", "empty", "c", "a", "b"]):
            _frame(fu, r, name, "fuse_frame" if i % 2 else "calls")
            assert fu.integrator_last()["clear"] == ("full" if i == 0 else "incremental")
            # the rows the owner integrates: its slab and the halo of ceil(limit * Z) + 2 rows on either side
            halo = int(np.ceil(np.float32(BASE["limit"]) * np.float32(80))) + 2
            _check(fu, r, name, f"slab step {i}", slab=(20, 60), rows=(20 - halo, 60 + halo))
    finally:
        fu.close()


def test_two_member_group(rig):
    from rrpy import capi
    r = rig
    sc = r["scene"]
    g = capi.Group([0, 0], sc.N, sc.W, sc.H, sc.CW, sc.CH)
    try:
        capi.load_scene(g, sc, r["inv"])
        g.configure(**BASE)
        bounds = g.slabs()
        for i, name in enumerate(["a", "b", "empty", "c", "a"]):
            f = r["frames"][name]
            g.upload_frames(f.color, f.depth)
            g.fuse_frame() if i % 2 else g.frame()
            want = _fresh(r, name)[0]
            for m in range(2):
                fu = g.member(m)
                z0, z1 = int(bounds[m]), int(bounds[m + 1])
                got = fu.download_tsdf()[z0:z1]
                assert bits_equal(got, want[z0:z1]).all(), mismatch_report(f"group member {m} step {i}", got, want[z0:z1])
    finally:
        g.close()
