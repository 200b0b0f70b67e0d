"""The part-tracking contract on the oracle alone (oracle/oracle_track.py): hand-made volumes with their expected arrays
written out, and the oracle's sequential greedy against an independent matching by rounds of locally dominant pairs on
random blob volumes. The device kernels are held to the oracle by test_track_gpu.py."""
import numpy as np
import oracle_parts
import oracle_track
import pytest

N = oracle_track.NONE
BMIN, BMAX = (-1.0, 0.0, -1.0), (1.0, 2.0, 1.0)


def _vol(*spans, X=16):
    """Blocks [x0, x1) through the whole of a (Z, Y, X) = (2, 2, X) volume: 4 voxels per column, parts ordered by x0."""
    t = np.full((2, 2, X), -1.0, np.float32)
    for x0, x1 in spans:
        t[:, :, x0:x1] = 1.0
    return t


def _run(tracker, vol, min_voxels=1):
    labels, voxels, _, _, ids, prev, ovl, ended = tracker.step(vol, min_voxels)
    return voxels, ids, prev, ovl, ended


def _expect(got, ids, prev, ovl, ended):
    _, g_ids, g_prev, g_ovl, g_ended = got
    assert g_ids.dtype == np.uint32 and g_ended.dtype == np.uint32
    assert g_ids.tolist() == ids, ("track_ids", g_ids.tolist())
    assert g_prev.tolist() == prev, ("prev_parts", g_prev.tolist())
    assert g_ovl.tolist() == ovl, ("overlaps", g_ovl.tolist())
    assert g_ended.tolist() == ended, ("ended", g_ended.tolist())


def _pair(a, b, min_voxels=1):
    t = oracle_track.Tracker(BMIN, BMAX)
    _run(t, a, min_voxels)
    return t, _run(t, b, min_voxels)


def test_first_call_numbers_tracked_parts_in_part_order():
    t = oracle_track.Tracker(BMIN, BMAX)
    _expect(_run(t, _vol((0, 3), (5, 9))), [0, 1], [N, N], [0, 0], [])
    assert t.next_id == 2


def test_identity():
    _, got = _pair(_vol((0, 3), (5, 9)), _vol((0, 3), (5, 9)))
    _expect(got, [0, 1], [0, 1], [12, 16], [])
    assert got[0].tolist() == got[3].tolist()              # overlaps == voxels


def test_one_voxel_shift():
    _, got = _pair(_vol((0, 3), (5, 9)), _vol((1, 4), (6, 10)))
    _expect(got, [0, 1], [0, 1], [8, 12], [])


def test_merge_keeps_the_larger_overlap():
    t, got = _pair(_vol((0, 3), (4, 9)), _vol((0, 9)))
    _expect(got, [1], [1], [20], [0])
    assert t.next_id == 2


def test_split_gives_the_smaller_piece_a_new_id():
    t, got = _pair(_vol((0, 9)), _vol((0, 3), (4, 9)))
    _expect(got, [1, 0], [N, 0], [0, 20], [])
    assert t.next_id == 2


def test_tie_on_overlap_is_broken_by_previous_part():
    _, got = _pair(_vol((0, 2), (4, 6)), _vol((1, 5)))      # the bridge overlaps both by 4
    _expect(got, [0], [0], [4], [1])


def test_tie_on_overlap_and_previous_part_is_broken_by_current_part():
    _, got = _pair(_vol((0, 6)), _vol((0, 2), (4, 6)))      # both pieces overlap part 0 by 8
    _expect(got, [0, 1], [0, N], [8, 0], [])


def test_birth_and_death():
    t, got = _pair(_vol((0, 3), (6, 9)), _vol((0, 3), (12, 15)))
    _expect(got, [0, 2], [0, N], [12, 0], [1])
    assert t.next_id == 3


def test_min_voxels_below_and_at():
    t = oracle_track.Tracker(BMIN, BMAX)
    v = _vol((0, 1), (3, 6))                                # 4 and 12 voxels
    _expect(_run(t, v, 12), [N, 0], [N, N], [0, 0], [])     # 4 < 12: untracked; 12 == 12: tracked
    _expect(_run(t, v, 12), [N, 0], [N, 1], [0, 12], [])    # an untracked part is no candidate
    _expect(_run(t, v, 4), [1, 0], [N, 1], [0, 12], [])     # tracked now, but its previous part was no candidate
    _expect(_run(t, v, 13), [N, N], [N, N], [0, 0], [1, 0])  # nothing tracked: both tracks end, by previous part


def test_empty_previous_and_empty_current():
    t = oracle_track.Tracker(BMIN, BMAX)
    _expect(_run(t, _vol()), [], [], [], [])
    _expect(_run(t, _vol((0, 3))), [0], [N], [0], [])
    _expect(_run(t, _vol()), [], [], [], [0])
    _expect(_run(t, _vol((0, 3))), [1], [N], [0], [])       # ids are not reused
    t.reset()
    _expect(_run(t, _vol((0, 3))), [0], [N], [0], [])       # a reset starts at 0 with no candidates


def test_pair_overlaps_counts_shared_voxels():
    a, _, _, _ = oracle_parts.label_parts(_vol((0, 3), (4, 9)), BMIN, BMAX)
    b, _, _, _ = oracle_parts.label_parts(_vol((2, 6)), BMIN, BMAX)
    q, p, O = oracle_track.pair_overlaps(a, b)
    assert q.tolist() == [0, 1] and p.tolist() == [0, 0] and O.tolist() == [4, 8]


def _locally_dominant(q, p, O, P, prev_ids):
    """Rounds: a pair that comes first in the order (O desc, q asc, p asc) among all remaining pairs sharing its q or its p
    is accepted, and the pairs sharing an end with an accepted pair are removed."""
    rank = lambda k: (-O[k], q[k], p[k])
    alive = set(range(len(q)))
    prev, ovl, ids = np.full(P, N, np.uint32), np.zeros(P, np.uint32), np.full(P, N, np.uint32)
    while alive:
        win = [k for k in alive if all(rank(k) <= rank(j) for j in alive if q[j] == q[k] or p[j] == p[k])]
        assert win
        for k in win:
            prev[p[k]], ovl[p[k]], ids[p[k]] = q[k], O[k], prev_ids[q[k]]
        taken_q, taken_p = {q[k] for k in win}, {p[k] for k in win}
        alive = {j for j in alive if q[j] not in taken_q and p[j] not in taken_p}
    return prev, ovl, ids


def _blobs(shape, centres, radii):
    Z, Y, X = shape
    g = np.stack(np.meshgrid(np.arange(Z), np.arange(Y), np.arange(X), indexing="ij"), -1).astype(np.float32)
    t = np.full(shape, -1.0, np.float32)
    for c, r in zip(centres, radii):
        t = np.maximum(t, r - np.linalg.norm(g - c, axis=-1))
    return t


@pytest.mark.parametrize("seed", range(6))
def test_greedy_equals_locally_dominant_rounds(seed):
    rng = np.random.default_rng(seed)
    shape = (16, 20, 24)
    centres, radii = rng.uniform(0, 1, (30, 3)) * np.array(shape), rng.uniform(1.0, 2.6, 30)
    a = _blobs(shape, centres[:24], radii[:24])
    b = _blobs(shape, np.r_[centres[:20] + rng.normal(0, 1.2, (20, 3)), centres[24:]], np.r_[radii[:20], radii[24:]])   # moved, gone, new
    la, va, _, _ = oracle_parts.label_parts(a, BMIN, BMAX)
    lb, vb, _, _ = oracle_parts.label_parts(b, BMIN, BMAX)
    prev_ids = np.where(rng.uniform(size=len(va)) < 0.8, rng.permutation(len(va)) + 100, N).astype(np.uint32)
    min_voxels = int(rng.integers(1, 8))
    ids, prev, ovl, ended, nxt = oracle_track.track(la, prev_ids, lb, vb, min_voxels, 1000)
    q, p, O = oracle_track.pair_overlaps(la, lb)
    keep = (prev_ids[q] != N) & (vb[p] >= min_voxels)
    q, p, O = q[keep], p[keep], O[keep]
    assert len(q) > 8 and (len(set(q.tolist())) < len(q) or len(set(p.tolist())) < len(p))   # pairs that compete
    w_prev, w_ovl, w_ids = _locally_dominant(q, p, O, len(vb), prev_ids)
    assert np.array_equal(prev, w_prev) and np.array_equal(ovl, w_ovl)
    fresh = (vb >= min_voxels) & (w_prev == N)
    w_ids[fresh] = 1000 + np.arange(fresh.sum())
    assert np.array_equal(ids, w_ids) and nxt == 1000 + fresh.sum()
    accepted = set(w_prev[w_prev != N].tolist())
    assert ended.tolist() == [int(prev_ids[j]) for j in range(len(va)) if prev_ids[j] != N and j not in accepted]
    # every matched part shares voxels with its previous part, and every accepted overlap is exact
    for k in np.flatnonzero(prev != N):
        assert ovl[k] == np.count_nonzero((la == prev[k]) & (lb == k))
