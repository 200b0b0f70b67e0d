"""ORACLE (test infrastructure, NOT product code): part tracking between two labellings, restated with numpy and a plain
Python loop, independent of the device algorithm. Import this only from tests/.

pair_overlaps  the distinct (q, p) label pairs of two label volumes and their voxel counts O(q, p) (np.unique);
track          the contract's greedy matching: candidate pairs ordered by O descending, then q, then p (np.lexsort), accepted
               when neither end is taken; new ids for the unmatched tracked parts, ended ids for the unaccepted candidates;
Tracker        a context's tracking state over a sequence of volumes (labels from oracle_parts.label_parts).
"""
from __future__ import annotations

import numpy as np

import oracle_parts

NONE = 0xFFFFFFFF


def pair_overlaps(prev_labels, labels):
    """(q int64 [D], p int64 [D], O int64 [D]) in ascending (q, p): every pair of labels that share a voxel, with the count."""
    a = np.asarray(prev_labels, np.uint32).ravel()
    b = np.asarray(labels, np.uint32).ravel()
    both = (a != NONE) & (b != NONE)
    keys = (a[both].astype(np.uint64) << np.uint64(32)) | b[both].astype(np.uint64)
    k, counts = np.unique(keys, return_counts=True)
    return (k >> np.uint64(32)).astype(np.int64), (k & np.uint64(NONE)).astype(np.int64), counts.astype(np.int64)


def track(prev_labels, prev_ids, labels, voxels, min_voxels, next_id):
    """One rr_track_parts. prev_labels / prev_ids: the tracked labelling and its per-part ids (None: no tracked labelling);
    labels / voxels: the current labelling and its part sizes. Returns (track_ids uint32 [P], prev_parts uint32 [P],
    overlaps uint32 [P], ended uint32 [E], next_id)."""
    voxels = np.asarray(voxels, np.int64)
    P = len(voxels)
    ids = np.full(P, NONE, np.uint32)
    prev = np.full(P, NONE, np.uint32)
    ovl = np.zeros(P, np.uint32)
    tracked = voxels >= min_voxels
    cand = np.zeros(0, bool) if prev_ids is None else np.asarray(prev_ids, np.uint32) != NONE
    taken_q = np.zeros(len(cand), bool)
    if prev_labels is not None and P and len(cand):
        q, p, O = pair_overlaps(prev_labels, labels)
        keep = cand[q] & tracked[p]
        q, p, O = q[keep], p[keep], O[keep]
        for k in np.lexsort((p, q, -O)):             # the last key is the primary one
            if taken_q[q[k]] or prev[p[k]] != NONE:
                continue
            taken_q[q[k]] = True
            prev[p[k]] = q[k]
            ovl[p[k]] = O[k]
            ids[p[k]] = prev_ids[q[k]]
    for k in range(P):
        if tracked[k] and prev[k] == NONE:
            ids[k] = next_id
            next_id += 1
    ended = np.asarray([prev_ids[j] for j in range(len(cand)) if cand[j] and not taken_q[j]], np.uint32)
    return ids, prev, ovl, ended, next_id


class Tracker:
    """The tracking state of a context: feed it the volumes of consecutive rr_track_parts calls."""

    def __init__(self, bbox_min, bbox_max):
        self.bbox_min, self.bbox_max = bbox_min, bbox_max
        self.reset()

    def reset(self):
        self.labels, self.ids, self.next_id = None, None, 0

    def step(self, tsdf, min_voxels):
        """rr_track_parts on tsdf: (labels, voxels, boxes, centroids, track_ids, prev_parts, overlaps, ended)."""
        labels, voxels, boxes, cen = oracle_parts.label_parts(tsdf, self.bbox_min, self.bbox_max)
        ids, prev, ovl, ended, self.next_id = track(self.labels, self.ids, labels, voxels, min_voxels, self.next_id)
        self.labels, self.ids = labels, ids
        return labels, voxels, boxes, cen, ids, prev, ovl, ended
