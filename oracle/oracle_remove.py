"""ORACLE (test infrastructure, NOT product code): removing connected parts from the fused volume (rr_remove_parts), restated
with numpy on the labels of oracle_parts (scipy.ndimage.label). Import this only from tests/.

removed_flags  which parts go: voxels[p] < min_voxels, or keep given and keep[p] == 0;
cleared_voxel  the voxel the bricks-mode clear writes, as the stored 4 bytes and as the (tsdf, weight) pair the downloads give;
remove_parts   the volume (and weight volume) after the removal, with the counts the call returns.
"""
from __future__ import annotations

import numpy as np

import oracle_parts

VOXELS_F32, VOXELS_F32_WEIGHT, VOXELS_HALF2 = 0, 1, 2


def removed_flags(voxels, min_voxels=0, keep=None):
    voxels = np.asarray(voxels, np.uint32)
    flags = voxels < np.uint32(min_voxels)
    if keep is not None:
        keep = np.asarray(keep).reshape(-1)
        assert keep.shape == voxels.shape, "keep needs one entry per part"
        flags |= keep == 0
    return flags


def cleared_voxel(store_weight, limit):
    """(stored uint32 bits, tsdf float32, weight float32) of the cleared voxel: -limit (R32F; F32_WEIGHT with weight 0 in its
    own volume), or __floats2half2_rn(-limit, 0) for half2 voxels (tsdf in the low half), widened as the downloads widen."""
    neg = np.float32(-np.float32(limit))
    if store_weight == VOXELS_HALF2:
        h = np.array([neg], np.float16)
        return np.uint32(h.view(np.uint16)[0]), np.float32(h[0]), np.float32(0)
    return neg.view(np.uint32), neg, np.float32(0)


def remove_parts(tsdf, limit, store_weight=VOXELS_F32, min_voxels=0, keep=None, weight=None, labels=None, voxels=None):
    """tsdf float32 [Z][Y][X] as rr_download_tsdf gives it; weight float32 [Z][Y][X] as rr_download_weight gives it (F32_WEIGHT,
    or the high half of half2 voxels), or None. labels / voxels: the labelling the call acts on (default oracle_parts.label_parts
    of tsdf). Returns (tsdf, weight, removed_parts, removed_voxels); the inputs are not modified."""
    t = np.array(tsdf, np.float32, copy=True)
    if labels is None:
        labels, voxels, _, _ = oracle_parts.label_parts(t, (0, 0, 0), (1, 1, 1))
    flags = removed_flags(voxels, min_voxels, keep)
    lab = np.asarray(labels, np.uint32)
    inside = lab != oracle_parts.OUTSIDE
    gone = np.zeros(lab.shape, bool)
    gone[inside] = flags[lab[inside]]
    _, tv, wv = cleared_voxel(store_weight, limit)
    t[gone] = tv
    w = None
    if weight is not None:
        w = np.array(weight, np.float32, copy=True)
        w[gone] = wv
    return t, w, int(flags.sum()), int(np.asarray(voxels, np.uint64)[flags].sum())
