#!/usr/bin/env python
"""Times part removal (rr_remove_parts, include/rgbd_recon_b200.h) next to the frame step, on consecutive frame sets of a
moving scene (bench.make_inputs: the scene turns by 7 degrees per frame set):
  headline         4 sensors at 512x424, 512^3 R32F, bricks mode
  headline_dense   the same frame sets in dense mode
  c5               8 sensors, 1024^3, half2 voxels, bricks mode
Per item, each call right after a fuse of the next frame set, the median milliseconds over --calls frame sets after
--warmup, from CUDA events on the context's stream around the timed calls:
  fuse             rr_fuse_frame (the frame step the removal would follow)
  label_remove     rr_label_parts, then rr_remove_parts of the parts below --min-voxels (floaters)
  remove           rr_remove_parts of the floaters alone, after an untimed rr_label_parts
  keep_only        rr_remove_parts of every part but the largest (keep flags from host memory), after an untimed labelling;
                   on these frame sets every other part is a floater, so this is the floater removal driven by keep flags
  remove_largest   rr_remove_parts of the largest part alone (keep flags from host memory), after an untimed labelling:
                   the case with a large box (the subject's, millions of voxels)
and the part count, the removed parts and voxels of one step, and the voxels of the largest part and of its box. Prints one
JSON line with the device name and power limit read in the same run; --out also writes it to a file."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "oracle")]

import numpy as np
from bench_cloud import _device


def _fuse(fu, s):
    fu.upload_frames(s.color, s.depth)
    fu.fuse_frame()


def _timed(fu, frames, setup, call, calls, warmup):
    """Median / min / max ms of call() after fusing the next frame set and running setup() (untimed)."""
    import torch
    ext = torch.cuda.ExternalStream(fu.stream())
    ms = []
    for i in range(warmup + calls):
        fu.upload_frames(frames[i % len(frames)].color, frames[i % len(frames)].depth)
        arg = setup()
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b.record(ext)
        call(arg)
        e.record(ext)
        e.synchronize()
        if i >= warmup:
            ms.append(b.elapsed_time(e))
    return dict(ms_median=round(float(np.median(ms)), 4), ms_min=round(float(np.min(ms)), 4), ms_max=round(float(np.max(ms)), 4))


def _measure(n_sensors, res, fmt, use_bricks, a):
    import bench
    from rrpy import capi, synth
    voxel = np.float32(bench.EXTENT / res)
    first = synth.make_scene(N=n_sensors, W=bench.W, H=bench.H, CW=bench.CW, CH=bench.CH, cv_res=bench.CV_RES, bbox=bench.BBOX, frame=0, seed=1234)
    frames = [first] + [synth.rerender(first, 7 * t) for t in range(1, 4)]
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, first, synth.analytic_inverse(first, bench.INV_RES))
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
    assert tuple(int(v) for v in fu.volume_res()) == (res, res, res)
    _fuse(fu, frames[0])
    voxels, boxes, _ = fu.label_parts()
    big = int(np.argmax(voxels))
    k, v = fu.remove_parts(a.min_voxels)
    r = dict(sensors=n_sensors, res=res, voxel_format=fmt, bricks=use_bricks, min_voxels=a.min_voxels, parts=int(len(voxels)),
             removed_parts=k, removed_voxels=v, largest_part_voxels=int(voxels[big]),
             largest_box_voxels=int(np.prod((boxes[big, 1::2] - boxes[big, 0::2]).astype(np.int64))))

    def keep_largest(value):
        def setup():
            fu.fuse_frame()
            vox, _, _ = fu.label_parts()
            keep = np.full(len(vox), 1 - value, np.uint8)
            if len(vox):
                keep[int(np.argmax(vox))] = value
            return keep
        return setup

    def label():
        fu.fuse_frame()
        fu.label_parts_count()

    r["fuse"] = _timed(fu, frames, lambda: None, lambda _: fu.fuse_frame(), a.calls, a.warmup)
    r["label_remove"] = _timed(fu, frames, fu.fuse_frame, lambda _: (fu.label_parts_count(), fu.remove_parts(a.min_voxels)), a.calls, a.warmup)
    r["remove"] = _timed(fu, frames, label, lambda _: fu.remove_parts(a.min_voxels), a.calls, a.warmup)
    r["keep_only"] = _timed(fu, frames, keep_largest(1), lambda keep: fu.remove_parts(0, keep), a.calls, a.warmup)
    r["remove_largest"] = _timed(fu, frames, keep_largest(0), lambda keep: fu.remove_parts(0, keep), a.calls, a.warmup)
    fu.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--min-voxels", type=int, default=1000, help="floater threshold: parts of fewer voxels are removed")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from rrpy import capi
    name, power = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    res["headline"] = _measure(4, 512, capi.VOXELS_F32, True, a)
    res["headline_dense"] = _measure(4, 512, capi.VOXELS_F32, False, a)
    res["c5"] = _measure(8, 1024, capi.VOXELS_HALF2, True, a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
