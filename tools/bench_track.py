#!/usr/bin/env python
"""Times part tracking (rr_track_parts / rr_download_part_tracks, include/rgbd_recon_b200.h) against the labelling alone
(rr_label_parts) on consecutive frame sets of a moving scene (bench.make_inputs: the scene turns by 7 degrees per frame set):
  headline         4 sensors at 512x424, 512^3 R32F, bricks mode: only the voxels of occupied bricks
  headline_dense   the same frame sets in dense mode: every voxel of the volume
  c5               8 sensors, 1024^3, half2 voxels, bricks mode
Each timed call follows a fuse of the next frame set, so it compares two different labellings. Per item the median
milliseconds of rr_track_parts, of rr_track_parts followed by rr_download_part_tracks into host memory, and of
rr_label_parts, over --calls frame sets after --warmup, from CUDA events on the context's stream around the calls; and the
part count P and the distinct overlap pairs D of one step (the pairs the matching walks, counted on the host from the two
label volumes). With --kernels the device time of each kernel per call from a torch.profiler pass of its own. Prints one
JSON line with the device name and power limit read in the same run; --out also writes it to a file."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "oracle")]

import numpy as np
from bench_cloud import _device

KERNELS = ("k_parts_", "k_track_", "DeviceScan", "DeviceRadixSort", "DeviceSegmentedRadixSort", "DeviceOnesweep",
           "DeviceReduceByKey", "Memset")
MIN_VOXELS = 1000


def _kernels(fu, frames, n=10):
    """Device time per call of each kernel of rr_track_parts (torch.profiler, a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            _fuse(fu, frames[i % len(frames)])
            torch.cuda.synchronize()
            fu.track_parts_counts(MIN_VOXELS)
        torch.cuda.synchronize()
    k = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        key = next((s for s in KERNELS if s in ev.key), None)
        if t > 0 and key:
            name = ev.key if key in ("k_parts_", "k_track_") else key
            k[name[:60]] = round(k.get(name[:60], 0.0) + t / 1000.0 / n, 4)
    return k


def _fuse(fu, s):
    fu.upload_frames(s.color, s.depth)
    fu.fuse_frame()


def _timed(fu, frames, call, calls, warmup):
    """Median / min / max ms of call() right after fusing the next frame set, CUDA events on the context's stream."""
    import torch
    ext = torch.cuda.ExternalStream(fu.stream())
    ms = []
    for i in range(warmup + calls):
        _fuse(fu, frames[i % len(frames)])
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b.record(ext)
        call()
        e.record(ext)
        e.synchronize()
        if i >= warmup:
            ms.append(b.elapsed_time(e))
    return dict(ms_median=round(float(np.median(ms)), 4), ms_min=round(float(np.min(ms)), 4), ms_max=round(float(np.max(ms)), 4))


def _measure(n_sensors, res, fmt, use_bricks, a):
    import bench
    import oracle_track
    from rrpy import capi, synth
    voxel = np.float32(bench.EXTENT / res)
    first = synth.make_scene(N=n_sensors, W=bench.W, H=bench.H, CW=bench.CW, CH=bench.CH, cv_res=bench.CV_RES, bbox=bench.BBOX, frame=0, seed=1234)
    frames = [first] + [synth.rerender(first, 7 * t) for t in range(1, 4)]
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, first, synth.analytic_inverse(first, bench.INV_RES))
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
    assert tuple(int(v) for v in fu.volume_res()) == (res, res, res)
    _fuse(fu, frames[0])
    fu.track_parts_counts(MIN_VOXELS)
    prev = fu.part_labels()
    _fuse(fu, frames[1])
    n, e = fu.track_parts_counts(MIN_VOXELS)
    q, p, O = oracle_track.pair_overlaps(prev, fu.part_labels())
    ids = fu.download_part_tracks(n, e)[0]
    del prev
    r = dict(sensors=n_sensors, res=res, voxel_format=fmt, bricks=use_bricks, min_voxels=MIN_VOXELS, parts=n,
             tracked=int((ids != oracle_track.NONE).sum()), pairs_distinct=int(len(q)), ended=e)
    dl = {}

    def track_and_download():
        n, e = fu.track_parts_counts(MIN_VOXELS)
        dl["out"] = fu.download_part_tracks(n, e)
    r["track"] = _timed(fu, frames, lambda: fu.track_parts_counts(MIN_VOXELS), a.calls, a.warmup)
    r["track_download"] = _timed(fu, frames, track_and_download, a.calls, a.warmup)
    r["label"] = _timed(fu, frames, fu.label_parts_count, a.calls, a.warmup)
    if a.kernels:
        r["kernel_ms_per_call"] = _kernels(fu, frames)
    fu.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
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
