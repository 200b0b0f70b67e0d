#!/usr/bin/env python
"""Times the connected-part labelling (rr_label_parts / rr_download_parts, include/rgbd_recon_b200.h):
  headline         bench.make_inputs() (4 sensors at 512x424, 512^3 R32F), bricks mode: only the voxels of occupied bricks
  headline_dense   the same frame set in dense mode: every voxel of the volume
  c5               8 sensors, 1024^3, half2 voxels, bricks mode
  group            the headline frame set on a group of every visible device (only when more than one is visible): the peer
                   gather of the volume onto member 0, then the labelling there
Per item the median milliseconds per rr_label_parts call over --calls calls after --warmup calls, from CUDA events on the
context's stream around the call; for the headline frame set also rr_download_parts of the labels into pageable host
memory (numpy), pinned host memory and device memory. With --kernels the device time of each kernel per call from a
torch.profiler pass of its own. Prints one JSON line with the device name and power limit read in the same run; --out also
writes it to a file."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT, os.path.join(ROOT, "tools")]

import numpy as np
from bench_cloud import _device, _time

KERNELS = ("k_parts_init", "k_parts_merge", "k_parts_compress", "k_parts_number", "k_parts_relabel", "k_parts_finish",
           "DeviceScanInitKernel", "DeviceScanKernel", "Memset")


def _kernels(call, n=20):
    """Device time per call of each kernel and memset of the labelling (torch.profiler, a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            call()
        torch.cuda.synchronize()
    k = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        key = next((s for s in KERNELS if s in ev.key), None)
        if t > 0 and key:
            k[key] = round(k.get(key, 0.0) + t / 1000.0 / n, 4)
    return k


def _fusion(n_sensors, res, fmt, use_bricks):
    import bench
    from rrpy import capi, synth
    voxel = np.float32(bench.EXTENT / res)
    sc = synth.make_scene(N=n_sensors, W=bench.W, H=bench.H, CW=bench.CW, CH=bench.CH, cv_res=bench.CV_RES, bbox=bench.BBOX, frame=0, seed=1234)
    inv = synth.analytic_inverse(sc, bench.INV_RES)
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
    assert tuple(int(v) for v in fu.volume_res()) == (res, res, res)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    return fu, sc, inv


def _measure(n_sensors, res, fmt, use_bricks, a, downloads=False):
    fu, _, _ = _fusion(n_sensors, res, fmt, use_bricks)
    n = fu.label_parts_count()
    voxels = fu.download_parts(n)[0]
    occ = fu.bricks_count()
    r = dict(sensors=n_sensors, res=res, voxel_format=fmt, bricks=use_bricks, occupied_bricks=occ[0], parts=n,
             inside_voxels=int(voxels.sum()), largest_part=int(voxels.max()) if n else 0,
             label=_time(fu.label_parts_count, fu.stream(), a.calls, a.warmup))
    if downloads:
        import torch
        shape = (res, res, res)
        for kind, buf in (("pageable", np.empty(shape, np.uint32)), ("pinned", torch.empty(shape, dtype=torch.int32, pin_memory=True)),
                          ("device", torch.empty(shape, dtype=torch.int32, device="cuda:0"))):
            ptr = buf.ctypes.data if isinstance(buf, np.ndarray) else buf.data_ptr()
            r["download_labels_" + kind] = _time(lambda: fu._ck(fu.L.rr_download_parts(fu.h, None, None, None, ptr)), fu.stream(), a.calls, a.warmup)
        r["label_bytes"] = res ** 3 * 4
    if a.kernels:
        r["kernel_ms_per_call"] = _kernels(fu.label_parts_count)
    fu.close()
    return r


def _measure_group(devices, a):
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs(n_frames=1)
    sc = scenes[0]
    g = capi.Group(devices, sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    cnt = C.c_uint32()

    def call():
        g._ck(g.L.rr_group_label_parts(g.h, C.byref(cnt)))
    r = dict(devices=devices, label=_time(call, g.member(0).stream(), a.calls, a.warmup), parts=int(cnt.value))
    g.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    from rrpy import capi
    name, power = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    res["headline"] = _measure(4, 512, capi.VOXELS_F32, True, a, downloads=True)
    res["headline_dense"] = _measure(4, 512, capi.VOXELS_F32, False, a)
    res["c5"] = _measure(8, 1024, capi.VOXELS_HALF2, True, a)
    if torch.cuda.device_count() > 1:
        res["group"] = _measure_group(list(range(torch.cuda.device_count())), a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
