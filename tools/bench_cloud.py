#!/usr/bin/env python
"""Times the point-cloud export (rr_extract_points / rr_download_points, include/rgbd_recon_b200.h) on the headline frame set
(bench.make_inputs(): 4 sensors at 512x424, colour 1280x1080) and on the same scene with 8 sensors:
  extract          rr_extract_points over every sensor: flag pass, scan, count read-back (the call's one synchronisation),
                   write pass
  download_*       rr_download_points of the whole cloud into preallocated buffers: pageable host memory (numpy), pinned host
                   memory (torch pin_memory) and device memory of the context's GPU (torch CUDA tensors)
Per item the median milliseconds per call over --calls calls after --warmup calls, from CUDA events on the context's stream
around the call. With --kernels the device time of each kernel per extraction from a torch.profiler pass of its own. Prints
one JSON line with the device name and power limit read in the same run; --out also writes it to a file."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT]

import numpy as np


def _device():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(q.splitlines()[0])
    except Exception:
        power = None
    return name, power


def _time(call, stream, calls, warmup):
    import torch
    for _ in range(warmup):
        call()
    ext = torch.cuda.ExternalStream(stream)
    ms = []
    for _ in range(calls):
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b.record(ext)
        call()
        e.record(ext)
        e.synchronize()
        ms.append(b.elapsed_time(e))
    return dict(ms_median=round(float(np.median(ms)), 4), ms_min=round(float(np.min(ms)), 4), ms_max=round(float(np.max(ms)), 4))


def _kernels(call, n=20):
    """Device time per call of each kernel of the extraction (torch.profiler, a pass of its own)."""
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
        key = next((s for s in ("k_cloud_flags", "k_cloud_write", "DeviceScanInitKernel", "DeviceScanKernel") if s in ev.key), None)
        if t > 0 and key:
            k[key] = round(k.get(key, 0.0) + t / 1000.0 / n, 4)
    return k


def _buffers(n, kind):
    import torch
    shapes = (((n, 3), torch.float32), ((n, 3), torch.float32), ((n, 3), torch.float32), ((n,), torch.float32), ((n,), torch.uint32))
    if kind == "pageable":
        return [np.empty(s, np.uint32 if d == torch.uint32 else np.float32) for s, d in shapes]
    if kind == "pinned":
        return [torch.empty(s, dtype=d, pin_memory=True) for s, d in shapes]
    return [torch.empty(s, dtype=d, device="cuda:0") for s, d in shapes]


def _ptr(b):
    return b.ctypes.data if isinstance(b, np.ndarray) else b.data_ptr()


def _measure(n_sensors, a):
    import bench
    from rrpy import capi
    scenes, inv, voxel = bench.make_inputs(n_sensors=n_sensors, n_frames=1)
    sc = scenes[0]
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    n = fu.extract_points_count()
    r = dict(sensors=n_sensors, depth=[bench.W, bench.H], pixels=n_sensors * bench.W * bench.H, points=n,
             bytes=n * 44, extract=_time(fu.extract_points_count, fu.stream(), a.calls, a.warmup))
    for kind in ("pageable", "pinned", "device"):
        bufs = _buffers(n, kind)
        ptrs = [_ptr(b) for b in bufs]
        r["download_" + kind] = _time(lambda: fu._ck(fu.L.rr_download_points(fu.h, *ptrs)), fu.stream(), a.calls, a.warmup)
    if a.kernels:
        r["kernel_ms_per_call"] = _kernels(fu.extract_points_count)
    fu.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    name, power = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    res["headline"] = _measure(4, a)
    res["sensors_8"] = _measure(8, a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
