#!/usr/bin/env python
"""Times rr_extract_mesh (marching cubes on the device, include/rgbd_recon_b200.h) on three workloads:
  headline  bench.make_inputs(): 512^3, 4 sensors, bricks mode (the occupied-brick shortcut applies)
  dense     the same frame set integrated in dense mode (every cell row is scanned)
  c5        8 sensors, 1024^3, half2 voxels, bricks mode (tools/bench_configs.py's config 5)
Per workload: vertices, triangles, and the median milliseconds per call over --calls calls after --warmup calls, from CUDA
events recorded on the context's stream around rr_extract_mesh (which synchronises once for its count read-back) plus the
rr_download_mesh read-back into pageable numpy arrays, and around rr_extract_mesh alone; with --kernels the device time of
each kernel per call; the same for rr_group_extract_mesh over every visible device (--group). Prints one JSON line,
with the device name and power limit read in the same run; --out also writes it to a file (e.g. under profiles/)."""
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
    return name, power, torch.cuda.device_count()


def _time(extract, download, stream_of, calls, warmup):
    """Median ms of extract() + download() and of extract() alone, CUDA events on the stream of the context that extracts
    (rr_extract_mesh synchronises once inside; the host time of that read-back is part of the interval)."""
    import torch
    for _ in range(warmup):
        download(*extract())
    ms, ms_ex = [], []
    ext = torch.cuda.ExternalStream(stream_of())
    for _ in range(calls):
        b, m, e = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        b.record(ext)
        n = extract()
        m.record(ext)
        download(*n)
        e.record(ext)
        e.synchronize()
        ms.append(b.elapsed_time(e))
        ms_ex.append(b.elapsed_time(m))
    return n, float(np.median(ms)), float(np.min(ms)), float(np.max(ms)), float(np.median(ms_ex))


def _kernels(extract, calls=10):
    """Device time per call of each kernel of the extraction (torch.profiler, a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            extract()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            key = "k_mesh_" + ev.key.split("k_mesh_")[1].split("(")[0].split("E")[0] if "k_mesh_" in ev.key else ev.key[:48]
            out[key] = round(out.get(key, 0.0) + t / 1000.0 / calls, 4)
    return out


def _workload(name, bench, capi, scenes, inv, voxel, n_sensors, use_bricks, fmt, a, ngpu):
    sc = scenes[0]
    out = {}
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    (nv, nt), med, lo, hi, ex = _time(fu.extract_mesh_counts, fu.download_mesh, fu.stream, a.calls, a.warmup)
    out.update(res=[int(v) for v in fu.volume_res()], sensors=n_sensors, bricks=bool(use_bricks), voxel_format=fmt, vertices=nv, triangles=nt,
               ms_median=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4), ms_extract_only=round(ex, 4),
               download_mb=round((nv * 40 + nt * 12) / 1e6, 2))
    if a.kernels:
        out["kernel_ms_per_call"] = _kernels(fu.extract_mesh_counts)
    fu.close()
    if a.group and ngpu > 1:
        g = capi.Group(list(range(ngpu)), n_sensors, bench.W, bench.H, bench.CW, bench.CH)
        g.set_bbox(sc.bbox_min, sc.bbox_max)
        for i in range(n_sensors):
            g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
            g.calib_upload_inv(i, inv[i])
        g.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
        g.upload_frames(sc.color, sc.depth)
        g.fuse_frame()
        m0 = g.member(0)
        (gv, gt), med, lo, hi, ex = _time(g.extract_mesh_counts, m0.download_mesh, m0.stream, a.calls, a.warmup)
        assert (gv, gt) == (nv, nt), f"{name}: the group's mesh has other counts"
        out["group"] = dict(devices=ngpu, ms_median=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4), ms_extract_only=round(ex, 4))
        g.close()
    elif a.group:
        out["group"] = "not measured: one device visible"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--group", action="store_true", help="also time rr_group_extract_mesh over every visible device")
    ap.add_argument("--workloads", default="headline,dense,c5")
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import bench
    from rrpy import capi
    name, power, ngpu = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    wl = a.workloads.split(",")
    if "headline" in wl or "dense" in wl:
        scenes, inv, voxel = bench.make_inputs()
        if "headline" in wl:
            res["headline"] = _workload("headline", bench, capi, scenes, inv, voxel, bench.N_SENSORS, True, 0, a, ngpu)
        if "dense" in wl:
            res["dense"] = _workload("dense", bench, capi, scenes, inv, voxel, bench.N_SENSORS, False, 0, a, ngpu)
        del scenes, inv
    if "c5" in wl:
        scenes, inv, voxel = bench.make_inputs(res=1024, n_sensors=8, n_frames=1)
        res["c5"] = _workload("c5", bench, capi, scenes, inv, voxel, 8, True, capi.VOXELS_HALF2, a, ngpu)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
