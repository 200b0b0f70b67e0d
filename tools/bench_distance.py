#!/usr/bin/env python
"""Times the distance field and distance queries (rr_distance_field / rr_download_distance_field / rr_sample_distance,
include/rgbd_recon_b200.h) on the bench's frame sets (bench.make_inputs):
  headline         4 sensors at 512x424, 512^3 R32F, bricks mode: pass x reads only the voxels of occupied bricks
  headline_dense   the same frame set in dense mode: pass x reads every voxel
  c5               8 sensors, 1024^3, half2 voxels, bricks mode
Per item the median / min / max milliseconds over --calls calls after --warmup, from CUDA events on the context's stream
around the calls, of rr_distance_field; of the nearest read-back (4 bytes per voxel) into pageable, pinned and device
memory; and of rr_sample_distance on 1 M random points over the bbox and 1 M mesh vertices, from host (pageable) and from
device arrays. The achieved rate of rr_distance_field is the bytes the three passes need (field_bytes: pass x writes the
field and reads the voxels of the occupied bricks, overlaps counted twice, or every voxel in dense mode; passes y and z read and write it once each) over its median time. With
--group, the same field and queries through a group of every visible device (skipped with one device). With --kernels
the device time of each kernel per call from a torch.profiler pass of its own. Prints one JSON line with the device name
and power limit read in the same run; --out also writes it to a file."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "oracle")]

import numpy as np
from bench_cloud import _device

KERNELS = ("k_dist_", "k_sample_distance", "Memset", "Memcpy")
N_POINTS = 1 << 20


def _timed(stream, call, calls, warmup):
    """Median / min / max ms of call(), CUDA events on the given stream."""
    import torch
    ext = torch.cuda.ExternalStream(stream)
    ms = []
    for i in range(warmup + calls):
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b.record(ext)
        call()
        e.record(ext)
        e.synchronize()
        if i >= warmup:
            ms.append(b.elapsed_time(e))
    return dict(ms_median=round(float(np.median(ms)), 4), ms_min=round(float(np.min(ms)), 4), ms_max=round(float(np.max(ms)), 4))


def _kernels(fu, pts, n=10):
    """Device time per call of each kernel and copy of rr_distance_field and rr_sample_distance (torch.profiler)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fu.distance_field()
            fu.sample_distance(pts)
        torch.cuda.synchronize()
    k = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0 and any(s in ev.key for s in KERNELS):
            k[ev.key[:60]] = round(k.get(ev.key[:60], 0.0) + t / 1000.0 / n, 4)
    return k


def _points(sc, fu):
    rng = np.random.default_rng(7)
    rand = rng.uniform(sc.bbox_min, sc.bbox_max, (N_POINTS, 3)).astype(np.float32)
    pos = fu.extract_mesh()[0]
    surf = pos[rng.integers(0, len(pos), N_POINTS)].astype(np.float32)
    return rand, surf


def _queries(fu, stream, rand, surf, a):
    import torch
    r = {}
    for name, pts in (("random", rand), ("surface", surf)):
        dev = torch.from_numpy(pts).cuda(fu.device if hasattr(fu, "device") else 0)
        r[f"sample_{name}_host"] = _timed(stream, lambda: fu.sample_distance(pts), a.calls, a.warmup)
        r[f"sample_{name}_device"] = _timed(stream, lambda: fu.sample_distance(dev), a.calls, a.warmup)
    return r


def _measure(n_sensors, res, fmt, use_bricks, a):
    import bench
    import torch
    from rrpy import capi, synth
    voxel = np.float32(bench.EXTENT / res)
    sc = synth.make_scene(N=n_sensors, W=bench.W, H=bench.H, CW=bench.CW, CH=bench.CH, cv_res=bench.CV_RES, bbox=bench.BBOX, frame=0, seed=1234)
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, synth.analytic_inverse(sc, bench.INV_RES))
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=use_bricks, store_weight=fmt)
    assert tuple(int(v) for v in fu.volume_res()) == (res, res, res)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    fu.fuse_frame()
    n_inside = fu.distance_field()
    nvox = res ** 3
    # pass x reads the candidate voxels (bricks: those of occupied bricks, counted from the brick ranges) and writes the
    # field; passes y and z read and write it once each
    if use_bricks:
        _, occupied = fu.download_bricks()
        rng = fu.brick_ranges()[np.asarray(occupied, np.int64)]
        read_x = int(np.prod((rng[:, 1::2] - rng[:, 0::2]).astype(np.int64), axis=1).sum()) * 4
    else:
        read_x = nvox * 4
    field_bytes = read_x + nvox * 4 * 5
    stream = fu.stream()
    r = dict(sensors=n_sensors, res=res, voxel_format=fmt, bricks=use_bricks, inside_voxels=n_inside, field_bytes=field_bytes)
    r["distance_field"] = _timed(stream, fu.distance_field, a.calls, a.warmup)
    r["distance_field"]["achieved_gb_s"] = round(field_bytes / (r["distance_field"]["ms_median"] * 1e6), 1)
    host = np.empty((res, res, res), np.uint32)
    pinned = torch.empty((res, res, res), dtype=torch.int32).pin_memory()
    device = torch.empty((res, res, res), dtype=torch.int32, device=f"cuda:{fu.device}")
    for name, buf in (("pageable", host.ctypes.data), ("pinned", pinned.data_ptr()), ("device", device.data_ptr())):
        r[f"download_{name}"] = _timed(stream, lambda: fu._ck(fu.L.rr_download_distance_field(fu.h, buf)), a.calls, a.warmup)
    del host, pinned, device
    rand, surf = _points(sc, fu)
    fu.distance_field()
    r.update(_queries(fu, stream, rand, surf, a))
    if a.kernels:
        r["kernel_ms_per_call"] = _kernels(fu, rand)
    fu.close()
    return r


def _group(a):
    import bench
    import torch
    from rrpy import capi
    n = torch.cuda.device_count()
    if n < 2:
        return None
    scenes, inv, voxel = bench.make_inputs(n_frames=1)
    sc = scenes[0]
    g = capi.Group(list(range(n)), bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, inv[i])
    g.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    g.upload_frames(sc.color, sc.depth)
    g.fuse_frame()
    m0 = g.member(0)
    r = dict(devices=n, distance_field=_timed(m0.stream(), g.distance_field, a.calls, a.warmup))
    rand = np.random.default_rng(7).uniform(sc.bbox_min, sc.bbox_max, (N_POINTS, 3)).astype(np.float32)
    r["sample_random_host"] = _timed(m0.stream(), lambda: g.sample_distance(rand), a.calls, a.warmup)
    g.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--group", action="store_true", help="also through a group of every visible device")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from rrpy import capi
    name, power = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    res["headline"] = _measure(4, 512, capi.VOXELS_F32, True, a)
    res["headline_dense"] = _measure(4, 512, capi.VOXELS_F32, False, a)
    res["c5"] = _measure(8, 1024, capi.VOXELS_HALF2, True, a)
    if a.group:
        res["group"] = _group(a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
