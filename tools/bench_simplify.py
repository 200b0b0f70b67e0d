#!/usr/bin/env python
"""Times rr_simplify_mesh (vertex clustering of the last mesh on the device, include/rgbd_recon_b200.h) on two workloads:
  headline  bench.make_inputs(): 512^3, 4 sensors, bricks mode
  c5        8 sensors, 1024^3, half2 voxels, bricks mode (tools/bench_configs.py's config 5)
with clusters of c = 2, 3 and 4 voxels (--sizes). Per workload: the full mesh's counts and its rr_download_mesh read-back
into pageable and pinned host memory (rr_download_mesh copies to the host only); per c: the simplified counts, the median
milliseconds of rr_simplify_mesh over --calls calls after --warmup calls (CUDA events on the context's stream around the
call, which synchronises once for its counts), and the rr_download_simplified_mesh read-back into pageable, pinned and
device memory; with --kernels the device time of each kernel per call (torch.profiler, a pass of its own). Prints one JSON
line, with the device name and power limit read in the same run; --out also writes it to a file (e.g. under profiles/)."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT, os.path.join(ROOT, "tools")]

import numpy as np

from bench_mesh import _device


def _median_ms(call, stream, calls, warmup):
    """Median, min and max ms of call() between CUDA events on the context's stream (the call synchronises inside)."""
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
    return round(float(np.median(ms)), 4), round(float(np.min(ms)), 4), round(float(np.max(ms)), 4)


def _buffers(kind, shapes, device):
    """Output arrays of one kind of memory (pageable numpy, pinned or device torch) and their pointers."""
    import torch
    out = []
    for shape, dt in shapes:
        if kind == "pageable":
            out.append(np.empty(shape, dt))
        else:
            t = torch.empty(shape, dtype=torch.float32 if dt == np.float32 else torch.int32,
                            device=device if kind == "device" else "cpu")
            out.append(t.pin_memory() if kind == "pinned" else t)
    ptrs = [C.c_void_p(o.ctypes.data if isinstance(o, np.ndarray) else o.data_ptr()) for o in out]
    return out, ptrs


def _kernels(call, calls=10):
    """Device time per call of each kernel and copy (torch.profiler, a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            call()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            key = "k_simp_" + ev.key.split("k_simp_")[1].split("(")[0].split("E")[0] if "k_simp_" in ev.key else ev.key[:48]
            out[key] = round(out.get(key, 0.0) + t / 1000.0 / calls, 4)
    return out


def _workload(bench, capi, scenes, inv, voxel, n_sensors, fmt, a):
    import torch
    sc = scenes[0]
    fu = capi.Fusion(n_sensors, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True, store_weight=fmt)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    nv, nt = fu.extract_mesh_counts()
    dev = torch.device("cuda", fu.device)
    out = dict(res=[int(v) for v in fu.volume_res()], sensors=n_sensors, voxel_format=fmt, vertices=nv, triangles=nt,
               mesh_mb=round((nv * 40 + nt * 12) / 1e6, 2), mesh_download_ms={})
    full = [((nv, 3), np.float32), ((nv, 3), np.float32), ((nv, 4), np.float32), ((nt, 3), np.uint32)]
    for kind in ("pageable", "pinned"):
        bufs, ptrs = _buffers(kind, full, dev)
        ptrs = [C.cast(q, t) for q, t in zip(ptrs, fu.L.rr_download_mesh.argtypes[1:])]
        out["mesh_download_ms"][kind] = _median_ms(lambda: fu._ck(fu.L.rr_download_mesh(fu.h, *ptrs)), fu.stream(), a.calls, a.warmup)[0]
    for c in a.sizes:
        n = {}

        def simplify():
            n["c"] = fu.simplify_mesh_counts(c)
        med, lo, hi = _median_ms(simplify, fu.stream(), a.calls, a.warmup)
        sv, st = n["c"]
        r = dict(vertices=sv, triangles=st, vertex_ratio=round(nv / max(sv, 1), 2), triangle_ratio=round(nt / max(st, 1), 2),
                 mb=round((sv * 40 + st * 16) / 1e6, 2), ms_median=med, ms_min=lo, ms_max=hi, download_ms={})
        simple = [((sv, 3), np.float32), ((sv, 3), np.float32), ((sv, 4), np.float32), ((st, 3), np.uint32), ((st,), np.uint32)]
        for kind in ("pageable", "pinned", "device"):
            bufs, ptrs = _buffers(kind, simple, dev)
            r["download_ms"][kind] = _median_ms(lambda: fu._ck(fu.L.rr_download_simplified_mesh(fu.h, *ptrs)), fu.stream(),
                                                a.calls, a.warmup)[0]
        if a.kernels:
            r["kernel_ms_per_call"] = _kernels(lambda: fu.simplify_mesh_counts(c))
        out[f"c{c}"] = r
    fu.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sizes", default="2,3,4", help="cluster sizes in voxels")
    ap.add_argument("--workloads", default="headline,c5")
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    a.sizes = [int(s) for s in a.sizes.split(",")]
    import bench
    from rrpy import capi
    name, power, _ = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup}
    wl = a.workloads.split(",")
    if "headline" in wl:
        scenes, inv, voxel = bench.make_inputs()
        res["headline"] = _workload(bench, capi, scenes, inv, voxel, bench.N_SENSORS, 0, a)
        del scenes, inv
    if "c5" in wl:
        scenes, inv, voxel = bench.make_inputs(res=1024, n_sensors=8, n_frames=1)
        res["c5"] = _workload(bench, capi, scenes, inv, voxel, 8, capi.VOXELS_HALF2, a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
