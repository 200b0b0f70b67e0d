#!/usr/bin/env python
"""Times the volume queries (rr_cast_rays / rr_sample_points, include/rgbd_recon_b200.h) on the headline frame set
(bench.make_inputs(): 512^3, 4 sensors, bricks mode with space skipping):
  view_rays        the 921,600 rays of a 1280x720 view (world space, from the eye through each pixel centre, row-major):
                   compare with k_raymarch of the same view, which the kernel pass also times
  random_rays      1,000,000 incoherent rays: origins and directions at random in and around the bbox
  random_points    1,000,000 points at random in the bbox
  surface_points   1,000,000 points on the surface: the extracted mesh's vertices, repeated to 1 M
  single_ray       one ray from host memory: the latency of a pick
Per workload the median milliseconds per call over --calls calls after --warmup calls, from CUDA events on the context's
stream around the call (which copies the inputs in, runs the kernel, copies the results out and synchronises once): with
numpy inputs and outputs (pageable host memory) and with torch CUDA tensors (device-resident). With --kernels the device
time of each kernel per call from a torch.profiler pass of its own. --group: the same over every visible device
(rr_group_*). Prints one JSON line with the device name and power limit read in the same run; --out also writes it to a file."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rgbd-recon_b200"), ROOT]

import numpy as np

VW, VH = 1280, 720
EYE, TARGET = (1.6, 1.5, 2.2), (0.0, 1.1, 0.0)


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


def _view_rays(mv, pr):
    """World rays through the pixel centres of a VW x VH view (GL window coordinates, row 0 = bottom), in double."""
    iM, iP = np.linalg.inv(mv.reshape(4, 4).T.astype(np.float64)), np.linalg.inv(pr.reshape(4, 4).T.astype(np.float64))
    y, x = np.mgrid[0:VH, 0:VW]
    ndc = np.stack([(x + 0.5) / VW * 2 - 1, (y + 0.5) / VH * 2 - 1, np.ones_like(x, float), np.ones_like(x, float)], -1).reshape(-1, 4)
    w = ndc @ (iM @ iP).T
    far = w[:, :3] / w[:, 3:]
    o = iM[:3, 3] / iM[3, 3]
    return np.broadcast_to(o, far.shape).astype(np.float32), (far - o).astype(np.float32)


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


def _kernels(calls_by_name, n=10):
    """Device time per call of each kernel (torch.profiler, a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, call in calls_by_name.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                call()
            torch.cuda.synchronize()
        k = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            key = next((s for s in ("k_cast_rays", "k_sample_points", "k_query_rays_composite", "k_query_points_composite", "k_raymarch")
                        if s in ev.key), None)
            if t > 0 and key:
                k[key] = round(k.get(key, 0.0) + t / 1000.0 / n, 4)
        out[name] = k
    return out


def _inputs(fu_like, sc, mesh_vertices, mv, pr):
    rng = np.random.default_rng(7)
    lo, hi = np.asarray(sc.bbox_min, np.float32), np.asarray(sc.bbox_max, np.float32)
    n = 1_000_000
    vo, vd = _view_rays(mv, pr)
    ro = (lo - 0.2 + rng.random((n, 3)).astype(np.float32) * (hi - lo + 0.4)).astype(np.float32)
    rd = rng.normal(size=(n, 3)).astype(np.float32)
    rp = (lo + rng.random((n, 3)).astype(np.float32) * (hi - lo)).astype(np.float32)
    sp = np.resize(mesh_vertices, (n, 3)).astype(np.float32)
    return dict(view_rays=(vo, vd), random_rays=(ro, rd), random_points=(rp,), surface_points=(sp,), single_ray=(vo[VW * VH // 2 + VW // 2:][:1], vd[VW * VH // 2 + VW // 2:][:1]))


def _measure(q, stream, inputs, a, device):
    import torch
    out = {}
    for name, args in inputs.items():
        fn = q.cast_rays if len(args) == 2 else q.sample_points
        r = dict(entries=int(len(args[0])), host=_time(lambda: fn(*args), stream, a.calls, a.warmup))
        if name != "single_ray":
            dargs = tuple(torch.from_numpy(np.ascontiguousarray(x)).to(device) for x in args)
            r["device"] = _time(lambda: fn(*dargs), stream, a.calls, a.warmup)
        if len(args) == 2:
            r["hits"] = int((fn(*args)[3] != 0xFFFFFFFF).sum())
        out[name] = r
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--group", action="store_true", help="also time rr_group_cast_rays / rr_group_sample_points over every visible device")
    ap.add_argument("--kernels", action="store_true", help="also the device time of each kernel (torch.profiler, separate pass)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    import bench
    from rrpy import capi, synth
    name, power, ngpu = _device()
    res = {"device": name, "power_limit_w": power, "calls": a.calls, "warmup": a.warmup, "view": [VW, VH]}
    scenes, inv, voxel = bench.make_inputs(n_frames=1)
    sc = scenes[0]
    mv, pr = synth.look_at(EYE, TARGET), synth.perspective(50.0, VW / VH, 0.1, 10.0)
    fu = capi.Fusion(bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
    capi.load_scene(fu, sc, inv)
    fu.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    inputs = _inputs(fu, sc, fu.extract_mesh()[0], mv, pr)
    dev = torch.device("cuda", 0)
    res["single_context"] = _measure(fu, fu.stream(), inputs, a, dev)
    res["single_context"]["raymarch_view"] = _time(lambda: fu.raymarch(mv, pr, VW, VH, shade_mode=0, download=False) or fu.synchronize(),
                                                   fu.stream(), a.calls, a.warmup)
    if a.kernels:
        res["kernel_ms_per_call"] = _kernels({
            "view_rays": lambda: fu.cast_rays(*inputs["view_rays"]),
            "random_rays": lambda: fu.cast_rays(*inputs["random_rays"]),
            "random_points": lambda: fu.sample_points(*inputs["random_points"]),
            "surface_points": lambda: fu.sample_points(*inputs["surface_points"]),
            "raymarch_view": lambda: fu.raymarch(mv, pr, VW, VH, shade_mode=0, download=False)})
    fu.close()
    if a.group and ngpu > 1:
        g = capi.Group(list(range(ngpu)), bench.N_SENSORS, bench.W, bench.H, bench.CW, bench.CH)
        g.set_bbox(sc.bbox_min, sc.bbox_max)
        for i in range(bench.N_SENSORS):
            g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
            g.calib_upload_inv(i, inv[i])
        g.configure(limit=bench.LIMIT, voxel_size=voxel, brick_size=bench.BRICK, min_voxels=bench.MIN_VOX, use_bricks=True)
        g.upload_frames(sc.color, sc.depth)
        g.fuse_frame()
        res["group"] = dict(devices=ngpu, **_measure(g, g.member(0).stream(), inputs, a, dev))
        g.close()
    elif a.group:
        res["group"] = "not measured: one device visible"
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
