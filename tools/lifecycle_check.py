"""Device-memory lifecycle of one context and of a 2-member group, through every call that allocates device memory: create,
configure, fuse frames in RGB8 and in DXT5 colour with 8-bit depth, invert a calibration (kept and not kept), raymarch,
colour fill, point and trigrid draws, mesh, parts, simplification, point cloud, queries, reconfigure to another volume size
and to the weight volume, destroy.

Run once under a leak checker to see every allocation freed:
    compute-sanitizer --tool memcheck --leak-check full python tools/lifecycle_check.py --repeats 1
On its own it runs each lifecycle --repeats times and checks that the device's free memory comes back to the level after
the first run (which has loaded the kernels). That catches any leaked buffer of about 2 MB or more per context (frames,
stage images, views, volume); smaller allocations share the driver's 2 MB pages with others and need the leak checker."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rgbd-recon_b200"))
import torch  # noqa: E402

from rrpy import capi, synth  # noqa: E402

INV_RES = (40, 44, 40)
NEAR_FAR = [0.5, 4.5]
VW, VH = 320, 200


def make_inputs():
    sc = synth.make_scene(N=2, W=512, H=424, CW=640, CH=540, cv_res=(32, 32, 64))     # colour: multiples of 4 (DXT)
    frames = [sc, synth.rerender(sc, 3)]
    dxt5 = np.stack([synth.encode_dxt5(sc.color[i], seed=i) for i in range(sc.N)])
    d8 = np.stack([synth.encode_depth8(sc.depth[i], *NEAR_FAR) for i in range(sc.N)])
    mv = synth.look_at((1.4, 1.5, 2.0), (0.0, 1.1, 0.0))
    pr = synth.perspective(50.0, VW / VH, 0.1, 10.0)
    rng = np.random.default_rng(0)
    pts = (rng.uniform(-0.5, 0.5, (4096, 3)) + [0.0, 1.1, 0.0]).astype(np.float32)
    dirs = np.tile(np.float32([[0.0, 0.0, -1.0]]), (4096, 1))
    origins = pts + np.float32([0.0, 0.0, 2.0])
    return dict(sc=sc, frames=frames, inv=synth.analytic_inverse(sc, INV_RES), dxt5=dxt5, d8=d8, mv=mv, pr=pr,
                pts=pts, origins=origins, dirs=dirs)


def context_lifecycle(x, device):
    sc = x["sc"]
    fu = capi.Fusion(sc.N, sc.W, sc.H, sc.CW, sc.CH, device=device)
    fu.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        fu.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
    fu.calib_invert(0, INV_RES, keep=False)                  # a temporary output, downloaded
    for i in range(sc.N):
        fu.calib_invert(i, INV_RES, keep=True, download=False)
    fu.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    for s in x["frames"]:
        fu.upload_frames(s.color, s.depth)
        fu.fuse_frame()
    fu.set_frame_format(dxt5_color=True, depth8=True, near_far=np.float32([NEAR_FAR] * sc.N))
    fu.upload_frames(x["dxt5"], x["d8"])
    fu.frame(True, False, True, sync_bricks=True)
    fu.set_frame_format()
    fu.upload_frames(sc.color, sc.depth)
    fu.fuse_frame()
    fu.download_stage("lab")                                 # a temporary unpadding buffer
    fu.raymarch(x["mv"], x["pr"], VW, VH)
    fu.fill_colors()
    fu.draw_points(x["mv"], x["pr"], VW, VH)
    fu.draw_trigrid(x["mv"], x["pr"], VW, VH)
    nv, nt = fu.extract_mesh_counts()
    fu.download_mesh(nv, nt)
    fu.label_parts()
    fu.mesh_parts(counts=(nv, nt))
    fu.simplify_mesh(2)
    fu.track_parts()
    fu.label_parts()
    fu.track_parts()
    fu.extract_points()
    fu.sample_points(x["pts"])
    fu.cast_rays(x["origins"], x["dirs"])
    fu.configure(limit=0.01, voxel_size=0.025, brick_size=0.1, min_voxels=10, use_bricks=True)         # another volume
    fu.fuse_frame()
    fu.configure(limit=0.01, voxel_size=0.025, brick_size=0.1, min_voxels=10, use_bricks=True, store_weight=True)
    fu.fuse_frame()
    fu.raymarch(x["mv"], x["pr"], VW, VH)
    fu.close()


def group_lifecycle(x, devices):
    sc = x["sc"]
    g = capi.Group(devices, sc.N, sc.W, sc.H, sc.CW, sc.CH)
    g.set_bbox(sc.bbox_min, sc.bbox_max)
    for i in range(sc.N):
        g.calib_upload(i, sc.cv_xyz[i], sc.cv_uv[i])
        g.calib_upload_inv(i, x["inv"][i])
    g.configure(limit=0.01, voxel_size=0.02, brick_size=0.1, min_voxels=10, use_bricks=True)
    for s in x["frames"]:
        g.upload_frames(s.color, s.depth)
        g.fuse_frame()
    g.raymarch(x["mv"], x["pr"], VW, VH)
    g.fill_colors()
    g.extract_mesh()
    g.label_parts()
    g.simplify_mesh(2)
    g.track_parts()
    g.track_parts()
    g.extract_points()
    g.sample_points(x["pts"])
    g.cast_rays(x["origins"], x["dirs"])
    g.close()


def free_bytes(devices):
    for d in devices:
        torch.cuda.synchronize(d)
    return [torch.cuda.mem_get_info(d)[0] for d in devices]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--repeats", type=int, default=4)
    ap.add_argument("--tolerance-mb", type=float, default=2.0)
    args = ap.parse_args()
    x = make_inputs()
    ndev = torch.cuda.device_count()
    devices = sorted({0, 1 % ndev})
    runs = [("context", [0], lambda: context_lifecycle(x, 0)),
            ("group of 2 on devices %s" % [0, 1 % ndev], devices, lambda: group_lifecycle(x, [0, 1 % ndev]))]
    ok = True
    for name, devs, run in runs:
        levels = []
        for _ in range(args.repeats):
            run()
            levels.append(free_bytes(devs))
        drift = [(levels[0][k] - levels[-1][k]) / 2**20 for k in range(len(devs))]
        good = all(d <= args.tolerance_mb for d in drift)
        ok = ok and good
        print(f"{name}: {args.repeats} lifecycles, free MiB after each: "
              f"{[[round(v / 2**20, 1) for v in lv] for lv in levels]}, lost since the first: "
              f"{[round(d, 2) for d in drift]} MiB -> {'ok' if good else 'LEAK'}")
    print("lifecycle check:", "passed" if ok else "FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
