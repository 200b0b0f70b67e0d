#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native volumetric-fusion path.

Metric (BASELINE.json): 4-sensor TSDF Gvoxel-updates/s (+ fused frames/s) at 512^3.
A "step" is one fused frame set: clearOccupiedBricks -> processTextures (5 passes) -> updateOccupiedBricks ->
integrate, i.e. kinect_client.cpp:572-600 after NetKinectArray::update. `value` is measured with the frame set
already resident in HBM; `e2e` runs the same step through the C ABI from pinned HOST buffers (H2D of the colour and
depth frames inside the timed region, D2H of the occupied-brick count the reference reads back every frame).

  python bench.py --gpus N --steps K --warmup W          # our arm (torchrun launches N ranks for N > 1)
  python bench.py --impl reference ...                   # the reference's algorithm on the host cores (oracle port)

Beside the headline the line carries sub-records measured in the same run: `dense` (setUseBricks(false)), `config5`
(BASELINE.json configs[4]: 8 sensors, 1024^3 half2 voxels, the same slab code at every N), the view path, and for N > 1
`verified` (every rank's slab and the composited view compared bit for bit with a single-context run on rank 0)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

_RESULT_FD = None      # the process' real stdout once main() has pointed fd 1 at stderr (see emit)


def emit(record):
    """The ONE JSON line of the contract. Libraries print to the C-level stdout on their own (NCCL's version banner on the first
    collective), so main() points fd 1 at stderr for the whole run and the result line alone goes to the real stdout."""
    line = json.dumps(record) + "\n"
    if _RESULT_FD is None:
        sys.stdout.write(line); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line.encode())

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "rgbd-recon_b200"))

R = 512                       # TSDF resolution (R^3)
N_SENSORS = 4
W, H, CW, CH = 512, 424, 1280, 1080
CV_RES = (128, 128, 256)      # forward calibration volumes
INV_RES = (128, 128, 256)     # inverse calibration volumes (4,194,304 voxels each, SURVEY.md §8d)
EXTENT = 2.048
BBOX = ((-EXTENT / 2, 1.1 - EXTENT / 2, -EXTENT / 2), (EXTENT / 2, 1.1 + EXTENT / 2, EXTENT / 2))
LIMIT, BRICK, MIN_VOX = 0.01, 0.1, 10
N_FRAMES = 2                  # distinct synthetic frame sets cycled through the steps
VW, VH = 1280, 720            # view of the raymarch sub-record
# one description of the workload for both arms (the driver compares the strings)
WORKLOAD = (f"4 Kinect-v2 sensors 512x424 depth + 1280x1080 RGB8, {R}^3 R32F TSDF ({EXTENT} m cube), inverse calibration volumes "
            f"128x128x256, step = clear bricks + 5 pre-process passes + brick update + integrate")
INTEGRATION = {True: "occupied bricks (reference default m_use_bricks=true)", False: "dense (every voxel x every sensor)"}


def host_cores():
    """Host threads this process may use. torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, so the OpenMP
    default is not the box's core count there: the CPU arms set their thread count from the affinity mask instead."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(bricks):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload
    (profiles/integrate_traffic.json, written by tools/ncu_summary.py --traffic); None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "integrate_traffic.json")
    if not os.path.exists(p):
        return None, None
    t = json.load(open(p)).get("bricks" if bricks else "dense")
    if not t:
        return None, None
    return int(t["dram_bytes_read"] + t["dram_bytes_write"]), t.get("source")


def make_inputs(res=R, n_sensors=N_SENSORS, n_frames=N_FRAMES):
    from rrpy import synth
    voxel = EXTENT / res
    scenes = [synth.make_scene(N=n_sensors, W=W, H=H, CW=CW, CH=CH, cv_res=CV_RES, bbox=BBOX, frame=0, seed=1234)]
    scenes += [synth.rerender(scenes[0], 7 * t) for t in range(1, n_frames)]
    inv = synth.analytic_inverse(scenes[0], INV_RES)
    return scenes, inv, np.float32(voxel)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=100):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(int(period_ms)),
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(res, n_occ_vox, covered_inv_vox, nbricks, bricks, n_sensors=N_SENSORS, slab_frac=1.0):
    """SURVEY.md §8(d): bytes one integrate launch must move. Bricked: 4·XYZ (clear) + 4·V_occ (overwrite) +
    16·covered·N (inverse volumes where occupied bricks cover them) + 16·P·N (depth_b 8 + quality 4 + silhouette 4 per
    pixel) + 4·#bricks. Dense: 4·XYZ + 16·V_inv·N + 16·P·N."""
    P = W * H
    vinv = INV_RES[0] * INV_RES[1] * INV_RES[2]
    if not bricks:
        return int(4 * res ** 3 * slab_frac + 16 * vinv * n_sensors * slab_frac + 16 * P * n_sensors)
    return int(4 * res ** 3 * slab_frac + 4 * n_occ_vox + 16 * covered_inv_vox * n_sensors + 16 * P * n_sensors + 4 * nbricks)


class Rig:
    """One rank of one configuration: a context, its frame sets (pinned host + device), the slab, the broadcast
    pipeline for N > 1, and the timed loops."""

    def __init__(self, torch, dist, rank, world, local, scenes, inv, voxel, n_sensors, res, bricks, fmt):
        from rrpy import capi, multigpu
        self.torch, self.dist, self.rank, self.world, self.local = torch, dist, rank, world, local
        self.capi, self.multigpu = capi, multigpu
        self.res, self.bricks, self.n_sensors = res, bricks, n_sensors
        self.dev = torch.device("cuda", local)
        fu = self.fu = capi.Fusion(n_sensors, W, H, CW, CH, device=local)
        capi.load_scene(fu, scenes[0], inv)
        fu.configure(limit=LIMIT, voxel_size=voxel, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=bricks, store_weight=fmt)
        assert tuple(int(v) for v in fu.volume_res()) == (res, res, res), fu.volume_res()
        # z-slab of this rank (SURVEY.md §8e): contiguous slices, remainder spread over the first ranks
        self.z0, self.z1 = multigpu.slab_range(rank, world, res)
        self.slab_how = "single volume"
        self.slabs = [(0, res)]
        if world > 1 and bricks:
            # slab boundaries balanced on the brick occupancy of one pre-processed frame set (every rank computes the same
            # counters, so every rank derives the same boundaries): equal-thickness slabs leave the outer ranks idle
            fu.upload_frames(scenes[0].color, scenes[0].depth)
            fu.bricks_clear(); fu.preprocess(); fu.bricks_update(sync=True)
            _, occ0 = fu.download_bricks()
            # cost of an occupied voxel against a cleared one: 45 at four sensors (DESIGN.md §5), proportional to the sensor count
            self.slabs = multigpu.balanced_slabs(world, res, res * res, fu.brick_ranges(), occ0, compute_to_fill=45.0 * n_sensors / 4.0,
                                                      halo_slices=multigpu.halo(LIMIT, res))
            self.z0, self.z1 = self.slabs[rank]
            self.slab_how = f"z-slabs balanced on occupied-brick cost: {self.slabs}"
        elif world > 1:
            self.slabs = [multigpu.slab_range(r, world, res) for r in range(world)]
            self.slab_how = "equal z-slabs"
        fu.set_slab(self.z0, self.z1)
        halo = multigpu.halo(LIMIT, res) if world > 1 else 0
        self.zc0, self.zc1 = max(0, self.z0 - halo), min(res, self.z1 + halo)     # slices this rank actually writes (slab + halo)
        self.stream = torch.cuda.ExternalStream(fu.stream(), device=self.dev)
        # frame sets: pinned host copies (e2e) and device copies (value)
        self.h_color = [torch.from_numpy(s.color).pin_memory() for s in scenes]
        self.h_depth = [torch.from_numpy(s.depth).pin_memory() for s in scenes]
        self.d_color = [t.to(self.dev) for t in self.h_color]
        self.d_depth = [t.to(self.dev) for t in self.h_depth]
        self.cb, self.db = self.h_color[0].numel(), self.h_depth[0].numel() * 4
        self.h_src_c, self.h_src_d, self.h_src_cb, self.h_src_db = self.h_color, self.h_depth, self.cb, self.db
        self.nf = len(scenes)
        self.flags = (True, True, True)      # filterTextures, useProcessedDepths, refineBoundary (8-bit depth streams: no pre_morph)
        # N > 1: one packed broadcast per frame set, double-buffered (the broadcast of set i+1 overlaps the fusion of set i)
        self.fb = multigpu.FrameBroadcaster(dist, self.dev, self.cb, self.db, src=0) if world > 1 else None
        if world > 1 and rank == 0:
            # the ingest rank holds every frame set packed like a server message (colour bytes then depth bytes)
            self.d_packed = [torch.cat([c.reshape(-1), d.reshape(-1).view(torch.uint8)]) for c, d in zip(self.d_color, self.d_depth)]
            self.h_packed = [torch.cat([c.reshape(-1), d.reshape(-1).view(torch.uint8)]).pin_memory() for c, d in zip(self.h_color, self.h_depth)]
        else:
            self.d_packed = self.h_packed = [None] * self.nf

    def consume_broadcast(self):
        packed, slot = self.fb.consume(self.stream)
        self.fu.upload_frames_ptr(packed.data_ptr(), self.cb, packed.data_ptr() + self.cb, self.db, device=True)   # into the current frame slot, on the compute stream
        self.fb.release(slot, self.stream)

    def step_device(self, i):
        k = i % self.nf
        fu, fb = self.fu, self.fb
        if self.world > 1:
            # each frame set arrives on rank 0 and is broadcast over NVLink (NCCL) before every GPU pre-processes it
            if fb.in_flight() == 0:
                fb.issue(packed=self.d_packed[k])                         # pipeline prologue (first step only)
            self.consume_broadcast()
            # the next set's broadcast is enqueued BEFORE this set's kernels: NCCL's CTAs then share the SMs with the small
            # pre-processing kernels instead of queueing behind the persistent integrate kernel, which fills every SM
            fb.issue(packed=self.d_packed[(i + 1) % self.nf])
            fu.fuse_frame()
        else:
            fu.upload_frames_ptr(self.d_color[k].data_ptr(), self.cb, self.d_depth[k].data_ptr(), self.db, device=True)
            fu.fuse_frame()                  # one call; a captured CUDA graph while stage timing is off, direct launches otherwise

    def step_host(self, i):
        """The reference's ingest is double-buffered (reader thread fills the back PBO while the front one is drawn,
        double_pixel_buffer.cpp): frame set i was staged during step i-1; this step swaps it in, starts the host->device
        copy of frame set i+1 on the copy stream, and runs the fused frame on set i: one rr_fuse_frame (a CUDA-graph launch)
        plus rr_bricks_count, the 4-byte device->host read of the occupied-brick count the reference does every frame.
        Every step issues one host->device copy of a whole frame set, all inside the timed region."""
        k, k1 = i % self.nf, (i + 1) % self.nf
        fu, fb = self.fu, self.fb
        if self.world > 1:
            # rank 0 copies the pinned host frame set into the broadcast slot (its host->device copy), then one broadcast
            if fb.in_flight() == 0:
                fb.issue(packed=self.h_packed[k])
            self.consume_broadcast()
            fb.issue(packed=self.h_packed[k1])                            # next set's host->device copy + broadcast run beside this set's kernels
            fu.fuse_frame(*self.flags)
            return fu.bricks_count()
        fu.swap_frames()
        fu.stage_frames_ptr(self.h_src_c[k1].data_ptr(), self.h_src_cb, self.h_src_d[k1].data_ptr(), self.h_src_db)
        fu.fuse_frame(*self.flags)
        return fu.bricks_count()

    def barrier(self):
        if self.fb is not None:
            while self.fb.in_flight():                     # drain the pipeline: every rank consumes what every rank issued
                self.consume_broadcast()
        self.fu.synchronize()
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()

    def timed(self, step, steps, warmup, with_stage_timers=False, finish=None):
        torch, fu = self.torch, self.fu
        for i in range(warmup):
            step(i)
        self.barrier()
        fu.set_timing(1 if with_stage_timers else 0)
        fu.stage_stats("2integrate"); fu.stage_stats("1preprocess")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = fu.launch_count()
        e0.record(self.stream)
        h0 = time.perf_counter()
        for i in range(steps):
            step(warmup + i)
        self.host_ms = (time.perf_counter() - h0) * 1e3 / steps      # host time to ENQUEUE one step (diagnostic)
        if finish:
            finish()
        e1.record(self.stream)
        self.barrier()
        self.launches = fu.launch_count() - l0
        ms = e0.elapsed_time(e1)
        fu.set_timing(0)
        return self.max_over_ranks(ms)

    def max_over_ranks(self, v):
        if self.world > 1:
            t = self.torch.tensor([v], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)

    def occupancy(self):
        """Occupied bricks of the last frame and the voxels of them this rank evaluates (slab + halo)."""
        n_occ, ratio = self.fu.bricks_update(sync=True)
        counters, occ = self.fu.download_bricks()
        rr = self.fu.brick_ranges()[occ]
        vox = int(((rr[:, 1] - rr[:, 0]) * (rr[:, 3] - rr[:, 2]) *
                   (np.clip(rr[:, 5], self.zc0, self.zc1) - np.clip(rr[:, 4], self.zc0, self.zc1)).clip(0)).sum()) if len(occ) else 0
        return int(n_occ), float(ratio), vox, len(counters)

    def roofline(self, int_avg_ms, n_occ_vox, nbricks):
        slab_frac = (self.zc1 - self.zc0) / self.res
        covered = int(INV_RES[0] * INV_RES[1] * INV_RES[2] * min(1.0, n_occ_vox / max(1, self.res ** 3 * slab_frac)) * slab_frac)
        abytes = algorithmic_bytes(self.res, n_occ_vox, covered, nbricks, self.bricks, self.n_sensors, slab_frac)
        achieved = abytes / (int_avg_ms / 1e3) / 1e9 if int_avg_ms > 0 else 0.0
        peak, peak_src = peaks()
        return abytes, achieved, peak, peak_src

    def close(self):
        self.fu.close()


def integrate_kernel_name(bricks, info):
    if not bricks:
        return "k_integrate_dense"
    if info.get("staged"):
        return ("k_integrate_staged (clear + occupied-brick integration, TMA-staged operands, one launch = the 2integrate stage; "
                f"tile {info['tile']} px, z-chunk {info['zchunk']}, {info['smem_bytes']} B smem)")
    return "k_integrate_fused (clear + occupied-brick integration, direct gathers)"


def sub_record(torch, dist, rank, world, local, what, n_sensors, res, bricks, fmt, steps, scenes=None, inv=None, voxel=None, view=False):
    """A secondary configuration through the same code path: frames device-resident (broadcast from rank 0 for N > 1),
    one rr_fuse_frame per step, CUDA events over `steps` steps after 5 warm-up steps, stage timers in a second pass."""
    if scenes is None:
        scenes, inv, voxel = make_inputs(res, n_sensors, 1)
    rig = Rig(torch, dist, rank, world, local, scenes, inv, voxel, n_sensors, res, bricks, fmt)
    ms = rig.timed(rig.step_device, steps, 5) / steps
    rig.timed(rig.step_device, max(10, steps // 2), 3, with_stage_timers=True)
    int_ms, int_n = rig.fu.stage_stats("2integrate")
    pre_ms, pre_n = rig.fu.stage_stats("1preprocess")
    int_avg = int_ms / max(1, int_n)
    int_slowest = rig.max_over_ranks(int_avg)          # the slab that gates the step (stage timers are per rank)
    n_occ, ratio, vox, nbricks = rig.occupancy()
    abytes, achieved, peak, _ = rig.roofline(int_avg, vox, nbricks)
    info = rig.fu.integrator_info()
    out = {"what": what, "value": round(res ** 3 / ms / 1e6, 3), "unit": "Gvoxel-updates/s", "frames_per_s": round(1e3 / ms, 2),
           "ms_per_step": round(ms, 5), "steps": steps,
           "stages_ms": {"1preprocess": round(pre_ms / max(1, pre_n), 5), "2integrate": round(int_avg, 5),
                         **({"2integrate_slowest_rank": round(int_slowest, 5)} if world > 1 else {})},
           "roofline": {"achieved": round(achieved, 1), "frac": round(achieved / peak, 4), "algorithmic_bytes_per_launch": int(abytes),
                        "kernel": integrate_kernel_name(bricks, info)},
           "occupied_bricks": n_occ, "slabs": rig.slab_how if world > 1 else None}
    if view and world == 1:
        from rrpy import synth
        mv, pr = synth.look_at((1.7, 1.6, 2.3), (0.0, 1.1, 0.0)), synth.perspective(50.0, VW / VH, 0.1, 10.0)
        for _ in range(3):
            rig.fu.raymarch(mv, pr, VW, VH, shade_mode=1, download=False); rig.fu.fill_colors(download=False)
        rig.fu.synchronize()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record(rig.stream)
        for _ in range(10):
            rig.fu.raymarch(mv, pr, VW, VH, shade_mode=1, download=False); rig.fu.fill_colors(download=False)
        v1.record(rig.stream)
        rig.fu.synchronize()
        out["view_ms"] = round(v0.elapsed_time(v1) / 10, 4)
        out["view"] = f"raymarch {VW}x{VH} (shaded, brick space skipping) + colour hole filling"
    rig.close()
    return out


def invert_record(torch):
    """BASELINE.json configs[0]: CalibrationInverter on one synthetic 128x128x256 cv_xyz -> inverse volume at ceil(bbox / 0.007 m)
    (exact 8-NN + inverse-distance weighting + frustum cull, k_invert). GPU time per volume from the context's stage timer;
    parity of this size against the oracle port is tests/test_calib_invert_gpu.py, the CPU timing tools/bench_invert.py."""
    from rrpy import capi, synth
    sc = synth.make_scene(N=1, W=W, H=H, CW=CW, CH=CH, cv_res=CV_RES)
    res = tuple(int(np.ceil((sc.bbox_max[i] - sc.bbox_min[i]) / np.float32(0.007))) for i in range(3))
    fu = capi.Fusion(1, W, H, CW, CH)
    capi.load_scene(fu, sc)
    fu.set_timing(2)
    times = []
    for _ in range(4):
        fu.calib_invert(0, res, download=False)
        times.append(fu.stage_ms("calib_invert"))
    fu.close()
    ms = float(np.median(times[1:]))
    nvox = res[0] * res[1] * res[2]
    return {"what": "BASELINE.json configs[0]: calib_inverter, one 128x128x256 calibration volume -> inverse volume (exact 8-NN + IDW + frustum cull)",
            "out_res": list(res), "ms_per_volume": round(ms, 3), "mvoxel_per_s": round(nvox / ms / 1e3, 1)}


def verify_against_single_context(torch, dist, rig, scenes, inv, voxel, bricks, mv, pr, view_once):
    """Run once, untimed: every rank fuses frame set 0 into its slab and hashes the slices it owns; rank 0 also fuses the whole
    volume on a second, unsharded context and hashes the same slice ranges, marches the same view there, and compares the
    composited image of the sharded run with it bit for bit. True only if every slab and the view agree."""
    from rrpy import capi
    fu, dev, rank, world = rig.fu, rig.dev, rig.rank, rig.world
    fu.upload_frames(scenes[0].color, scenes[0].depth)
    fu.frame()
    mine = fu.download_tsdf()[rig.z0:rig.z1]
    digest = np.frombuffer(hashlib.sha256(mine.tobytes()).digest(), np.uint8).copy()
    all_digests = [torch.empty(32, dtype=torch.uint8, device=dev) for _ in range(world)]
    dist.all_gather(all_digests, torch.from_numpy(digest).to(dev))
    composited = view_once(download=True)
    rig.barrier()
    ok = True
    if rank == 0:
        rgba_s, depth_s = composited
        ref = capi.Fusion(N_SENSORS, W, H, CW, CH, device=rig.local)
        capi.load_scene(ref, scenes[0], inv)
        ref.configure(limit=LIMIT, voxel_size=voxel, brick_size=BRICK, min_voxels=MIN_VOX, use_bricks=bricks)
        ref.upload_frames(scenes[0].color, scenes[0].depth)
        ref.frame()
        full = ref.download_tsdf()
        for r, (z0, z1) in enumerate(rig.slabs):
            want = hashlib.sha256(full[z0:z1].tobytes()).digest()
            ok = ok and bytes(all_digests[r].cpu().numpy().tobytes()) == want
        rgba_r, depth_r = ref.raymarch(mv, pr, VW, VH, shade_mode=1)
        ok = ok and np.array_equal(rgba_s.view(np.uint32), rgba_r.view(np.uint32)) and np.array_equal(depth_s.view(np.uint32), depth_r.view(np.uint32))
        ref.close()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, 0)
    return bool(flag.item())


DUMP_DRAWS = 1 << 21           # seeded voxel draws of --dump-outputs over the whole volume (about 2.1 M distinct voxels, 25 MB with their indices)


def dump_outputs(out_dir, fu):
    """--dump-outputs: what the last timed step left for a caller of rr_fuse_frame, as float32 / float64 .npy files, about 55 MB.
    The TSDF (537 MB at 512^3) is written in two parts. `tsdf_occupied_bricks` is every voxel the integration wrote: the
    occupied bricks in `occupied_bricks` order, each brick as tsdf[z0:z1, y0:y1, x0:x1] flattened (ranges from
    rr_get_brick_ranges). `tsdf_sample` is a fixed, seeded sample of the whole volume, cleared space included, and
    `tsdf_sample_index` holds the sample's flat indices (z*Y*X + y*X + x). `brick_counters` and `occupied_bricks` are whole."""
    os.makedirs(out_dir, exist_ok=True)
    tsdf = fu.download_tsdf()
    idx = np.unique(np.random.default_rng(2024).integers(0, tsdf.size, DUMP_DRAWS))
    counters, occupied = fu.download_bricks()
    rr = fu.brick_ranges()[occupied]
    in_bricks = np.concatenate([tsdf[z0:z1, y0:y1, x0:x1].reshape(-1) for x0, x1, y0, y1, z0, z1 in rr] or [np.zeros(0, np.float32)])
    for name, a in (("tsdf_occupied_bricks", in_bricks), ("tsdf_sample", tsdf.reshape(-1)[idx]), ("tsdf_sample_index", idx.astype(np.float64)),
                    ("brick_counters", counters.astype(np.float64)), ("occupied_bricks", occupied.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single-GPU run (each rank of a sharded run holds only its slab)")
    import torch
    from rrpy import capi, multigpu, synth
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    for kv in filter(None, args.tune.split(",")):
        capi.set_tunable(kv.split("=")[0], int(kv.split("=")[1]))
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=300))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bricks = args.mode == "bricks"

    scenes, inv, voxel = make_inputs()
    rig = Rig(torch, dist, rank, world, local, scenes, inv, voxel, N_SENSORS, R, bricks, capi.VOXELS_F32)
    fu, stream = rig.fu, rig.stream
    cb, db = rig.cb, rig.db

    sampler = ClockSampler(local, args.clock_ms) if (rank == 0 and args.clock_ms > 0) else None
    ms_total = rig.timed(rig.step_device, args.steps, args.warmup)
    gpu_launches, host_enqueue_ms = rig.launches, rig.host_ms
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fu)
    # stage breakdown and the dominant kernel's launch duration: the same steps again with CUDA-event stage timers on the
    # context's stream (timers need direct launches, so this pass is not the one `value` comes from)
    stage_steps = max(10, min(args.steps, 100))
    ms_stage_pass = rig.timed(rig.step_device, stage_steps, 3, with_stage_timers=True)
    int_ms, int_n = fu.stage_stats("2integrate")
    pre_ms, pre_n = fu.stage_stats("1preprocess")
    int_slowest = rig.max_over_ranks(int_ms / max(1, int_n))      # the slab that gates the step (stage timers are per rank)

    # ---- end to end from pinned host buffers ------------------------------------------------------------------------
    e2e_warm = max(50, args.warmup)                 # >= 50 untimed steps: lets the PCIe link leave its idle state
    if world == 1:
        fu.stage_frames_ptr(rig.h_color[0].data_ptr(), cb, rig.h_depth[0].data_ptr(), db)     # prologue of the ingest pipeline
    # the closing swap makes the compute stream (and so the end event) wait for the last staged copy: all K host->device
    # copies issued inside the timed region are also completed inside it
    ms_e2e = rig.timed(rig.step_host, args.steps, e2e_warm, finish=(fu.swap_frames if world == 1 else None))
    e2e_path = ("rr_stage_frames / rr_swap_frames (20 MB host->device per step on a copy stream) + rr_fuse_frame (one CUDA-graph launch) + "
                "rr_bricks_count (4-byte read when the frame set is done)") if world == 1 else \
               "rank 0: pinned host -> broadcast slot, NCCL broadcast, every rank rr_fuse_frame + rr_bricks_count"
    link_gbs = None
    e2e_streams = {}
    if world == 1:
        # what bounds e2e: the host->device link. Bandwidth of the same 20 MB pinned copy alone (CUDA events, copy stream idle).
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_copies = 50
        for _ in range(5):
            rig.d_color[0].copy_(rig.h_color[0], non_blocking=True); rig.d_depth[0].copy_(rig.h_depth[0], non_blocking=True)
        torch.cuda.synchronize(dev)
        l0.record()
        for _ in range(n_copies):
            rig.d_color[0].copy_(rig.h_color[0], non_blocking=True); rig.d_depth[0].copy_(rig.h_depth[0], non_blocking=True)
        l1.record()
        torch.cuda.synchronize(dev)
        link_gbs = (cb + db) * n_copies / (l0.elapsed_time(l1) / 1e3) / 1e9
        # the same step fed the reference's stream formats (compress_rgb: 1 is its default, KinectCalibrationFile.cpp:94):
        # DXT1 colour blocks, and DXT1 + 8-bit sqrt-compressed depth, decoded on the device inside the captured frame graph
        h_dxt = [torch.from_numpy(np.stack([synth.encode_dxt1(s.color[i]) for i in range(N_SENSORS)])).pin_memory() for s in scenes]
        near_far = np.tile(np.array([0.5, 4.5], np.float32), (N_SENSORS, 1))
        h_d8 = [torch.from_numpy(np.stack([synth.encode_depth8(s.depth[i], 0.5, 4.5) for i in range(N_SENSORS)])).pin_memory() for s in scenes]
        for key, dxt1, d8 in (("dxt1_stream", True, False), ("dxt1_depth8_stream", True, True)):
            fu.synchronize()
            fu.set_frame_format(dxt1_color=dxt1, depth8=d8, near_far=near_far if d8 else None)
            rig.h_src_c, rig.h_src_cb = h_dxt, h_dxt[0].numel()
            rig.h_src_d, rig.h_src_db = (h_d8, h_d8[0].numel()) if d8 else (rig.h_depth, db)
            rig.flags = (True, not d8, True)      # pre_morph.fs validates metres: 8-bit streams run with useProcessedDepths(false)
            fu.stage_frames_ptr(rig.h_src_c[0].data_ptr(), rig.h_src_cb, rig.h_src_d[0].data_ptr(), rig.h_src_db)
            ms_s = rig.timed(rig.step_host, args.steps, e2e_warm, finish=fu.swap_frames)
            fps_s = args.steps / (ms_s / 1e3)
            e2e_streams[key] = {"value": round(R ** 3 * fps_s / 1e9, 3), "unit": "Gvoxel-updates/s", "frames_per_s": round(fps_s, 2),
                                "h2d_bytes_per_step": int(rig.h_src_cb + rig.h_src_db), "d2h_bytes_per_step": 4,
                                "what": "same step through rr_fuse_frame, colour streamed as DXT1 blocks" + (" and depth as 8-bit sqrt-compressed bytes" if d8 else "") +
                                        ", decoded on the device (different input precision than the RGB8 / float32 headline)"}
        fu.synchronize()
        fu.set_frame_format(dxt1_color=False)
        rig.flags = (True, True, True)
        rig.h_src_c, rig.h_src_d, rig.h_src_cb, rig.h_src_db = rig.h_color, rig.h_depth, cb, db
        fu.upload_frames_ptr(rig.d_color[0].data_ptr(), cb, rig.d_depth[0].data_ptr(), db, device=True)
    if world > 1:
        # N > 1: the same end-to-end step with the frame set streamed and BROADCAST in the reference's compressed formats (DXT1
        # colour + 8-bit depth: 3.6 MB instead of 20 MB over the host link and over NVLink), decoded on every GPU
        rig.barrier()
        near_far = np.tile(np.array([0.5, 4.5], np.float32), (N_SENSORS, 1))
        fu.synchronize()
        fu.set_frame_format(dxt1_color=True, depth8=True, near_far=near_far)
        cb2, db2 = N_SENSORS * CW * CH // 2, N_SENSORS * W * H
        keep = (rig.fb, rig.cb, rig.db, rig.h_packed)
        rig.fb, rig.cb, rig.db = multigpu.FrameBroadcaster(dist, dev, cb2, db2, src=0), cb2, db2
        if rank == 0:
            rig.h_packed = [torch.from_numpy(np.concatenate([np.stack([synth.encode_dxt1(s.color[i]) for i in range(N_SENSORS)]).reshape(-1),
                                                             np.stack([synth.encode_depth8(s.depth[i], 0.5, 4.5) for i in range(N_SENSORS)]).reshape(-1)])).pin_memory()
                            for s in scenes]
        rig.flags = (True, False, True)
        ms_s = rig.timed(rig.step_host, args.steps, e2e_warm)
        rig.flags = (True, True, True)
        fps_s = args.steps / (ms_s / 1e3)
        e2e_streams["dxt1_depth8_stream"] = {
            "value": round(R ** 3 * fps_s / 1e9, 3), "unit": "Gvoxel-updates/s", "frames_per_s": round(fps_s, 2),
            "h2d_bytes_per_step": int(cb2 + db2), "d2h_bytes_per_step": 4,
            "what": "same step, the frame set streamed to rank 0 and broadcast as DXT1 colour blocks + 8-bit sqrt-compressed depth, decoded on every GPU "
                    "(different input precision than the RGB8 / float32 headline; pre_morph skipped as for every 8-bit stream)"}
        rig.barrier()
        fu.synchronize()
        fu.set_frame_format(dxt1_color=False)
        rig.fb, rig.cb, rig.db, rig.h_packed = keep
    bcast_ms = None
    if world > 1:
        # the broadcast alone (nothing else on the GPUs): what the pipelined step hides, or is bound by
        rig.barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            rig.fb.issue(packed=rig.d_packed[0]); rig.fb.consume(stream)
        torch.cuda.synchronize(dev)
        b0.record()
        for _ in range(20):
            rig.fb.issue(packed=rig.d_packed[0]); rig.fb.consume(stream)
        b1.record()
        torch.cuda.synchronize(dev)
        bcast_ms = rig.max_over_ranks(b0.elapsed_time(b1) / 20)
    # keep the GPU busy until nvidia-smi has a few samples under load (the timed region can be < 100 ms). Every rank
    # runs the same number of extra steps (derived from the all-reduced step time), since steps contain collectives.
    n_extra = int(min(20000, max(64, 1200.0 / max(1e-3, ms_total / args.steps))))
    for i in range(n_extra):
        rig.step_device(i)
        if i % 64 == 63:
            fu.synchronize()
    rig.barrier()
    clocks = sampler.stop() if sampler else None

    n_occ, ratio, n_occ_vox, nbricks = rig.occupancy()
    info = fu.integrator_info()

    # ---- the view path (reported beside the headline and combined with it): raymarch at 1280x720 + colour hole filling; for
    # N > 1 every rank marches its slab into partial records and two reductions composite them on rank 0
    mv = synth.look_at((1.7, 1.6, 2.3), (0.0, 1.1, 0.0))
    pr = synth.perspective(50.0, VW / VH, 0.1, 10.0)
    # N > 1: every rank marches its slab into its own view images; rank 0 composites them with ONE kernel that reads the other
    # ranks' first-hit keys and the winners' pixels straight out of their memory (CUDA IPC over NVLink: rr_view_export /
    # rr_composite_peers, the kernel of rr_group_raymarch). Two stream-ordered one-element all-reduces fence the ranks: the
    # peers' marches are complete before rank 0 reads them, and no peer marches again before rank 0 has finished.
    peer_handles = []
    fence = torch.zeros(1, dtype=torch.int32, device=dev) if world > 1 else None
    if world > 1:
        fu.raymarch(mv, pr, VW, VH, shade_mode=1, download=False)          # allocates the view images at this size
        fu.synchronize()
        blobs = [None] * world
        dist.all_gather_object(blobs, fu.view_export(VW, VH))
        peer_handles = [blobs[r] for r in range(world) if r != 0]

    def stream_fence():
        cur = torch.cuda.current_stream(dev)
        cur.wait_stream(stream)
        dist.all_reduce(fence)
        stream.wait_stream(cur)

    def view_once(download=False):
        if world == 1:
            fu.raymarch(mv, pr, VW, VH, shade_mode=1, download=False)
            fu.fill_colors(download=False)          # m_fill_holes is on by default (recon_integration.cpp:54)
            return None
        fu.raymarch(mv, pr, VW, VH, shade_mode=1, download=False)
        stream_fence()
        out = None
        if rank == 0:
            out = fu.composite_peers(peer_handles, VW, VH, download=download)
            fu.fill_colors(download=False)
        stream_fence()
        return out

    for _ in range(3):
        view_once()
    rig.barrier()
    v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_views = 20
    v0.record(stream)
    for _ in range(n_views):
        view_once()
    v1.record(stream)
    rig.barrier()
    view_ms = rig.max_over_ranks(v0.elapsed_time(v1) / n_views)

    # ---- the other reconstructions of SURVEY.md 8f-4 on the same maps, one view each (device time of the library's `draw`
    # stage timer; tools/bench_renderers.py is the same measurement on its own). Evidence beside the headline, never a
    # reason to fail the line.
    renderers = None
    if world == 1 and args.subrecords:
        try:
            fu.set_timing(2)
            renderers = {"resolution": [VW, VH], "what": "one view of rr_draw_points / rr_draw_calibs / rr_draw_trigrid (ReconPoints, ReconCalibs, "
                         "ReconTrigrid) on the last frame set's maps; median device ms of 10 views"}
            for name, call in (("draw_points", lambda: fu.draw_points(mv, pr, VW, VH, shade_mode=1)),
                               ("draw_calibs", lambda: fu.draw_calibs(mv, pr, VW, VH, active_kinect=0, limit=LIMIT)),
                               ("draw_trigrid", lambda: fu.draw_trigrid(mv, pr, VW, VH, shade_mode=1))):
                ms = []
                for i in range(12):
                    img = call()
                    if i >= 2:
                        ms.append(fu.stage_ms("draw"))
                renderers[name] = {"ms_per_view": round(float(np.median(ms)), 4), "covered_px": int((img[1] < 1.0).sum())}
            fu.set_timing(0)
        except Exception as e:                                   # pragma: no cover
            renderers = {"error": str(e)[:200]}

    # ---- N > 1: this run's slabs and composited view against a single-context run, bit for bit ---------------------------
    verified = None
    if world > 1:
        verified = verify_against_single_context(torch, dist, rig, scenes, inv, voxel, bricks, mv, pr, view_once)

    frames_s = args.steps / (ms_total / 1e3)
    value = R ** 3 * frames_s / 1e9
    e2e_frames_s = args.steps / (ms_e2e / 1e3)
    int_avg_ms = int_ms / max(1, int_n)
    abytes, achieved, peak, peak_src = rig.roofline(int_avg_ms, n_occ_vox, nbricks)
    traffic, traffic_src = measured_traffic(bricks) if world == 1 else (None, None)
    ms_step = ms_total / args.steps
    slab_vox = R ** 3 * (rig.zc1 - rig.zc0) / R
    rig.close()

    # ---- sub-records through the same code (device-resident frames, rr_fuse_frame): dense mode and BASELINE config 5 -----
    dense = config5 = config1 = config2 = config3 = None
    if args.subrecords and world == 1:
        # the other BASELINE.json configurations, single GPU (their parity tests are in tests/; bench lines of the same in tools/)
        config1 = invert_record(torch)
        config2 = sub_record(torch, dist, rank, world, local, "BASELINE.json configs[1]: 1 sensor 512x424, 128^3 R32F TSDF, occupied bricks, + raymarch",
                             1, 128, True, capi.VOXELS_F32, 50, view=True)
        config3 = sub_record(torch, dist, rank, world, local, "BASELINE.json configs[2]: 4 sensors, 256^3 R32F TSDF, brick culling, + raymarch and colour fill",
                             4, 256, True, capi.VOXELS_F32, 50, view=True)
    if args.subrecords:
        if bricks:
            dense = sub_record(torch, dist, rank, world, local, "same workload with setUseBricks(false): every voxel x every sensor",
                               N_SENSORS, R, False, capi.VOXELS_F32, 20, scenes[:1], inv, voxel)
        config5 = sub_record(torch, dist, rank, world, local,
                             "BASELINE.json configs[4]: 8 sensors 512x424, 1024^3 TSDF with half2 (tsdf, weight) voxels, occupied bricks, "
                             "same z-slab code (one NCCL broadcast of the 40 MB frame set per step for N > 1)", 8, 1024, True, capi.VOXELS_HALF2, 30)

    out = {
        "metric": "4-sensor TSDF Gvoxel-updates/s at 512^3 (fused frames/s in frames_per_s)",
        "value": round(value, 3), "unit": "Gvoxel-updates/s", "frames_per_s": round(frames_s, 2),
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 5),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "integration": INTEGRATION[bricks],
                   "parallelism": f"z-slabs x{world}" if world > 1 else "single GPU", "slabs": rig.slab_how,
                   "l2": "inputs+outputs per step (268 MB inverse volumes, 537 MB TSDF) exceed the 126 MB L2; no explicit flush",
                   "occupied_bricks": int(n_occ), "occupied_ratio": round(float(ratio), 4), "frames_cycled": N_FRAMES, "integrator": info},
        "e2e": {"value": round(R ** 3 * e2e_frames_s / 1e9, 3), "unit": "Gvoxel-updates/s", "frames_per_s": round(e2e_frames_s, 2),
                "h2d_bytes_per_step": int(cb + db), "d2h_bytes_per_step": 4, "path": e2e_path,
                "h2d_link_gbs": round(link_gbs, 2) if link_gbs else None,
                "bound": (f"host->device link: {cb + db} B/step at the measured {link_gbs:.1f} GB/s caps e2e at {link_gbs * 1e9 / (cb + db):.0f} frames/s" if link_gbs else None),
                **e2e_streams},
        "gpu_launches": int(gpu_launches), "host_enqueue_ms_per_step": round(host_enqueue_ms, 5),
        # SURVEY.md 8d: beside voxel-updates/s, the evaluations actually performed (this rank's slab for N > 1)
        "occupied_voxel_updates_per_s": round(float(n_occ_vox if bricks else slab_vox) * frames_s, 1),
        "voxel_sensor_evaluations_per_s": round(float(n_occ_vox if bricks else slab_vox) * N_SENSORS * frames_s, 1),
        "stages_ms": {"1preprocess": round(pre_ms / max(1, pre_n), 5), "2integrate": round(int_avg_ms, 5),
                      **({"2integrate_slowest_rank": round(int_slowest, 5)} if world > 1 else {}),
                      "how": f"CUDA-event stage timers over {stage_steps} further steps of the same loop with direct launches "
                             f"({ms_stage_pass / stage_steps:.5f} ms/step); `value` is timed with the frame replayed as one CUDA graph"},
        "view": {"ms_per_view": round(view_ms, 4), "resolution": [VW, VH],
                 "what": "tsdf_raymarch (shaded, brick space skipping) + colour hole filling" +
                         (" per slab; one compositing kernel on rank 0 reads the other ranks' first-hit keys and the winners' pixels through CUDA IPC peer memory (rr_composite_peers), fenced by two one-element all-reduces" if world > 1 else "")},
        # SURVEY.md 8d "reported separately and combined": one fused frame set followed by one view
        "combined_frames_per_s": round(1e3 / (ms_step + view_ms), 2),
        "renderers": renderers,
        "roofline": {"bound": "hbm", "kernel": integrate_kernel_name(bricks, info),
                     "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": int(abytes), "peak_source": peak_src,
                     "algorithmic_bytes": "SURVEY.md 8d: 4*XYZ + 4*V_occ + 16*covered_inverse_voxels*N + 16*pixels*N + 4*bricks"},
        "dense": dense, "config5": config5, "config1": config1, "config2": config2, "config3": config3,
        "clocks": clocks,
    }
    if world > 1:
        out["verified"] = verified
        out["broadcast"] = {"bytes": int(cb + db), "ms_alone": round(bcast_ms, 4), "gbs": round((cb + db) / bcast_ms / 1e6, 1),
                            "what": "one packed NCCL broadcast per frame set, double-buffered beside the previous set's kernels",
                            "nccl_min_nchannels": os.environ.get("NCCL_MIN_NCHANNELS")}
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(scenes[0], inv, voxel, bricks, budget_s=12.0)
        emit(out)


def cpu_frame(scene, inv, voxel, bricks, threads, int_fraction=1.0):
    """One fused frame with the oracle port on `threads` host threads. Returns (seconds_pre, seconds_int, n_occ)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    O.set_threads(threads)
    grid = O.brick_grid(scene.bbox_min, scene.bbox_max, voxel, BRICK)
    cams = [O.frustum(scene.cv_xyz[i])[1] for i in range(scene.N)]
    t0 = time.perf_counter()
    pre = O.preprocess(scene, grid, cams)
    occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
    t1 = time.perf_counter()
    if bricks:
        sub = occ[:: max(1, int(round(1.0 / int_fraction)))]
        O.integrate(inv, pre, grid, LIMIT, True, sub)
        scale = len(occ) / max(1, len(sub))
    else:
        raise NotImplementedError
    t2 = time.perf_counter()
    return t1 - t0, (t2 - t1) * scale, len(occ), len(sub)


def cpu_baseline(scene, inv, voxel, bricks, budget_s):
    """The oracle port timed on this box's host cores on a bounded sample of the same workload: whole fused frames
    (all pixels, all occupied bricks) repeated until ~budget_s seconds of CPU work are spent."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    cores = host_cores()
    O.set_threads(cores)
    times, tps, tis = [], [], []
    t_start = time.perf_counter()
    n_occ = 0
    while True:
        tp, ti, n_occ, _ = cpu_frame(scene, inv, voxel, True, cores, 1.0)
        times.append(tp + ti); tps.append(tp); tis.append(ti)
        if (time.perf_counter() - t_start >= budget_s and len(times) >= 2) or len(times) >= 200:
            break
    fps = 1.0 / float(np.mean(times))
    # SURVEY.md 8d also asks for the single-threaded figure: one whole frame set on one thread
    tp1, ti1, _, _ = cpu_frame(scene, inv, voxel, True, 1, 1.0)
    O.set_threads(cores)
    return {"value": round(R ** 3 * fps / 1e9, 5), "unit": "Gvoxel-updates/s", "frames_per_s": round(fps, 4), "cores": cores, "kind": "port",
            "single_thread_frames_per_s": round(1.0 / (tp1 + ti1), 4),
            "sample": f"{len(times)} whole 4-sensor frame sets at {R}^3 ({sum(times):.1f} s of wall time on {cores} threads): per frame all 5 "
                      f"pre-process passes on every pixel ({np.mean(tps) * 1e3:.0f} ms) + brick integration of all {n_occ} occupied bricks "
                      f"({np.mean(tis) * 1e3:.0f} ms); oracle port (-O2, OpenMP), bricks mode"}


def run_reference(args):
    """The reference's own algorithm for this path on the host cores. The reference (GLSL, needs an OpenGL 4.4 context,
    CGAL, ZeroMQ) cannot be built here, so this is the oracle port — the scalar C++ transcription of its shaders."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    scenes, inv, voxel = make_inputs()
    cores = host_cores()                 # every host thread of the box, whatever OMP_NUM_THREADS the launcher exported
    O.set_threads(cores)
    frac = 1.0
    times = []
    n_occ = n_sub = 0
    total = args.warmup + args.steps
    for i in range(total):
        tp, ti, n_occ, n_sub = cpu_frame(scenes[i % N_FRAMES], inv, voxel, True, cores, frac)
        if i == 0 and (tp + ti / 1.0) * total > 150.0:
            # bound the whole run to a few minutes: shrink the integrated brick sample for the remaining steps
            frac = max(1.0 / 64.0, frac * 150.0 / ((tp + ti) * total))
        if i >= args.warmup:
            times.append(tp + ti)
    t = float(np.mean(times))
    fps = 1.0 / t
    value = R ** 3 * fps / 1e9
    shader_harness = None
    try:
        # beside the port: the reference's OWN shaders compiled as C++ (oracle/_ref/libref_glsl.so, a correctness tool: one
        # shader object is copied per fragment) on one frame set - pre-processing in full, integration on a brick sample
        import ref_glsl_py as G
        if G.available():
            sc = scenes[0]
            grid = O.brick_grid(sc.bbox_min, sc.bbox_max, voxel, BRICK)
            cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
            t0 = time.perf_counter()
            pre = G.preprocess(sc, grid, cams)
            t1 = time.perf_counter()
            occ = O.occupied_bricks(pre["bricks"], MIN_VOX)
            sub = occ[::16]
            tc0 = time.perf_counter()
            G.integrate(inv, pre, grid, LIMIT, True, occ[:0])                   # the clear alone (not scaled with the brick sample)
            t2 = time.perf_counter()
            G.integrate(inv, pre, grid, LIMIT, True, sub)
            t3 = time.perf_counter()
            t_clear = t2 - tc0
            sec = (t1 - t0) + t_clear + max(0.0, (t3 - t2) - t_clear) * len(occ) / max(1, len(sub))
            shader_harness = {"kind": "reference", "frames_per_s": round(1.0 / sec, 4), "cores": cores,
                              "sample": f"1 frame set: 5 shader passes on every pixel ({(t1 - t0) * 1e3:.0f} ms) + tsdf_integration.vs on "
                                        f"{len(sub)} of {len(occ)} occupied bricks, scaled"}
    except Exception as e:                                   # the harness is optional evidence, never a reason to fail the arm
        shader_harness = {"unavailable": str(e)[:120]}
    out = {"impl": "reference", "metric": "4-sensor TSDF Gvoxel-updates/s at 512^3 (fused frames/s in frames_per_s)",
           "value": round(value, 5), "unit": "Gvoxel-updates/s", "frames_per_s": round(fps, 4), "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": round(t * 1e3, 2), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": WORKLOAD, "integration": INTEGRATION[True]},
           "cpu_baseline": {"value": round(value, 5), "unit": "Gvoxel-updates/s", "cores": cores, "kind": "port",
                            "sample": f"per step: full pre-processing of 4x512x424 pixels + integration of {n_sub} of {n_occ} occupied bricks, "
                                      f"integration time scaled to all occupied bricks"},
           "e2e": {"value": round(value, 5), "unit": "Gvoxel-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "reference_shaders_on_cpu": shader_harness}
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="bricks", choices=["bricks", "dense"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-subrecords", dest="subrecords", action="store_false", help="skip the dense and config5 sub-records")
    ap.add_argument("--tune", default="", help="integrator tunables k=v,k=v applied on every rank (A/B measurements; results never depend on them)")
    ap.add_argument("--clock-ms", type=int, default=100, help="nvidia-smi sampling period during the timed regions (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
