"""ctypes binding of librr_b200.so (include/rgbd_recon_b200.h) for tests and bench.py.

This is harness code: the product's host side is the C++ in rgbd-recon_b200/host/. Loading fails loudly when the
CUDA library has not been built; there is no CPU fallback of any kind.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RR_B200_LIB") or os.path.join(os.path.dirname(_HERE), "librr_b200.so")   # RR_B200_LIB: the profiling build (make prof)
HEADER_PATH = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "include", "rgbd_recon_b200.h")

STAGES = dict(morph=0, depth=1, lab=2, depth_b=3, sil=4, normal=5, quality=6)
_STAGE_CH = dict(morph=1, depth=2, lab=3, depth_b=2, sil=1, normal=3, quality=1)


class Config(C.Structure):
    _fields_ = [("limit", C.c_float), ("voxel_size", C.c_float), ("brick_size", C.c_float),
                ("min_voxels_per_brick", C.c_uint32), ("use_bricks", C.c_int32), ("skip_space", C.c_int32),
                ("store_weight", C.c_int32)]


# rr_voxel_format (rr_config.store_weight)
VOXELS_F32, VOXELS_F32_WEIGHT, VOXELS_HALF2 = 0, 1, 2

# rr_integrator_last()[0]
INTEGRATE_PATHS = ("none", "staged", "fused", "two_kernel", "dense")
# rr_integrator_last()[5]
INTEGRATE_CLEARS = ("none", "full", "incremental")


class View(C.Structure):
    _fields_ = [("modelview", C.c_float * 16), ("projection", C.c_float * 16), ("viewport", C.c_int32 * 4),
                ("shade_mode", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `make -C rgbd-recon_b200` (or __graft_entry__.build()); "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, f32, u32, i32 = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_int32)
    L.rr_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.rr_destroy.argtypes = [vp]
    L.rr_destroy.restype = None
    L.rr_last_error.argtypes = [vp]
    L.rr_last_error.restype = C.c_char_p
    L.rr_synchronize.argtypes = [vp]
    L.rr_stream.argtypes = [vp]
    L.rr_stream.restype = vp
    L.rr_set_bbox.argtypes = [vp, f32, f32]
    L.rr_calib_upload.argtypes = [vp, C.c_int, f32, f32, u32, f32]
    L.rr_calib_upload_inv.argtypes = [vp, C.c_int, f32, u32]
    L.rr_get_camera_positions.argtypes = [vp, f32]
    L.rr_get_frustum_planes.argtypes = [vp, C.c_int, f32]
    L.rr_calib_invert.argtypes = [vp, C.c_int, u32, f32, C.c_int]
    L.rr_configure.argtypes = [vp, C.POINTER(Config)]
    L.rr_get_volume_res.argtypes = [vp, u32]
    L.rr_get_brick_info.argtypes = [vp, u32, f32, u32]
    L.rr_get_brick_ranges.argtypes = [vp, i32]
    L.rr_set_slab.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.rr_upload_frames.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t]
    L.rr_upload_frames_device.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t]
    L.rr_stage_frames.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t]
    L.rr_swap_frames.argtypes = [vp]
    L.rr_set_frame_format.argtypes = [vp, C.c_int, C.c_int, f32]
    L.rr_stage_sync.argtypes = [vp]
    L.rr_bricks_clear.argtypes = [vp]
    L.rr_preprocess.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rr_bricks_update.argtypes = [vp, u32, f32]
    L.rr_integrate.argtypes = [vp]
    L.rr_fuse_frame.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rr_bricks_count.argtypes = [vp, u32, f32]
    L.rr_raymarch.argtypes = [vp, C.POINTER(View), f32, f32]
    L.rr_raymarch_partial.argtypes = [vp, C.POINTER(View), vp]
    L.rr_composite.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, f32, f32]
    L.rr_partial_keys.argtypes = [vp, vp, C.c_int, vp]
    L.rr_partial_keep_winners.argtypes = [vp, vp, vp, C.c_int]
    L.rr_fill_colors.argtypes = [vp, f32]
    L.rr_upload_view.argtypes = [vp, C.c_int, C.c_int, f32, f32]
    L.rr_download_tsdf.argtypes = [vp, f32]
    L.rr_download_weight.argtypes = [vp, f32]
    L.rr_download_stage.argtypes = [vp, C.c_int, f32]
    L.rr_download_bricks.argtypes = [vp, u32, u32, u32]
    L.rr_download_num_samples.argtypes = [vp, f32]
    L.rr_download_hit_positions.argtypes = [vp, f32]
    L.rr_set_timing.argtypes = [vp, C.c_int]
    L.rr_get_stage_ms.argtypes = [vp, C.c_char_p, f32]
    L.rr_get_stage_stats.argtypes = [vp, C.c_char_p, f32, u32]
    L.rr_integrator_info.argtypes = [vp, u32]
    L.rr_integrator_profile.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.rr_integrator_last.argtypes = [vp, u32]
    L.rr_integrator_cleared.argtypes = [vp, u32]
    L.rr_draw_points.argtypes = [vp, C.POINTER(View), f32, f32]
    L.rr_draw_calibs.argtypes = [vp, C.POINTER(View), C.c_int, C.c_float, f32, f32]
    L.rr_draw_trigrid.argtypes = [vp, C.POINTER(View), C.c_float, f32, f32]
    L.rr_view_export.argtypes = [vp, C.c_int, C.c_int, vp]
    L.rr_composite_peers.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, f32, f32]
    # one process, several GPUs
    L.rr_group_create.argtypes = [C.POINTER(vp), i32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.rr_group_destroy.argtypes = [vp]
    L.rr_group_destroy.restype = None
    L.rr_group_size.argtypes = [vp]
    L.rr_group_member.argtypes = [vp, C.c_int]
    L.rr_group_member.restype = vp
    L.rr_group_last_error.argtypes = [vp]
    L.rr_group_last_error.restype = C.c_char_p
    L.rr_group_synchronize.argtypes = [vp]
    L.rr_group_set_bbox.argtypes = [vp, f32, f32]
    L.rr_group_calib_upload.argtypes = [vp, C.c_int, f32, f32, u32, f32]
    L.rr_group_calib_upload_inv.argtypes = [vp, C.c_int, f32, u32]
    L.rr_group_set_frame_format.argtypes = [vp, C.c_int, C.c_int, f32]
    L.rr_group_set_timing.argtypes = [vp, C.c_int]
    L.rr_group_configure.argtypes = [vp, C.POINTER(Config)]
    L.rr_group_set_slabs.argtypes = [vp, u32]
    L.rr_group_get_slabs.argtypes = [vp, u32]
    L.rr_group_balance_slabs.argtypes = [vp, C.c_float]
    L.rr_group_stage_frames.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t]
    L.rr_group_swap_frames.argtypes = [vp]
    L.rr_group_stage_sync.argtypes = [vp]
    L.rr_group_upload_frames.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t]
    L.rr_group_bricks_clear.argtypes = [vp]
    L.rr_group_preprocess.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rr_group_bricks_update.argtypes = [vp, u32, f32]
    L.rr_group_integrate.argtypes = [vp]
    L.rr_group_fuse_frame.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rr_group_bricks_count.argtypes = [vp, u32, f32]
    L.rr_group_raymarch.argtypes = [vp, C.POINTER(View), f32, f32]
    L.rr_group_fill_colors.argtypes = [vp, f32]
    L.rr_group_download_tsdf.argtypes = [vp, f32]
    L.rr_extract_mesh.argtypes = [vp, u32, u32]
    L.rr_download_mesh.argtypes = [vp, f32, f32, f32, u32]
    L.rr_group_extract_mesh.argtypes = [vp, u32, u32]
    L.rr_sample_points.argtypes = [vp, C.c_int, vp, C.c_uint32, vp, vp, vp]
    L.rr_cast_rays.argtypes = [vp, C.c_int, vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.rr_group_sample_points.argtypes = [vp, C.c_int, vp, C.c_uint32, vp, vp, vp]
    L.rr_group_cast_rays.argtypes = [vp, C.c_int, vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.rr_extract_points.argtypes = [vp, C.c_uint32, u32]
    L.rr_download_points.argtypes = [vp, vp, vp, vp, vp, vp]
    L.rr_group_extract_points.argtypes = [vp, C.c_uint32, u32]
    L.rr_label_parts.argtypes = [vp, u32]
    L.rr_download_parts.argtypes = [vp, vp, vp, vp, vp]
    L.rr_download_mesh_parts.argtypes = [vp, vp, vp]
    L.rr_group_label_parts.argtypes = [vp, u32]
    L.rr_track_parts.argtypes = [vp, C.c_uint32, u32, u32]
    L.rr_download_part_tracks.argtypes = [vp, vp, vp, vp, vp]
    L.rr_reset_part_tracks.argtypes = [vp]
    L.rr_group_track_parts.argtypes = [vp, C.c_uint32, u32, u32]
    L.rr_simplify_mesh.argtypes = [vp, C.c_uint32, u32, u32]
    L.rr_download_simplified_mesh.argtypes = [vp, vp, vp, vp, vp, vp]
    L.rr_group_simplify_mesh.argtypes = [vp, C.c_uint32, u32, u32]
    L.rr_launch_count.argtypes = [vp]
    L.rr_launch_count.restype = C.c_uint64
    L.rr_version.restype = C.c_int
    L.rr_set_tunable.argtypes = [C.c_char_p, C.c_int]
    _lib = L
    return L


def set_tunable(name, value):
    if lib().rr_set_tunable(name.encode(), int(value)) != 0:
        raise ValueError(f"unknown tunable {name}")


def _f32(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _u32(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


# rr_sample_points / rr_cast_rays: RR_QUERY_WORLD (metres) or RR_QUERY_VOLUME (texture coordinates over the bbox)
QUERY_SPACES = dict(world=0, volume=1)


def _query_inputs(*arrays):
    """[n, 3] float32 query inputs as (pointers, n, keep-alive, torch device or None). numpy-like inputs go as host memory;
    torch tensors by data_ptr(), on the host or on the context's GPU (the caller's stream is synchronised first, as the
    library reads them on its own stream)."""
    ptrs, keep, device = [], [], None
    for a in arrays:
        if type(a).__module__.startswith("torch"):
            import torch
            t = a.detach().to(torch.float32).contiguous().reshape(-1, 3)
            if t.is_cuda:
                torch.cuda.current_stream(t.device).synchronize()
                device = t.device
            ptrs.append(t.data_ptr())
            keep.append(t)
        else:
            arr = np.ascontiguousarray(a, np.float32).reshape(-1, 3)
            ptrs.append(arr.ctypes.data)
            keep.append(arr)
    n = keep[0].shape[0]
    if any(k.shape[0] != n for k in keep):
        raise ValueError("origins and directions differ in length")
    return ptrs, n, keep, device


def _query_outputs(device, *shapes_and_types):
    """Output arrays: torch tensors on `device` when the inputs were CUDA tensors, numpy arrays otherwise; and their pointers."""
    outs = []
    for shape, dt in shapes_and_types:
        if device is not None:
            import torch
            outs.append(torch.empty(shape, dtype=dict(f4=torch.float32, u4=torch.uint32)[dt], device=device))
        else:
            outs.append(np.empty(shape, np.dtype(dt)))
    ptrs = [o.data_ptr() if device is not None else o.ctypes.data for o in outs]
    return outs, ptrs


def _sample_points(call, points, space):
    ptrs, n, keep, device = _query_inputs(points)
    outs, op = _query_outputs(device, ((n,), "f4"), ((n, 3), "f4"), ((n, 4), "f4"))
    call(QUERY_SPACES[space], ptrs[0], n, *op)
    return tuple(outs)


def _cast_rays(call, origins, directions, space):
    ptrs, n, keep, device = _query_inputs(origins, directions)
    outs, op = _query_outputs(device, ((n, 3), "f4"), ((n, 3), "f4"), ((n, 4), "f4"), ((n,), "u4"))
    call(QUERY_SPACES[space], ptrs[0], ptrs[1], n, *op)
    return tuple(outs)


def _sensor_mask(sensors, n_sensors):
    """rr_extract_points' sensor_mask of an iterable of sensor indices (None: every sensor). Indices at or above the sensor
    count are left for the library to refuse."""
    if sensors is None:
        return (1 << n_sensors) - 1
    mask = 0
    for i in sensors:
        i = int(i)
        if not 0 <= i < 32:
            raise ValueError(f"sensor index {i} out of range")
        mask |= 1 << i
    return mask


class RRError(RuntimeError):
    pass


class Fusion:
    """Thin object wrapper: one rr_ctx. Method names follow the C ABI."""

    def __init__(self, N, W, H, CW, CH, device=0):
        self.L = lib()
        self.h = C.c_void_p()
        self.N, self.W, self.H, self.CW, self.CH = N, W, H, CW, CH
        self.device = int(device)
        rc = self.L.rr_create(C.byref(self.h), device, N, W, H, CW, CH)
        if rc != 0:
            raise RRError(f"rr_create failed with status {rc} (no CUDA device? there is no CPU fallback)")

    def close(self):
        if self.h:
            self.L.rr_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise RRError(f"status {rc}: {self.L.rr_last_error(self.h).decode()}")

    # calibration
    def set_bbox(self, bmin, bmax):
        bmin = np.ascontiguousarray(bmin, np.float32)
        bmax = np.ascontiguousarray(bmax, np.float32)
        self._ck(self.L.rr_set_bbox(self.h, _f32(bmin), _f32(bmax)))

    def calib_upload(self, sensor, cv_xyz, cv_uv, depth_limits=(0.5, 4.5)):
        Z, Y, X, _ = cv_xyz.shape
        xyz = np.ascontiguousarray(cv_xyz, np.float32)
        uv = np.ascontiguousarray(cv_uv, np.float32)
        res = np.array([X, Y, Z], np.uint32)
        dl = np.array(depth_limits, np.float32)
        self._ck(self.L.rr_calib_upload(self.h, sensor, _f32(xyz), _f32(uv), _u32(res), _f32(dl)))

    def calib_upload_inv(self, sensor, inv):
        Z, Y, X, _ = inv.shape
        a = np.ascontiguousarray(inv, np.float32)
        res = np.array([X, Y, Z], np.uint32)
        self._ck(self.L.rr_calib_upload_inv(self.h, sensor, _f32(a), _u32(res)))

    def camera_positions(self):
        out = np.zeros((self.N, 3), np.float32)
        self._ck(self.L.rr_get_camera_positions(self.h, _f32(out)))
        return out

    def frustum_planes(self, sensor):
        out = np.zeros((6, 4), np.float32)
        self._ck(self.L.rr_get_frustum_planes(self.h, sensor, _f32(out)))
        return out

    def calib_invert(self, sensor, out_res, keep=False, download=True):
        ox, oy, oz = [int(v) for v in out_res]
        res = np.array([ox, oy, oz], np.uint32)
        out = np.zeros((oz, oy, ox, 4), np.float32) if download else None
        self._ck(self.L.rr_calib_invert(self.h, sensor, _u32(res), _f32(out) if download else None, int(keep)))
        return out

    # settings
    def configure(self, limit=0.01, voxel_size=0.01, brick_size=0.1, min_voxels=10, use_bricks=True, skip_space=True,
                  store_weight=False):
        """store_weight: False/0 R32F tsdf, True/1 + R32F weight volume, VOXELS_HALF2 (2) half2 (tsdf, weight) voxels."""
        cfg = Config(limit, voxel_size, brick_size, min_voxels, int(use_bricks), int(skip_space), int(store_weight))
        self._ck(self.L.rr_configure(self.h, C.byref(cfg)))

    def volume_res(self):
        r = np.zeros(3, np.uint32)
        self._ck(self.L.rr_get_volume_res(self.h, _u32(r)))
        return r

    def brick_info(self):
        rb = np.zeros(3, np.uint32)
        bs = C.c_float()
        nb = C.c_uint32()
        self._ck(self.L.rr_get_brick_info(self.h, _u32(rb), C.byref(bs), C.byref(nb)))
        return dict(res_bricks=rb, brick_size=np.float32(bs.value), num_bricks=int(nb.value))

    def brick_ranges(self):
        nb = self.brick_info()["num_bricks"]
        out = np.zeros((nb, 6), np.int32)
        self._ck(self.L.rr_get_brick_ranges(self.h, out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def set_slab(self, z0, z1):
        self._ck(self.L.rr_set_slab(self.h, int(z0), int(z1)))

    def set_frame_format(self, dxt1_color=False, depth8=False, near_far=None, dxt5_color=False):
        """Stream formats (rr_set_frame_format): DXT1 / DXT5 colour blocks and / or 8-bit sqrt-compressed depth."""
        nf = np.ascontiguousarray(near_far, np.float32) if near_far is not None else None
        self._depth8 = bool(depth8)
        self._ck(self.L.rr_set_frame_format(self.h, 5 if dxt5_color else (1 if dxt1_color else 0), 1 if depth8 else 0, _f32(nf) if nf is not None else None))

    # per frame
    def upload_frames(self, color, depth):
        depth = np.ascontiguousarray(depth, np.uint8 if getattr(self, "_depth8", False) else np.float32)
        if color is not None:
            color = np.ascontiguousarray(color, np.uint8)
        self._ck(self.L.rr_upload_frames(self.h, color.ctypes.data if color is not None else None,
                                         color.nbytes if color is not None else 0, depth.ctypes.data, depth.nbytes))
        self.synchronize()   # numpy buffers are pageable and may be temporaries

    def upload_frames_ptr(self, color_ptr, color_bytes, depth_ptr, depth_bytes, device=False):
        f = self.L.rr_upload_frames_device if device else self.L.rr_upload_frames
        self._ck(f(self.h, color_ptr, color_bytes, depth_ptr, depth_bytes))

    def stage_frames_ptr(self, color_ptr, color_bytes, depth_ptr, depth_bytes):
        """Async copy of a (pinned) host frame set into the back device slot; see rr_stage_frames."""
        self._ck(self.L.rr_stage_frames(self.h, color_ptr, color_bytes, depth_ptr, depth_bytes))

    def swap_frames(self):
        self._ck(self.L.rr_swap_frames(self.h))

    def stage_sync(self):
        self._ck(self.L.rr_stage_sync(self.h))

    def bricks_clear(self):
        self._ck(self.L.rr_bricks_clear(self.h))

    def preprocess(self, filter_textures=True, use_processed_depth=True, refine=True):
        self._ck(self.L.rr_preprocess(self.h, int(filter_textures), int(use_processed_depth), int(refine)))

    def bricks_update(self, sync=True):
        if not sync:
            self._ck(self.L.rr_bricks_update(self.h, None, None))
            return None
        n = C.c_uint32()
        r = C.c_float()
        self._ck(self.L.rr_bricks_update(self.h, C.byref(n), C.byref(r)))
        return int(n.value), float(r.value)

    def integrate(self):
        self._ck(self.L.rr_integrate(self.h))

    def raymarch(self, modelview, projection, width, height, shade_mode=0, download=True):
        v = View()
        v.modelview[:] = [float(x) for x in np.asarray(modelview, np.float32).reshape(16)]
        v.projection[:] = [float(x) for x in np.asarray(projection, np.float32).reshape(16)]
        v.viewport[:] = [0, 0, int(width), int(height)]
        v.shade_mode = int(shade_mode)
        self._vw, self._vh = int(width), int(height)
        if not download:
            self._ck(self.L.rr_raymarch(self.h, C.byref(v), None, None))
            return None
        rgba = np.zeros((height, width, 4), np.float32)
        depth = np.zeros((height, width), np.float32)
        self._ck(self.L.rr_raymarch(self.h, C.byref(v), _f32(rgba), _f32(depth)))
        return rgba, depth

    def draw_points(self, modelview, projection, width, height, shade_mode=0):
        """ReconPoints::draw (rr_draw_points) of the maps of the last preprocess; returns (rgba, depth)."""
        v = self._view(modelview, projection, width, height, shade_mode)
        self._vw, self._vh = int(width), int(height)
        rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
        self._ck(self.L.rr_draw_points(self.h, C.byref(v), _f32(rgba), _f32(depth)))
        return rgba, depth

    def draw_calibs(self, modelview, projection, width, height, active_kinect=0, limit=0.01):
        """ReconCalibs::draw (rr_draw_calibs): the inverse-volume grid's voxel centres coloured by the TSDF; returns (rgba, depth)."""
        v = self._view(modelview, projection, width, height, 0)
        self._vw, self._vh = int(width), int(height)
        rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
        self._ck(self.L.rr_draw_calibs(self.h, C.byref(v), int(active_kinect), float(limit), _f32(rgba), _f32(depth)))
        return rgba, depth

    def draw_trigrid(self, modelview, projection, width, height, shade_mode=0, min_length=0.0125):
        """ReconTrigrid::draw (rr_draw_trigrid) of the maps of the last preprocess; returns (rgba, depth)."""
        v = self._view(modelview, projection, width, height, shade_mode)
        self._vw, self._vh = int(width), int(height)
        rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
        self._ck(self.L.rr_draw_trigrid(self.h, C.byref(v), float(min_length), _f32(rgba), _f32(depth)))
        return rgba, depth

    def fill_colors(self, download=True):
        """ReconIntegration::fillColors on the last view; returns the filled rgba [h, w, 4] when download."""
        if not download:
            self._ck(self.L.rr_fill_colors(self.h, None))
            return None
        out = np.zeros((self._vh, self._vw, 4), np.float32)
        self._ck(self.L.rr_fill_colors(self.h, _f32(out)))
        return out

    def upload_view(self, rgba, depth):
        rgba = np.ascontiguousarray(rgba, np.float32)
        depth = np.ascontiguousarray(depth, np.float32)
        self._vh, self._vw = depth.shape
        self._ck(self.L.rr_upload_view(self.h, self._vw, self._vh, _f32(rgba), _f32(depth)))

    def _view(self, modelview, projection, width, height, shade_mode):
        v = View()
        v.modelview[:] = [float(x) for x in np.asarray(modelview, np.float32).reshape(16)]
        v.projection[:] = [float(x) for x in np.asarray(projection, np.float32).reshape(16)]
        v.viewport[:] = [0, 0, int(width), int(height)]
        v.shade_mode = int(shade_mode)
        return v

    def raymarch_partial(self, modelview, projection, width, height, d_records_ptr, shade_mode=0):
        """Slab march into a DEVICE record buffer (width*height*32 bytes), see rr_raymarch_partial."""
        v = self._view(modelview, projection, width, height, shade_mode)
        self._ck(self.L.rr_raymarch_partial(self.h, C.byref(v), d_records_ptr))

    def partial_keys(self, d_records_ptr, rank, d_keys_ptr):
        self._ck(self.L.rr_partial_keys(self.h, d_records_ptr, int(rank), d_keys_ptr))

    def partial_keep_winners(self, d_records_ptr, d_keys_min_ptr, rank):
        self._ck(self.L.rr_partial_keep_winners(self.h, d_records_ptr, d_keys_min_ptr, int(rank)))

    def composite(self, d_records_ptr, n_parts, width, height, download=True):
        self._vw, self._vh = int(width), int(height)
        if not download:
            self._ck(self.L.rr_composite(self.h, d_records_ptr, n_parts, width, height, None, None))
            return None
        rgba = np.zeros((height, width, 4), np.float32)
        depth = np.zeros((height, width), np.float32)
        self._ck(self.L.rr_composite(self.h, d_records_ptr, n_parts, width, height, _f32(rgba), _f32(depth)))
        return rgba, depth

    def view_export(self, width, height):
        """rr_view_export: 256 bytes of CUDA IPC handles of this context's view images (for another process' composite_peers)."""
        buf = (C.c_ubyte * 256)()
        self._ck(self.L.rr_view_export(self.h, int(width), int(height), C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def composite_peers(self, peer_handles, width, height, download=True):
        """rr_composite_peers: this context's view (marched last) composited with the views behind `peer_handles` (a list of
        view_export blobs of OTHER processes), in place; returns (rgba, depth) when download."""
        blob = b"".join(peer_handles)
        buf = (C.c_ubyte * max(1, len(blob))).from_buffer_copy(blob) if blob else None
        self._vw, self._vh = int(width), int(height)
        ptr = C.cast(buf, C.c_void_p) if buf is not None else None
        if not download:
            self._ck(self.L.rr_composite_peers(self.h, ptr, len(peer_handles), width, height, None, None))
            return None
        rgba = np.zeros((height, width, 4), np.float32)
        depth = np.zeros((height, width), np.float32)
        self._ck(self.L.rr_composite_peers(self.h, ptr, len(peer_handles), width, height, _f32(rgba), _f32(depth)))
        return rgba, depth

    def frame(self, filter_textures=True, use_processed_depth=True, refine=True, sync_bricks=False):
        """The per-frame sequence of kinect_client.cpp:572-600 after update(): clear, process, update bricks, integrate."""
        self.bricks_clear()
        self.preprocess(filter_textures, use_processed_depth, refine)
        r = self.bricks_update(sync=sync_bricks)
        self.integrate()
        return r

    def fuse_frame(self, filter_textures=True, use_processed_depth=True, refine=True):
        """frame() as ONE call (rr_fuse_frame): replays a captured CUDA graph when stage timing is off."""
        self._ck(self.L.rr_fuse_frame(self.h, int(filter_textures), int(use_processed_depth), int(refine)))

    def bricks_count(self):
        """(occupied bricks, occupied ratio) of the last bricks_update / fuse_frame; waits for the stream, no launch."""
        n = C.c_uint32()
        r = C.c_float()
        self._ck(self.L.rr_bricks_count(self.h, C.byref(n), C.byref(r)))
        return int(n.value), float(r.value)

    # read-back
    def synchronize(self):
        self._ck(self.L.rr_synchronize(self.h))

    def download_tsdf(self):
        r = self.volume_res()
        out = np.zeros((int(r[2]), int(r[1]), int(r[0])), np.float32)
        self._ck(self.L.rr_download_tsdf(self.h, _f32(out)))
        return out

    def download_weight(self):
        r = self.volume_res()
        out = np.zeros((int(r[2]), int(r[1]), int(r[0])), np.float32)
        self._ck(self.L.rr_download_weight(self.h, _f32(out)))
        return out

    def download_stage(self, name):
        ch = _STAGE_CH[name]
        shape = (self.N, self.H, self.W) + ((ch,) if ch > 1 else ())
        out = np.zeros(shape, np.float32)
        self._ck(self.L.rr_download_stage(self.h, STAGES[name], _f32(out)))
        return out

    def download_bricks(self):
        nb = self.brick_info()["num_bricks"]
        counters = np.zeros(nb, np.uint32)
        occ = np.zeros(nb, np.uint32)
        n = C.c_uint32()
        self._ck(self.L.rr_download_bricks(self.h, _u32(counters), _u32(occ), C.byref(n)))
        return counters, occ[: n.value].copy()

    def download_num_samples(self, width, height):
        out = np.zeros((height, width), np.float32)
        self._ck(self.L.rr_download_num_samples(self.h, _f32(out)))
        return out

    def download_hit_positions(self, width, height):
        out = np.zeros((height, width, 4), np.float32)
        self._ck(self.L.rr_download_hit_positions(self.h, _f32(out)))
        return out

    def extract_mesh_counts(self):
        """rr_extract_mesh alone: extracts the surface on the device and returns (vertices, triangles)."""
        nv, nt = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_extract_mesh(self.h, C.byref(nv), C.byref(nt)))
        self._mesh_n = (int(nv.value), int(nt.value))
        return self._mesh_n

    def download_mesh(self, nv, nt):
        """rr_download_mesh of the last extraction (nv, nt: its counts)."""
        pos, nrm = np.zeros((nv, 3), np.float32), np.zeros((nv, 3), np.float32)
        rgba, tri = np.zeros((nv, 4), np.float32), np.zeros((nt, 3), np.uint32)
        self._ck(self.L.rr_download_mesh(self.h, _f32(pos), _f32(nrm), _f32(rgba), _u32(tri)))
        return pos, nrm, rgba, tri

    def extract_mesh(self):
        """The fused surface as a mesh (rr_extract_mesh + rr_download_mesh): positions float32 [V, 3] (metres), normals
        float32 [V, 3], rgba float32 [V, 4] (alpha 1 quality-weighted colour, -1 fallback blend), triangles uint32 [T, 3]."""
        return self.download_mesh(*self.extract_mesh_counts())

    def sample_points(self, points, space="world"):
        """rr_sample_points at points [n, 3] ("world": metres, "volume": texture coordinates over the bbox): (values [n],
        normals [n, 3], rgba [n, 4]) float32 - numpy arrays, or torch tensors on the inputs' GPU when given CUDA tensors."""
        return _sample_points(lambda *a: self._ck(self.L.rr_sample_points(self.h, *a)), points, space)

    def cast_rays(self, origins, directions, space="world"):
        """rr_cast_rays along rays origins [n, 3] + t * directions [n, 3]: (positions [n, 3], normals [n, 3], rgba [n, 4],
        steps uint32 [n]; 0xFFFFFFFF and NaN positions where a ray hits nothing), as numpy arrays or CUDA tensors."""
        return _cast_rays(lambda *a: self._ck(self.L.rr_cast_rays(self.h, *a)), origins, directions, space)

    def extract_points_count(self, sensors=None):
        """rr_extract_points alone: extracts the point cloud of `sensors` (indices; None: all) and returns its size."""
        n = C.c_uint32()
        self._ck(self.L.rr_extract_points(self.h, _sensor_mask(sensors, self.N), C.byref(n)))
        return int(n.value)

    def download_points(self, n, device=False):
        """rr_download_points of the last extraction (n: its size), as numpy arrays or, with device, CUDA tensors on the
        context's GPU: (positions [n, 3], normals [n, 3], colors [n, 3], quality [n], pixels uint32 [n])."""
        dev = None
        if device:
            import torch
            dev = torch.device("cuda", self.device)
        outs, op = _query_outputs(dev, ((n, 3), "f4"), ((n, 3), "f4"), ((n, 3), "f4"), ((n,), "f4"), ((n,), "u4"))
        self._ck(self.L.rr_download_points(self.h, *op))
        return tuple(outs)

    def extract_points(self, sensors=None, device=False):
        """The pre-processed sensor points of the last preprocess as a point cloud (rr_extract_points + rr_download_points):
        positions float32 [n, 3] (metres), normals float32 [n, 3], colors float32 [n, 3] in [0, 1], quality float32 [n] and
        pixel ids uint32 [n] (sensor * W * H + y * W + x, ascending). sensors: iterable of sensor indices, default all;
        device: return torch tensors on the context's GPU instead of numpy arrays."""
        return self.download_points(self.extract_points_count(sensors), device)

    def label_parts_count(self):
        """rr_label_parts alone: labels the connected parts of the volume on the device and returns their count."""
        n = C.c_uint32()
        self._ck(self.L.rr_label_parts(self.h, C.byref(n)))
        return int(n.value)

    def download_parts(self, n):
        """rr_download_parts of the last labelling (n: its part count): (voxels uint32 [n], boxes int32 [n, 6], centroids
        float32 [n, 3])."""
        voxels, boxes, centroids = np.empty(n, np.uint32), np.empty((n, 6), np.int32), np.empty((n, 3), np.float32)
        self._ck(self.L.rr_download_parts(self.h, voxels.ctypes.data, boxes.ctypes.data, centroids.ctypes.data, None))
        return voxels, boxes, centroids

    def label_parts(self):
        """The 6-connected parts of the inside voxels (v > 0, finite), numbered by ascending smallest linear index
        (rr_label_parts + rr_download_parts): (voxels uint32 [P], boxes int32 [P, 6] = x0, x1, y0, y1, z0, z1 half-open
        voxel ranges, centroids float32 [P, 3] in metres)."""
        return self.download_parts(self.label_parts_count())

    def part_labels(self, device=False):
        """The labels of the last labelling: uint32 [Z, Y, X], the part of every inside voxel and 0xFFFFFFFF elsewhere; a
        numpy array, or with device a CUDA tensor on the context's GPU."""
        X, Y, Z = (int(v) for v in self.volume_res())
        dev = None
        if device:
            import torch
            dev = torch.device("cuda", self.device)
        (labels,), (ptr,) = _query_outputs(dev, ((Z, Y, X), "u4"))
        self._ck(self.L.rr_download_parts(self.h, None, None, None, ptr))
        return labels

    def mesh_parts(self, device=False, counts=None):
        """rr_download_mesh_parts: (vertex_parts uint32 [V], triangle_parts uint32 [T]) of the last mesh, which must come
        from the same volume state as the last labelling; numpy arrays, or with device CUDA tensors. counts: the mesh's
        (V, T), by default those of this object's last extract_mesh."""
        nv, nt = counts if counts is not None else getattr(self, "_mesh_n", (0, 0))
        dev = None
        if device:
            import torch
            dev = torch.device("cuda", self.device)
        outs, ptrs = _query_outputs(dev, ((nv,), "u4"), ((nt,), "u4"))
        self._ck(self.L.rr_download_mesh_parts(self.h, *ptrs))
        return tuple(outs)

    def track_parts_counts(self, min_voxels=1):
        """rr_track_parts alone: labels the volume, tracks its parts against the tracked labelling and returns (parts P,
        ended tracks E)."""
        n, e = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_track_parts(self.h, int(min_voxels), C.byref(n), C.byref(e)))
        return int(n.value), int(e.value)

    def download_part_tracks(self, n, e, device=False):
        """rr_download_part_tracks of the last tracking (n, e: its counts): (track_ids uint32 [n], prev_parts uint32 [n],
        overlaps uint32 [n], ended uint32 [e]), as numpy arrays or, with device, CUDA tensors on the context's GPU."""
        dev = None
        if device:
            import torch
            dev = torch.device("cuda", self.device)
        outs, op = _query_outputs(dev, ((n,), "u4"), ((n,), "u4"), ((n,), "u4"), ((e,), "u4"))
        self._ck(self.L.rr_download_part_tracks(self.h, *op))
        return tuple(outs)

    def track_parts(self, min_voxels=1, device=False):
        """The parts of the volume with persistent track ids (rr_track_parts + rr_download_parts + rr_download_part_tracks):
        (voxels, boxes, centroids) as label_parts, then track_ids, prev_parts and overlaps uint32 [P] (0xFFFFFFFF, 0xFFFFFFFF
        and 0 for parts below min_voxels voxels; prev_parts 0xFFFFFFFF and overlaps 0 for a new track) and ended uint32 [E],
        the ids of the tracks that ended. device: the four tracking arrays as CUDA tensors on the context's GPU."""
        n, e = self.track_parts_counts(min_voxels)
        return self.download_parts(n) + self.download_part_tracks(n, e, device)

    def reset_part_tracks(self):
        """rr_reset_part_tracks: forget the tracked labelling; the next track_parts starts ids at 0."""
        self._ck(self.L.rr_reset_part_tracks(self.h))

    def simplify_mesh_counts(self, cluster_voxels):
        """rr_simplify_mesh alone: simplifies the last mesh on the device and returns (vertices, triangles)."""
        nv, nt = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_simplify_mesh(self.h, int(cluster_voxels), C.byref(nv), C.byref(nt)))
        return int(nv.value), int(nt.value)

    def download_simplified_mesh(self, nv, nt, device=False):
        """rr_download_simplified_mesh of the last simplification (nv, nt: its counts), as numpy arrays or, with device,
        CUDA tensors on the context's GPU: (positions [nv, 3], normals [nv, 3], rgba [nv, 4], triangles uint32 [nt, 3],
        sources uint32 [nt])."""
        dev = None
        if device:
            import torch
            dev = torch.device("cuda", self.device)
        outs, op = _query_outputs(dev, ((nv, 3), "f4"), ((nv, 3), "f4"), ((nv, 4), "f4"), ((nt, 3), "u4"), ((nt,), "u4"))
        self._ck(self.L.rr_download_simplified_mesh(self.h, *op))
        return tuple(outs)

    def simplify_mesh(self, cluster_voxels, device=False):
        """The last mesh simplified by vertex clustering with clusters of cluster_voxels voxels per side (rr_simplify_mesh +
        rr_download_simplified_mesh): positions float32 [V', 3] (the clusters' mean positions, metres), normals float32
        [V', 3] and rgba float32 [V', 4] (rr_sample_points at them), triangles uint32 [T', 3] and sources uint32 [T'] (each
        triangle's source triangle in the last mesh); numpy arrays, or with device CUDA tensors."""
        return self.download_simplified_mesh(*self.simplify_mesh_counts(cluster_voxels), device=device)

    def set_timing(self, level=1):
        self._ck(self.L.rr_set_timing(self.h, int(level)))

    def stage_stats(self, name):
        ms = C.c_float()
        n = C.c_uint32()
        self._ck(self.L.rr_get_stage_stats(self.h, name.encode(), C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def stage_ms(self, name):
        ms = C.c_float()
        self._ck(self.L.rr_get_stage_ms(self.h, name.encode(), C.byref(ms)))
        return float(ms.value)

    def integrator_info(self):
        """rr_integrator_info as a dict (which integrator bricks mode runs, staged geometry, device flags)."""
        out = np.zeros(16, np.uint32)
        self._ck(self.L.rr_integrator_info(self.h, _u32(out)))
        keys = ("staged", "tile", "box_x", "box_y", "box_z", "ychunk", "zchunk", "n_ychunks", "n_zchunks", "oversize_pairs",
                "smem_bytes", "consumer_warps", "fill_warps", "flags", "slots", "slot_bytes")
        return {k: int(v) for k, v in zip(keys, out)}

    def integrator_last(self):
        """rr_integrator_last as a dict: the kernel the last integrate launched (path name), its sensors, voxel format, CTA
        threads (consumer warps for the staged kernel), repair bits (1: stale staged item lists, 2: gather packed late) and the
        clear it did ("none", "full" or "incremental")."""
        out = np.zeros(8, np.uint32)
        self._ck(self.L.rr_integrator_last(self.h, _u32(out)))
        return dict(path=INTEGRATE_PATHS[int(out[0])], sensors=int(out[1]), voxel_mode=int(out[2]), threads=int(out[3]), repairs=int(out[4]),
                    clear=INTEGRATE_CLEARS[int(out[5])])

    def integrator_cleared(self):
        """rr_integrator_cleared: bricks the last integrate's incremental clear reset (0 unless it cleared incrementally)."""
        out = np.zeros(1, np.uint32)
        self._ck(self.L.rr_integrator_cleared(self.h, _u32(out)))
        return int(out[0])

    def integrator_profile(self):
        """rr_integrator_profile: cycle counters of the staged integrator's roles (stage_debug bit 7), reset on read."""
        out = np.zeros(16, np.uint64)
        self._ck(self.L.rr_integrator_profile(self.h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        keys = ("consumer_wait", "consumer_work", "consumer_idle_items", "active_sensor_items", "producer_meta", "producer_wait_empty", "producer_copy",
                "staged_items", "direct_items", "clear_warps", "clear_helpers", "cta_max", "warp_life_sum", "tile_need_max", "need_le30_items", "need_le36_items")
        return {k: int(v) for k, v in zip(keys, out) if not k.startswith("_")}

    def launch_count(self):
        return int(self.L.rr_launch_count(self.h))

    def stream(self):
        return self.L.rr_stream(self.h)


class Group:
    """Thin object wrapper of an rr_group: one process, one rr_ctx per device, z-slabs (include/rgbd_recon_b200.h)."""

    def __init__(self, devices, N, W, H, CW, CH):
        self.L = lib()
        self.h = C.c_void_p()
        self.N, self.W, self.H, self.CW, self.CH = N, W, H, CW, CH
        dev = np.ascontiguousarray(devices, np.int32)
        rc = self.L.rr_group_create(C.byref(self.h), dev.ctypes.data_as(C.POINTER(C.c_int32)), len(dev), N, W, H, CW, CH)
        if rc != 0:
            raise RRError(f"rr_group_create failed with status {rc}")
        self.n = len(dev)
        self.devices = [int(d) for d in dev]

    def close(self):
        if self.h:
            self.L.rr_group_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise RRError(f"status {rc}: {self.L.rr_group_last_error(self.h).decode()}")

    def member(self, i):
        """The i-th member as a (non-owning) Fusion, for queries and read-backs."""
        fu = Fusion.__new__(Fusion)
        fu.L, fu.h = self.L, C.c_void_p(self.L.rr_group_member(self.h, i))
        fu.N, fu.W, fu.H, fu.CW, fu.CH = self.N, self.W, self.H, self.CW, self.CH
        fu.device = self.devices[i]
        fu.close = lambda: None
        return fu

    def set_bbox(self, bmin, bmax):
        bmin = np.ascontiguousarray(bmin, np.float32)
        bmax = np.ascontiguousarray(bmax, np.float32)
        self._ck(self.L.rr_group_set_bbox(self.h, _f32(bmin), _f32(bmax)))

    def calib_upload(self, sensor, cv_xyz, cv_uv, depth_limits=(0.5, 4.5)):
        Z, Y, X, _ = cv_xyz.shape
        xyz = np.ascontiguousarray(cv_xyz, np.float32)
        uv = np.ascontiguousarray(cv_uv, np.float32)
        res = np.array([X, Y, Z], np.uint32)
        dl = np.array(depth_limits, np.float32)
        self._ck(self.L.rr_group_calib_upload(self.h, sensor, _f32(xyz), _f32(uv), _u32(res), _f32(dl)))

    def calib_upload_inv(self, sensor, inv):
        Z, Y, X, _ = inv.shape
        a = np.ascontiguousarray(inv, np.float32)
        res = np.array([X, Y, Z], np.uint32)
        self._ck(self.L.rr_group_calib_upload_inv(self.h, sensor, _f32(a), _u32(res)))

    def configure(self, limit=0.01, voxel_size=0.01, brick_size=0.1, min_voxels=10, use_bricks=True, skip_space=True, store_weight=False):
        cfg = Config(limit, voxel_size, brick_size, min_voxels, int(use_bricks), int(skip_space), int(store_weight))
        self._ck(self.L.rr_group_configure(self.h, C.byref(cfg)))

    def set_frame_format(self, dxt1_color=False, depth8=False, near_far=None, dxt5_color=False):
        nf = np.ascontiguousarray(near_far, np.float32) if near_far is not None else None
        self._ck(self.L.rr_group_set_frame_format(self.h, 5 if dxt5_color else (1 if dxt1_color else 0), 1 if depth8 else 0,
                                                  _f32(nf) if nf is not None else None))

    def set_slabs(self, bounds):
        b = np.ascontiguousarray(bounds, np.uint32)
        assert len(b) == self.n + 1
        self._ck(self.L.rr_group_set_slabs(self.h, _u32(b)))

    def slabs(self):
        b = np.zeros(self.n + 1, np.uint32)
        self._ck(self.L.rr_group_get_slabs(self.h, _u32(b)))
        return [int(v) for v in b]

    def balance_slabs(self, compute_to_fill=0.0):
        self._ck(self.L.rr_group_balance_slabs(self.h, float(compute_to_fill)))

    def upload_frames(self, color, depth):
        color = np.ascontiguousarray(color) if color is not None else None
        depth = np.ascontiguousarray(depth)
        self._ck(self.L.rr_group_upload_frames(self.h, color.ctypes.data if color is not None else None, color.nbytes if color is not None else 0,
                                               depth.ctypes.data, depth.nbytes))

    def stage_frames_ptr(self, color_ptr, color_bytes, depth_ptr, depth_bytes):
        self._ck(self.L.rr_group_stage_frames(self.h, color_ptr, color_bytes, depth_ptr, depth_bytes))

    def swap_frames(self):
        self._ck(self.L.rr_group_swap_frames(self.h))

    def stage_sync(self):
        self._ck(self.L.rr_group_stage_sync(self.h))

    def frame(self, filter_textures=True, use_processed_depth=True, refine=True):
        """The per-frame sequence call by call (kinect_client.cpp:572-600) on every member; returns (occupied, ratio)."""
        self.bricks_clear()
        self.preprocess(filter_textures, use_processed_depth, refine)
        r = self.bricks_update()
        self.integrate()
        return r

    def bricks_clear(self):
        self._ck(self.L.rr_group_bricks_clear(self.h))

    def preprocess(self, filter_textures=True, use_processed_depth=True, refine=True):
        self._ck(self.L.rr_group_preprocess(self.h, int(filter_textures), int(use_processed_depth), int(refine)))

    def bricks_update(self):
        n, r = C.c_uint32(), C.c_float()
        self._ck(self.L.rr_group_bricks_update(self.h, C.byref(n), C.byref(r)))
        return int(n.value), float(r.value)

    def integrate(self):
        self._ck(self.L.rr_group_integrate(self.h))

    def fuse_frame(self, filter_textures=True, use_processed_depth=True, refine=True):
        self._ck(self.L.rr_group_fuse_frame(self.h, int(filter_textures), int(use_processed_depth), int(refine)))

    def bricks_count(self):
        n, r = C.c_uint32(), C.c_float()
        self._ck(self.L.rr_group_bricks_count(self.h, C.byref(n), C.byref(r)))
        return int(n.value), float(r.value)

    def raymarch(self, modelview, projection, width, height, shade_mode=0, download=True):
        v = View()
        v.modelview[:] = [float(x) for x in np.asarray(modelview, np.float32).reshape(16)]
        v.projection[:] = [float(x) for x in np.asarray(projection, np.float32).reshape(16)]
        v.viewport[:] = [0, 0, int(width), int(height)]
        v.shade_mode = int(shade_mode)
        self._vw, self._vh = int(width), int(height)
        if not download:
            self._ck(self.L.rr_group_raymarch(self.h, C.byref(v), None, None))
            return None
        rgba = np.zeros((height, width, 4), np.float32)
        depth = np.zeros((height, width), np.float32)
        self._ck(self.L.rr_group_raymarch(self.h, C.byref(v), _f32(rgba), _f32(depth)))
        return rgba, depth

    def fill_colors(self, download=True):
        if not download:
            self._ck(self.L.rr_group_fill_colors(self.h, None))
            return None
        out = np.zeros((self._vh, self._vw, 4), np.float32)
        self._ck(self.L.rr_group_fill_colors(self.h, _f32(out)))
        return out

    def synchronize(self):
        self._ck(self.L.rr_group_synchronize(self.h))

    def download_tsdf(self):
        r = self.member(0).volume_res()
        out = np.zeros((int(r[2]), int(r[1]), int(r[0])), np.float32)
        self._ck(self.L.rr_group_download_tsdf(self.h, _f32(out)))
        return out

    def extract_mesh_counts(self):
        """rr_group_extract_mesh: the whole volume's surface, extracted on member 0; returns (vertices, triangles)."""
        nv, nt = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_group_extract_mesh(self.h, C.byref(nv), C.byref(nt)))
        self._mesh_n = (int(nv.value), int(nt.value))
        return self._mesh_n

    def extract_mesh(self):
        """As Fusion.extract_mesh, equal to a single context's bit for bit: (positions, normals, rgba, triangles)."""
        return self.member(0).download_mesh(*self.extract_mesh_counts())

    def extract_points(self, sensors=None, device=False):
        """As Fusion.extract_points (rr_group_extract_points on member 0; CUDA tensors on member 0's GPU), equal to a single
        context's bit for bit."""
        n = C.c_uint32()
        self._ck(self.L.rr_group_extract_points(self.h, _sensor_mask(sensors, self.N), C.byref(n)))
        return self.member(0).download_points(int(n.value), device)

    def label_parts(self):
        """As Fusion.label_parts (rr_group_label_parts: the whole volume, labelled on member 0), equal to a single context
        bit for bit: (voxels, boxes, centroids)."""
        n = C.c_uint32()
        self._ck(self.L.rr_group_label_parts(self.h, C.byref(n)))
        return self.member(0).download_parts(int(n.value))

    def part_labels(self, device=False):
        """As Fusion.part_labels, from member 0 (CUDA tensors on member 0's GPU)."""
        return self.member(0).part_labels(device)

    def mesh_parts(self, device=False):
        """As Fusion.mesh_parts, for the group's last extract_mesh and label_parts (member 0)."""
        return self.member(0).mesh_parts(device, getattr(self, "_mesh_n", (0, 0)))

    def track_parts(self, min_voxels=1, device=False):
        """As Fusion.track_parts (rr_group_track_parts: the whole volume, labelled and tracked on member 0), equal to a
        single context over the same sequence of frame sets."""
        n, e = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_group_track_parts(self.h, int(min_voxels), C.byref(n), C.byref(e)))
        m0 = self.member(0)
        return m0.download_parts(int(n.value)) + m0.download_part_tracks(int(n.value), int(e.value), device)

    def reset_part_tracks(self):
        """rr_reset_part_tracks on member 0, which holds the group's tracking state."""
        self.member(0).reset_part_tracks()

    def simplify_mesh(self, cluster_voxels, device=False):
        """As Fusion.simplify_mesh (rr_group_simplify_mesh on member 0 after the group's extract_mesh; CUDA tensors on member
        0's GPU), equal to a single context's bit for bit: (positions, normals, rgba, triangles, sources)."""
        nv, nt = C.c_uint32(), C.c_uint32()
        self._ck(self.L.rr_group_simplify_mesh(self.h, int(cluster_voxels), C.byref(nv), C.byref(nt)))
        return self.member(0).download_simplified_mesh(int(nv.value), int(nt.value), device)

    def sample_points(self, points, space="world"):
        """As Fusion.sample_points (CUDA tensors on member 0's GPU), equal to a single context's bit for bit."""
        return _sample_points(lambda *a: self._ck(self.L.rr_group_sample_points(self.h, *a)), points, space)

    def cast_rays(self, origins, directions, space="world"):
        """As Fusion.cast_rays (CUDA tensors on member 0's GPU), equal to a single context's bit for bit."""
        return _cast_rays(lambda *a: self._ck(self.L.rr_group_cast_rays(self.h, *a)), origins, directions, space)


def load_scene(fu: "Fusion", scene, inv=None):
    """Upload a synth.Scene (bbox, forward volumes, optional inverse volumes) into a context."""
    fu.set_bbox(scene.bbox_min, scene.bbox_max)
    for i in range(scene.N):
        fu.calib_upload(i, scene.cv_xyz[i], scene.cv_uv[i])
        if inv is not None:
            fu.calib_upload_inv(i, inv[i])
