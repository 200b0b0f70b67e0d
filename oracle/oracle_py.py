"""ORACLE binding (test infrastructure, NOT product code).

ctypes wrapper over oracle/librr_oracle.so, the scalar CPU restatement of the reference's volumetric-fusion path.
Import this only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")

# the volume block that ro_extract_mesh, ro_sample_points and ro_cast_rays start with (VolumeArgs)
_VOLUME_ARGS = [f32p, u32p, C.c_float, C.c_int, C.c_void_p, i32p, C.c_void_p, i32p, C.c_void_p, C.c_int, C.c_int,
                C.c_void_p, C.c_void_p, C.c_int, C.c_int, f32p, f32p]


def build():
    """make tracks the sources: a library older than any of them is rebuilt, a current one is left as it is."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "librr_oracle.so"])
    return os.path.join(_HERE, "librr_oracle.so")


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(build())
    L.ro_set_threads.argtypes = [C.c_int]
    L.ro_get_max_threads.restype = C.c_int
    for n in ("ro_kat_log2", "ro_kat_exp2"):
        getattr(L, n).argtypes = [C.c_float]
        getattr(L, n).restype = C.c_float
    L.ro_kat_pow.argtypes = [C.c_float, C.c_float]
    L.ro_kat_pow.restype = C.c_float
    L.ro_kat_tex3d.argtypes = [f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, f32p]
    L.ro_kat_tex2d.argtypes = [f32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int]
    L.ro_kat_tex2d.restype = C.c_float
    L.ro_kat_rgb_to_lab.argtypes = [f32p, f32p]
    L.ro_pre_morph.argtypes = [f32p, C.c_int, C.c_int, f32p]
    L.ro_pre_depth.argtypes = [f32p, C.c_int, C.c_int, f32p, f32p, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int,
                               f32p, f32p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, f32p, f32p]
    L.ro_pre_boundary.argtypes = [f32p, f32p, C.c_int, C.c_int, C.c_int, f32p, f32p]
    L.ro_pre_normal.argtypes = [f32p, C.c_int, C.c_int, f32p, C.c_int, C.c_int, C.c_int, f32p, C.c_float, u32p, C.c_uint32, u32p, f32p]
    L.ro_pre_quality.argtypes = [f32p, f32p, C.c_int, C.c_int, f32p, C.c_int, C.c_int, C.c_int, f32p, f32p]
    L.ro_volume_res.argtypes = [f32p, f32p, C.c_float, u32p]
    L.ro_adjust_brick_size.argtypes = [C.c_float, C.c_float]
    L.ro_adjust_brick_size.restype = C.c_float
    L.ro_divide_box.argtypes = [f32p, f32p, C.c_float, u32p, u32p, C.c_void_p]
    L.ro_divide_box.restype = C.c_uint32
    L.ro_divide_box_args.argtypes = [f32p, f32p, C.c_float, u32p, C.c_void_p, C.c_void_p]
    L.ro_divide_box_args.restype = C.c_uint32
    L.ro_occupied_bricks.argtypes = [u32p, C.c_uint32, C.c_uint32, u32p]
    L.ro_occupied_bricks.restype = C.c_uint32
    L.ro_integrate.argtypes = [C.c_int, f32p, i32p, f32p, f32p, f32p, C.c_int, C.c_int, C.c_float, u32p, C.c_int,
                               i32p, u32p, C.c_uint32, f32p, C.c_void_p]
    L.ro_frustum.argtypes = [f32p, C.c_int, C.c_int, C.c_int, f32p, f32p]
    L.ro_frustum_inside.argtypes = [f32p, f32p]
    L.ro_frustum_inside.restype = C.c_int
    L.ro_calib_invert.argtypes = [f32p, C.c_int, C.c_int, C.c_int, f32p, f32p, u32p, f32p, C.c_void_p, C.c_int]
    L.ro_raymarch_uniforms.argtypes = [f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p]
    L.ro_raymarch.argtypes = [f32p, u32p, C.c_float, C.c_int, f32p, i32p, f32p, i32p, u8p, C.c_int, C.c_int, f32p, f32p, C.c_int, C.c_int,
                              f32p, f32p, f32p, f32p, C.c_int, C.c_int, C.c_int, C.c_int, u32p, C.c_uint32, u32p, C.c_float,
                              f32p, f32p, f32p, f32p]
    L.ro_raymarch_rays.argtypes = [f32p, f32p, f32p, f32p, C.c_int, C.c_int, C.c_float, f32p, u8p]
    L.ro_decode_dxt1.argtypes = [u8p, C.c_int, C.c_int, u8p]
    L.ro_decode_dxt5.argtypes = [u8p, C.c_int, C.c_int, u8p]
    L.ro_depth8_to_float.argtypes = [u8p, C.c_size_t, f32p]
    L.ro_fill_num_lods.argtypes = [C.c_int, C.c_int]
    L.ro_fill_num_lods.restype = C.c_int
    L.ro_fill_colors.argtypes = [f32p, f32p, C.c_int, C.c_int, f32p, C.c_void_p, C.c_void_p]
    L.ro_mesh_case_table.argtypes = [i32p, i32p]
    L.ro_mesh_case_table.restype = C.c_int
    L.ro_extract_mesh.argtypes = _VOLUME_ARGS + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ro_sample_points.argtypes = _VOLUME_ARGS + [C.c_int, f32p, C.c_uint32, f32p, f32p, f32p]
    L.ro_cast_rays.argtypes = _VOLUME_ARGS + [C.c_int, C.c_void_p, C.c_uint32, u32p, C.c_float, C.c_int, f32p, f32p, C.c_uint32,
                                              f32p, f32p, f32p, u32p]
    L.ro_extract_points.argtypes = [C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, u8p, C.c_int, C.c_int, f32p, f32p, i32p, f32p, f32p,
                                    C.c_uint32, C.POINTER(C.c_uint32), f32p, f32p, f32p, f32p, u32p]
    _LIB = L
    return L


class VolumeArgs:
    """The volume block of ro_extract_mesh, ro_sample_points and ro_cast_rays (`args`): tsdf float32 [Z][Y][X] (res = (X, Y, Z)),
    and optionally the inverse volumes, scene (cv_uv, colour) and pre-processed stage images blendColors reads (all three or
    none). Holds the arrays the raw pointers of `args` point into."""

    def __init__(self, tsdf, res, limit, inv, scene, pre, bbox_min, bbox_max):
        self.keep = []
        tsdf = np.ascontiguousarray(tsdf, np.float32)
        bmin = np.ascontiguousarray(bbox_min, np.float32)
        bmax = np.ascontiguousarray(bbox_max, np.float32)
        head = (tsdf, np.ascontiguousarray(res, np.uint32), np.float32(limit))
        if inv is not None:
            N, IZ, IY, IX, _ = inv.shape
            X, Y, Z = scene.cv_res
            _, H, W = pre["quality"].shape
            self.args = head + (N, self._ptr(inv, np.float32), np.array([IX, IY, IZ], np.int32), self._ptr(scene.cv_uv, np.float32),
                                np.array([X, Y, Z], np.int32), self._ptr(scene.color, np.uint8), scene.CW, scene.CH,
                                self._ptr(pre["depth_b"], np.float32), self._ptr(pre["quality"], np.float32), W, H, bmin, bmax)
        else:
            z3 = np.zeros(3, np.int32)
            self.args = head + (0, None, z3, None, z3, None, 0, 0, None, None, 0, 0, bmin, bmax)

    def _ptr(self, a, dt):
        a = np.ascontiguousarray(a, dt)
        self.keep.append(a)
        return a.ctypes.data


def set_threads(n):
    lib().ro_set_threads(int(n))


def max_threads():
    return lib().ro_get_max_threads()


# ---------------------------------------------------------------------------------------------- brick grid

def brick_grid(bbox_min, bbox_max, voxel_size, brick_size_req):
    """setVoxelSize + setBrickSize + divideBox. Returns dict(res, brick_size, res_bricks, ranges[nb,6])."""
    L = lib()
    bmin = np.ascontiguousarray(bbox_min, np.float32)
    bmax = np.ascontiguousarray(bbox_max, np.float32)
    res = np.zeros(3, np.uint32)
    L.ro_volume_res(bmin, bmax, np.float32(voxel_size), res)
    bs = L.ro_adjust_brick_size(np.float32(voxel_size), np.float32(brick_size_req))
    rb = np.zeros(3, np.uint32)
    nb = L.ro_divide_box(bmin, bmax, bs, res, rb, None)
    ranges = np.zeros((nb, 6), np.int32)
    L.ro_divide_box(bmin, bmax, bs, res, rb, ranges.ctypes.data)
    return dict(res=res, brick_size=np.float32(bs), res_bricks=rb, ranges=ranges, num_bricks=int(nb))


def divide_box_args(bbox_min, bbox_max, brick_size, res, want_raw=False):
    """(pos_n, size_n) per brick as divideBox hands them to containedVoxels; optionally the unclamped loop bounds."""
    L = lib()
    bmin = np.ascontiguousarray(bbox_min, np.float32)
    bmax = np.ascontiguousarray(bbox_max, np.float32)
    res = np.ascontiguousarray(res, np.uint32)
    n = L.ro_divide_box_args(bmin, bmax, np.float32(brick_size), res, None, None)
    args = np.zeros((n, 6), np.float32)
    raw = np.zeros((n, 6), np.int32)
    L.ro_divide_box_args(bmin, bmax, np.float32(brick_size), res, args.ctypes.data, raw.ctypes.data)
    return (args, raw) if want_raw else args


def frustum(cv_xyz_one):
    Z, Y, X, _ = cv_xyz_one.shape
    planes = np.zeros((6, 4), np.float32)
    cam = np.zeros(3, np.float32)
    lib().ro_frustum(np.ascontiguousarray(cv_xyz_one), X, Y, Z, planes, cam)
    return planes, cam


def calib_invert(cv_xyz_one, bbox_min, bbox_max, out_res, want_neighbours=False, brute=False):
    Z, Y, X, _ = cv_xyz_one.shape
    ox, oy, oz = [int(v) for v in out_res]
    out = np.zeros((oz, oy, ox, 4), np.float32)
    neigh = np.zeros((oz, oy, ox, 8), np.uint32) if want_neighbours else None
    lib().ro_calib_invert(np.ascontiguousarray(cv_xyz_one), X, Y, Z, np.ascontiguousarray(bbox_min, np.float32),
                          np.ascontiguousarray(bbox_max, np.float32), np.array([ox, oy, oz], np.uint32), out,
                          neigh.ctypes.data if neigh is not None else None, int(brute))
    return (out, neigh) if want_neighbours else out


# ---------------------------------------------------------------------------------------------- frame

def decode_dxt5(blocks, W, H):
    """DXT5 block bytes (16 per 4x4 block) -> uint8 [H][W][3]; the alpha half of a block is not sampled downstream."""
    out = np.zeros((H, W, 3), np.uint8)
    lib().ro_decode_dxt5(np.ascontiguousarray(blocks, np.uint8), W, H, out)
    return out


def decode_dxt1(blocks, W, H):
    """DXT1 block bytes -> uint8 [H][W][3] (what the GL sampler returns as .rgb * 255)."""
    out = np.zeros((H, W, 3), np.uint8)
    lib().ro_decode_dxt1(np.ascontiguousarray(blocks, np.uint8), W, H, out)
    return out


def depth8_to_float(d8):
    d8 = np.ascontiguousarray(d8, np.uint8)
    out = np.zeros(d8.shape, np.float32)
    lib().ro_depth8_to_float(d8.reshape(-1), d8.size, out.reshape(-1))
    return out


def preprocess(scene, grid, camera_positions, filter_textures=True, use_processed_depth=True, refine=True, compress=None):
    """NetKinectArray::processTextures for all layers (+ ReconIntegration::clearOccupiedBricks before it).
    compress: None, or per sensor (near, far) when scene.depth holds the normalised 8-bit values byte/255
    (NetKinectArray.cpp:345-351: scale = far - near, scaled_near = scale / 255)."""
    L = lib()
    N, H, W = scene.depth.shape
    X, Y, Z = scene.cv_res
    out = dict(
        morph=np.zeros((N, H, W), np.float32), depth=np.zeros((N, H, W, 2), np.float32),
        lab=np.zeros((N, H, W, 3), np.float32), depth_b=np.zeros((N, H, W, 2), np.float32),
        sil=np.zeros((N, H, W), np.float32), normal=np.zeros((N, H, W, 3), np.float32),
        quality=np.zeros((N, H, W), np.float32), bricks=np.zeros(grid["num_bricks"], np.uint32))
    bmin = np.ascontiguousarray(scene.bbox_min, np.float32)
    bmax = np.ascontiguousarray(scene.bbox_max, np.float32)
    for i in range(N):
        raw = np.ascontiguousarray(scene.depth[i])
        L.ro_pre_morph(raw, W, H, out["morph"][i])
        src = out["morph"][i] if use_processed_depth else raw
        if compress is None:
            cz, scale, near, snear = 0, 0.0, 0.0, 0.0
        else:
            near = np.float32(compress[i][0])
            scale = np.float32(compress[i][1]) - near
            cz, snear = 1, scale / np.float32(255.0)
        L.ro_pre_depth(src, W, H, scene.cv_xyz[i], scene.cv_uv[i], X, Y, Z, scene.color[i], scene.CW, scene.CH, bmin, bmax,
                       0.5, 4.5, int(filter_textures), cz, float(scale), float(near), float(snear), out["depth"][i], out["lab"][i])
        L.ro_pre_boundary(out["depth"][i], out["lab"][i], W, H, int(refine), out["depth_b"][i], out["sil"][i])
        L.ro_pre_normal(out["depth_b"][i], W, H, scene.cv_xyz[i], X, Y, Z, bmin, grid["brick_size"], grid["res_bricks"],
                        grid["num_bricks"], out["bricks"], out["normal"][i])
        L.ro_pre_quality(out["depth_b"][i], out["normal"][i], W, H, scene.cv_xyz[i], X, Y, Z,
                         np.ascontiguousarray(camera_positions[i], np.float32), out["quality"][i])
    return out


def occupied_bricks(counters, min_voxels=10):
    occ = np.zeros(len(counters), np.uint32)
    n = lib().ro_occupied_bricks(np.ascontiguousarray(counters, np.uint32), len(counters), int(min_voxels), occ)
    return occ[:n].copy()


def integrate(inv, pre, grid, limit, use_bricks, occupied, want_weight=False):
    """ReconIntegration::integrate. inv: [N][IZ][IY][IX][4]."""
    N, IZ, IY, IX, _ = inv.shape
    _, H, W = pre["sil"].shape
    res = grid["res"]
    tsdf = np.zeros((int(res[2]), int(res[1]), int(res[0])), np.float32)
    weight = np.zeros_like(tsdf) if want_weight else None
    occ = np.ascontiguousarray(occupied, np.uint32) if len(occupied) else np.zeros(1, np.uint32)
    lib().ro_integrate(N, np.ascontiguousarray(inv), np.array([IX, IY, IZ], np.int32), pre["sil"], pre["depth_b"], pre["quality"],
                       W, H, np.float32(limit), res, int(use_bricks), grid["ranges"], occ, len(occupied), tsdf,
                       weight.ctypes.data if weight is not None else None)
    return (tsdf, weight) if want_weight else tsdf


def raymarch(tsdf, limit, inv, scene, pre, grid, occupied, modelview, projection, width, height, shade_mode=0, skip_space=True):
    """ReconIntegration::draw (+ drawDepthLimits). Returns dict(rgba[h,w,4], depth[h,w], samples[h,w], pos[h,w,3])."""
    N, IZ, IY, IX, _ = inv.shape
    X, Y, Z = scene.cv_res
    _, H, W = pre["quality"].shape
    res = np.array([tsdf.shape[2], tsdf.shape[1], tsdf.shape[0]], np.uint32)
    out = dict(rgba=np.zeros((height, width, 4), np.float32), depth=np.zeros((height, width), np.float32),
               samples=np.zeros((height, width), np.float32), pos=np.zeros((height, width, 3), np.float32))
    occ = np.ascontiguousarray(occupied, np.uint32) if len(occupied) else np.zeros(1, np.uint32)
    lib().ro_raymarch(np.ascontiguousarray(tsdf), res, np.float32(limit), N, np.ascontiguousarray(inv), np.array([IX, IY, IZ], np.int32),
                      np.ascontiguousarray(scene.cv_uv), np.array([X, Y, Z], np.int32), np.ascontiguousarray(scene.color), scene.CW, scene.CH,
                      pre["depth_b"], pre["quality"], W, H, np.ascontiguousarray(scene.bbox_min, np.float32),
                      np.ascontiguousarray(scene.bbox_max, np.float32), np.ascontiguousarray(modelview, np.float32).reshape(16),
                      np.ascontiguousarray(projection, np.float32).reshape(16), int(width), int(height), int(shade_mode), int(skip_space),
                      occ, len(occupied), grid["res_bricks"], grid["brick_size"], out["rgba"], out["depth"], out["samples"], out["pos"])
    return out


def draw_points(scene, pre, modelview, projection, width, height, shade_mode=0):
    """ReconPoints::draw on the pre-processed maps of `pre` (depth_b, normal). Returns (rgba [h,w,4], depth [h,w])."""
    L = lib()
    if not hasattr(L, "_points"):
        L.ro_draw_points.argtypes = [C.c_int, C.c_int, C.c_int, f32p, f32p, u8p, C.c_int, C.c_int, f32p, f32p, i32p, f32p, f32p, f32p, f32p,
                                     C.c_int, C.c_int, C.c_int, f32p, f32p]
        L.ro_draw_calibs.argtypes = [f32p, u32p, i32p, C.c_float, f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p]
        L._points = True
    X, Y, Z = scene.cv_res
    N, H, W = pre["quality"].shape
    rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
    L.ro_draw_points(N, W, H, np.ascontiguousarray(pre["depth_b"], np.float32), np.ascontiguousarray(pre["normal"], np.float32),
                     np.ascontiguousarray(scene.color), scene.CW, scene.CH, np.ascontiguousarray(scene.cv_xyz, np.float32),
                     np.ascontiguousarray(scene.cv_uv, np.float32), np.array([X, Y, Z], np.int32), np.ascontiguousarray(scene.bbox_min, np.float32),
                     np.ascontiguousarray(scene.bbox_max, np.float32), np.ascontiguousarray(modelview, np.float32).reshape(16),
                     np.ascontiguousarray(projection, np.float32).reshape(16), int(width), int(height), int(shade_mode), rgba, depth)
    return rgba, depth


def draw_calibs(tsdf, inv_res, limit, bbox_min, bbox_max, modelview, projection, width, height):
    """ReconCalibs::draw: the voxel centres of the inverse-volume grid (inv_res = (IX, IY, IZ)) coloured by the TSDF there."""
    draw_points.__doc__  # (argtypes are set by the first draw_points / below)
    L = lib()
    if not hasattr(L, "_points"):
        L.ro_draw_points.argtypes = [C.c_int, C.c_int, C.c_int, f32p, f32p, u8p, C.c_int, C.c_int, f32p, f32p, i32p, f32p, f32p, f32p, f32p,
                                     C.c_int, C.c_int, C.c_int, f32p, f32p]
        L.ro_draw_calibs.argtypes = [f32p, u32p, i32p, C.c_float, f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p]
        L._points = True
    res = np.array([tsdf.shape[2], tsdf.shape[1], tsdf.shape[0]], np.uint32)
    rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
    L.ro_draw_calibs(np.ascontiguousarray(tsdf, np.float32), res, np.array(inv_res, np.int32), np.float32(limit),
                     np.ascontiguousarray(bbox_min, np.float32), np.ascontiguousarray(bbox_max, np.float32),
                     np.ascontiguousarray(modelview, np.float32).reshape(16), np.ascontiguousarray(projection, np.float32).reshape(16),
                     int(width), int(height), rgba, depth)
    return rgba, depth


def draw_trigrid(scene, pre, modelview, projection, width, height, shade_mode=0, min_length=0.0125, epsilon=0.075, want_passes=False):
    """ReconTrigrid::draw on the pre-processed maps of `pre` (depth_b, quality). Returns (rgba [h,w,4], depth [h,w]) and, with
    want_passes, also the accumulation target of pass 2 and the depth buffer of pass 1."""
    L = lib()
    L.ro_draw_trigrid.argtypes = [C.c_int, C.c_int, C.c_int, f32p, f32p, u8p, C.c_int, C.c_int, f32p, f32p, i32p, f32p, f32p, f32p, f32p,
                                  C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, f32p, f32p, C.c_void_p, C.c_void_p]
    X, Y, Z = scene.cv_res
    N, H, W = pre["quality"].shape
    rgba, depth = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
    accum, depth1 = np.zeros((height, width, 4), np.float32), np.zeros((height, width), np.float32)
    L.ro_draw_trigrid(N, W, H, np.ascontiguousarray(pre["depth_b"], np.float32), np.ascontiguousarray(pre["quality"], np.float32),
                      np.ascontiguousarray(scene.color), scene.CW, scene.CH, np.ascontiguousarray(scene.cv_xyz, np.float32),
                      np.ascontiguousarray(scene.cv_uv, np.float32), np.array([X, Y, Z], np.int32), np.ascontiguousarray(scene.bbox_min, np.float32),
                      np.ascontiguousarray(scene.bbox_max, np.float32), np.ascontiguousarray(modelview, np.float32).reshape(16),
                      np.ascontiguousarray(projection, np.float32).reshape(16), int(width), int(height), int(shade_mode),
                      float(min_length), float(epsilon), rgba, depth, accum.ctypes.data, depth1.ctypes.data)
    return (rgba, depth, accum, depth1) if want_passes else (rgba, depth)


def raymarch_rays(modelview, projection, bbox_min, bbox_max, width, height, limit):
    """Per pixel the ray's target point in volume space and whether the cube proxy covers the pixel."""
    pts = np.zeros((height, width, 3), np.float32)
    cov = np.zeros((height, width), np.uint8)
    lib().ro_raymarch_rays(np.ascontiguousarray(modelview, np.float32).reshape(16), np.ascontiguousarray(projection, np.float32).reshape(16),
                           np.ascontiguousarray(bbox_min, np.float32), np.ascontiguousarray(bbox_max, np.float32), int(width), int(height),
                           np.float32(limit), pts, cov)
    return pts, cov


def raymarch_uniforms(modelview, projection, bbox_min, bbox_max, width, height):
    out = np.zeros(83, np.float32)
    lib().ro_raymarch_uniforms(np.ascontiguousarray(modelview, np.float32).reshape(16), np.ascontiguousarray(projection, np.float32).reshape(16),
                               np.ascontiguousarray(bbox_min, np.float32), np.ascontiguousarray(bbox_max, np.float32), int(width), int(height), out)
    return out


def fill_colors(rgba, depth, want_atlas=False):
    """ReconIntegration::fillColors on a raymarch result: rgba [H,W,4], depth [H,W] -> filled rgba [H,W,4]
    (and the final mip atlas when want_atlas)."""
    rgba = np.ascontiguousarray(rgba, np.float32)
    depth = np.ascontiguousarray(depth, np.float32)
    H, W, _ = rgba.shape
    out = np.zeros_like(rgba)
    if not want_atlas:
        lib().ro_fill_colors(rgba, depth, W, H, out, None, None)
        return out
    FW = int(np.float32(W) * np.float32(1.5))
    ac = np.zeros((H, FW, 4), np.float32)
    ad = np.zeros((H, FW), np.float32)
    lib().ro_fill_colors(rgba, depth, W, H, out, ac.ctypes.data, ad.ctypes.data)
    return out, ac, ad
