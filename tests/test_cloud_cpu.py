"""The point-cloud contract (include/rgbd_recon_b200.h, "point clouds") on the oracle alone (oracle/ro_cloud.cpp): ascending
pixel ids, the sensor mask, the keep rule and an independent float64 restatement of the lookups. No GPU."""
import numpy as np
import oracle_cloud
import pytest


@pytest.fixture(scope="module")
def cloud_inputs():
    import oracle_py as O
    from rrpy import synth
    sc = synth.make_scene(N=3, W=96, H=80, CW=128, CH=108, cv_res=(24, 24, 48))
    grid = O.brick_grid(sc.bbox_min, sc.bbox_max, 0.02, 0.1)
    cams = [O.frustum(sc.cv_xyz[i])[1] for i in range(sc.N)]
    return sc, O.preprocess(sc, grid, cams)


def _lin(s, n):
    """lin_coord in float64: the two taps and the weight of LINEAR + CLAMP_TO_EDGE at coordinate s over n texels."""
    u = s * n - 0.5
    f = np.floor(u)
    return np.clip(f, 0, n - 1).astype(np.int64), np.clip(f + 1, 0, n - 1).astype(np.int64), u - f


def _tex3d(T, s, t, r):
    Z, Y, X = T.shape[:3]
    x0, x1, a = _lin(s, X)
    y0, y1, b = _lin(t, Y)
    z0, z1, g = _lin(r, Z)
    a, b, g = a[:, None], b[:, None], g[:, None]
    T = T.astype(np.float64)

    def lerp(p, q, w):
        return p + (q - p) * w
    c0 = lerp(lerp(T[z0, y0, x0], T[z0, y0, x1], a), lerp(T[z0, y1, x0], T[z0, y1, x1], a), b)
    c1 = lerp(lerp(T[z1, y0, x0], T[z1, y0, x1], a), lerp(T[z1, y1, x0], T[z1, y1, x1], a), b)
    return lerp(c0, c1, g)


def _rgb8(img, s, t):
    H, W = img.shape[:2]
    x0, x1, a = _lin(s, W)
    y0, y1, b = _lin(t, H)
    a, b = a[:, None], b[:, None]
    im = img.astype(np.float64) / 255.0
    return (im[y0, x0] * (1 - a) + im[y0, x1] * a) * (1 - b) + (im[y1, x0] * (1 - a) + im[y1, x1] * a) * b


def _numpy_cloud(sc, pre, sensor):
    """Every pixel of one sensor in float64: positions, texture coordinates, colours and the keep decision with its distance
    to the nearest keep threshold."""
    H, W = sc.H, sc.W
    y, x = np.mgrid[0:H, 0:W]
    sx = ((x.ravel() + 0.5) * np.float64(np.float32(1.0) / np.float32(W))).astype(np.float32).astype(np.float64)
    sy = ((y.ravel() + 0.5) * np.float64(np.float32(1.0) / np.float32(H))).astype(np.float32).astype(np.float64)
    d = pre["depth_b"][sensor, ..., 0].ravel().astype(np.float64)
    p = _tex3d(sc.cv_xyz[sensor], sx, sy, d)
    t = _tex3d(sc.cv_uv[sensor], sx, sy, d)
    bmin, bmax = sc.bbox_min.astype(np.float64), sc.bbox_max.astype(np.float64)
    keep = (d > 0) & (p >= bmin).all(1) & (p <= bmax).all(1) & (t >= 0.01).all(1) & (t <= 0.99).all(1)
    margin = np.minimum(np.abs(p - bmin).min(1), np.abs(p - bmax).min(1))
    margin = np.minimum(margin, np.minimum(np.abs(t - 0.01).min(1), np.abs(t - 0.99).min(1)))
    margin = np.where(d > 0, margin, np.inf)
    return p, t, _rgb8(sc.color[sensor], t[:, 0], t[:, 1]), keep, margin


def test_ids_ascend_and_the_mask_selects_the_subset(cloud_inputs):
    sc, pre = cloud_inputs
    full = oracle_cloud.extract_points_scene(sc, pre)
    pix = full[4]
    assert len(pix) > 1000
    assert (np.diff(pix.astype(np.int64)) > 0).all()
    layer = pix // (sc.W * sc.H)
    assert set(np.unique(layer)) == set(range(sc.N))
    for mask in (0b001, 0b010, 0b100, 0b101, 0b110):
        sub = oracle_cloud.extract_points_scene(sc, pre, mask)
        sel = ((mask >> layer) & 1).astype(bool)
        for a, b in zip(sub, full):
            assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a,
                                  b[sel].view(np.uint32) if b.dtype == np.float32 else b[sel])


def test_points_lie_in_the_bbox_and_colours_in_range(cloud_inputs):
    sc, pre = cloud_inputs
    pos, nrm, rgb, q, pix = oracle_cloud.extract_points_scene(sc, pre)
    assert (pos >= sc.bbox_min).all() and (pos <= sc.bbox_max).all()
    assert np.isfinite(pos).all() and np.isfinite(rgb).all()
    assert (rgb >= 0).all() and (rgb <= 1).all()
    flat = pix.astype(np.int64)
    assert np.array_equal(q, pre["quality"].reshape(-1)[flat])
    assert np.array_equal(nrm, pre["normal"].reshape(-1, 3)[flat])
    assert (pre["depth_b"][..., 0].reshape(-1)[flat] > 0).all()


def test_float64_restatement_agrees(cloud_inputs):
    sc, pre = cloud_inputs
    pos, nrm, rgb, q, pix = oracle_cloud.extract_points_scene(sc, pre)
    px = sc.W * sc.H
    for i in range(sc.N):
        p, t, c, keep, margin = _numpy_cloud(sc, pre, i)
        clear = margin > 1e-4                                      # away from the keep thresholds
        mine = pix[(pix // px) == i] - i * px
        got_keep = np.zeros(px, bool)
        got_keep[mine] = True
        assert np.array_equal(got_keep[clear], keep[clear]), f"sensor {i}: keep decisions differ"
        sel = (pix // px) == i
        assert np.abs(pos[sel] - p[mine]).max() <= 1e-5
        assert np.abs(rgb[sel] - c[mine]).max() <= 1e-5


def test_empty_mask_gives_an_empty_cloud(cloud_inputs):
    sc, pre = cloud_inputs
    out = oracle_cloud.extract_points_scene(sc, pre, 0)
    assert [len(a) for a in out] == [0] * 5
    assert out[0].shape == (0, 3) and out[4].dtype == np.uint32
