import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "rgbd-recon_b200"), os.path.join(ROOT, "oracle"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def bits_equal(a, b):
    """Bit-exact float comparison that treats NaN == NaN (payload-insensitive) and +0 == +0 only."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    an, bn = np.isnan(a), np.isnan(b)
    return (an == bn) & (an | (a.view(np.uint32) == b.view(np.uint32)))


def mismatch_report(name, got, want, limit=5):
    eq = bits_equal(got, want)
    bad = np.argwhere(~eq)
    lines = [f"{name}: {len(bad)} of {eq.size} values differ"]
    for idx in bad[:limit]:
        t = tuple(idx)
        lines.append(f"  at {t}: got {got[t]!r} want {want[t]!r}")
    return "\n".join(lines)


GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gold(name):
    return np.load(os.path.join(GOLD, name))


def assert_raymarch(got, want_rgba, want_depth, want_samples, want_hit, what, proj, sample_flips=0.0):
    """A raymarch (the oracle's or the kernels') vs the reference's tsdf_raymarch.fs: same fragments kept, same sample counts;
    surface depth within 0.1 mm in eye space (BASELINE's bar is 1 mm) and 1e-5 in window depth; colours within 2e-3 (bilinear
    RGB8 lookups and gradient normals amplify the ~1e-7 differences of the hit position)."""
    hit = got["depth"] < 1.0
    assert np.array_equal(hit, want_hit > 0), f"{what}: hit masks differ on {(hit != (want_hit > 0)).sum()} pixels"
    assert hit.sum() > 100
    assert (got["samples"] != want_samples).mean() <= sample_flips, f"{what}: sample counts differ on {(got['samples'] != want_samples).sum()} pixels"
    assert np.abs(got["depth"] - want_depth).max() <= 1e-5, what
    p22, p32 = np.float64(proj.reshape(16)[10]), np.float64(proj.reshape(16)[14])

    def eye_z(d):                                                       # inverse of gl_FragDepth = ((p22 z + p32) / -z) / 2 + 1/2
        return p32 / (-(2.0 * d.astype(np.float64) - 1.0) - p22)

    dz_mm = np.abs(eye_z(got["depth"][hit]) - eye_z(want_depth[hit])) * 1000.0
    assert dz_mm.max() <= 0.1, f"{what}: surface differs by {dz_mm.max():.4f} mm"
    assert (np.isnan(got["rgba"]) == np.isnan(want_rgba)).all(), what
    ok = np.isfinite(got["rgba"]) & np.isfinite(want_rgba)
    assert np.abs(got["rgba"][ok] - want_rgba[ok]).max() <= 2e-3, what


def assert_points(got, want, what):
    """Point renderings agree when coverage is the same up to a handful of boundary pixels (the fixed-function stage is fp64 in
    the shader harness, fp32 in the oracle) and, where the same point won, depth to 2e-7 and colour to 2e-5."""
    (rgba, depth), (w_rgba, w_depth) = got, want
    cov, w_cov = depth < 1.0, w_depth < 1.0
    assert w_cov.sum() > 50, what
    assert (cov != w_cov).sum() <= max(2, int(0.002 * w_cov.sum())), f"{what}: coverage differs on {(cov != w_cov).sum()} pixels"
    both = cov & w_cov
    same = both & (np.abs(depth - w_depth) <= 2e-7)
    assert same.sum() >= 0.995 * both.sum(), f"{what}: another point won on {both.sum() - same.sum()} pixels"
    assert np.abs(rgba - w_rgba)[same].max() <= 2e-5, what


def assert_trigrid(got, want, what):
    """Triangle-mesh renderings agree when coverage is the same up to a handful of pixels (a fragment test that lands on the
    other side of a threshold), depth to 2e-5 (window depth of triangles cut by the near plane) and colour to 5e-5."""
    (rgba, depth), (w_rgba, w_depth) = got, want
    cov, w_cov = depth < 1.0, w_depth < 1.0
    assert w_cov.sum() > 100, what
    assert (cov != w_cov).sum() <= max(2, int(0.002 * w_cov.sum())), f"{what}: coverage differs on {(cov != w_cov).sum()} pixels"
    both = cov & w_cov
    assert np.abs(depth - w_depth)[both].max() <= 2e-5, what
    d = np.abs(rgba - w_rgba)[both]
    assert (d > 5e-5).any(axis=-1).sum() <= max(2, int(0.002 * both.sum())), f"{what}: colour differs by up to {d.max()}"


@pytest.fixture(scope="session")
def small_scene():
    from rrpy import synth
    return synth.make_scene(N=2, W=128, H=106, CW=160, CH=135, cv_res=(32, 32, 64))
