// ORACLE (test infrastructure, NOT product code): scalar restatement of the library's volume queries (rr_sample_points /
// rr_cast_rays, rgbd-recon_b200/csrc/rr_query.cu; the contract is stated in include/rgbd_recon_b200.h). The sample
// functions are the raymarch oracle's (ro_sample.h); the march is ro_raymarch.cpp's with the brute-force brick hull, from
// the caller's origin and direction instead of a pixel's.
#include "ro_math.h"
#include "ro_sample.h"
#include "rr_oracle.h"

#include <cmath>
#include <vector>

namespace {

const float kNaN = std::nanf("");

bool finite3(V3 v) { return std::isfinite(v.x) && std::isfinite(v.y) && std::isfinite(v.z); }

bool slab(V3 o, V3 invd, V3 lo, V3 hi, float& t0, float& t1) {
  const float ax = (lo.x - o.x) * invd.x, bx = (hi.x - o.x) * invd.x;
  const float ay = (lo.y - o.y) * invd.y, by = (hi.y - o.y) * invd.y;
  const float az = (lo.z - o.z) * invd.z, bz = (hi.z - o.z) * invd.z;
  t0 = gl_max(gl_max(gl_min(ax, bx), gl_min(ay, by)), gl_min(az, bz));
  t1 = gl_min(gl_min(gl_max(ax, bx), gl_max(ay, by)), gl_max(az, bz));
  return t0 <= t1;
}

struct Space {
  V3 bmin, size;
  bool world;
  V3 point(V3 p) const { return world ? V3{(p.x - bmin.x) / size.x, (p.y - bmin.y) / size.y, (p.z - bmin.z) / size.z} : p; }
  // a finite non-zero direction whose dot product would overflow or underflow is first scaled by an exact power of two
  V3 direction(V3 d) const {
    if (world) {
      V3 v{d.x / size.x, d.y / size.y, d.z / size.z};
      if (!finite3(v) && finite3(d)) { d = d * 0x1p-70f; v = V3{d.x / size.x, d.y / size.y, d.z / size.z}; }
      d = v;
    }
    const float s = dot3(d, d);
    if (s == INFINITY) {
      d = d * 0x1p-70f;
    } else if (s < 0x1p-100f) {
      d = d * 0x1p64f;
      if (dot3(d, d) < 0x1p-100f) d = d * 0x1p64f;
    }
    return normalize3(d);
  }
  V3 out(V3 q) const { return world ? V3{bmin.x + q.x * size.x, bmin.y + q.y * size.y, bmin.z + q.z * size.z} : q; }
};

// the mesh vertex normal: the raymarch's gradient at q, in world space
V3 world_normal(const RM& r, const Space& s, V3 q) {
  const V3 g = get_gradient(r, q, r.limit * 0.5f);
  return normalize3(V3{g.x / s.size.x, g.y / s.size.y, g.z / s.size.z});
}

RM make_rm(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
           const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
           const float* depth_b, const float* quality, int W, int H) {
  return RM{tsdf, (int)res[0], (int)res[1], (int)res[2], limit, N, inv, inv_res[0], inv_res[1], inv_res[2],
            cv_uv, cv_res[0], cv_res[1], cv_res[2], color, CW, CH, depth_b, quality, W, H, 0};
}

Space make_space(const float* bmin, const float* bmax, int space) {
  return Space{V3{bmin[0], bmin[1], bmin[2]}, V3{bmax[0] - bmin[0], bmax[1] - bmin[1], bmax[2] - bmin[2]}, space == 0};
}

void put3(float* a, size_t i, V3 v) { if (a) { a[i * 3] = v.x; a[i * 3 + 1] = v.y; a[i * 3 + 2] = v.z; } }
void put4(float* a, size_t i, V4 v) { if (a) { a[i * 4] = v.x; a[i * 4 + 1] = v.y; a[i * 4 + 2] = v.z; a[i * 4 + 3] = v.w; } }

}  // namespace

extern "C" {

void ro_sample_points(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                      const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                      const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                      int space, const float* points, uint32_t count, float* values, float* normals, float* rgba) {
  const RM r = make_rm(tsdf, res, limit, N, inv, inv_res, cv_uv, cv_res, color, CW, CH, depth_b, quality, W, H);
  const Space s = make_space(bbox_min, bbox_max, space);
#pragma omp parallel for schedule(dynamic, 256)
  for (int64_t i = 0; i < (int64_t)count; ++i) {
    const V3 q = s.point(V3{points[i * 3], points[i * 3 + 1], points[i * 3 + 2]});
    // the closed unit cube; NaN compares false
    const bool inside = q.x >= 0.0f && q.x <= 1.0f && q.y >= 0.0f && q.y <= 1.0f && q.z >= 0.0f && q.z <= 1.0f;
    if (!inside) {
      if (values) values[i] = kNaN;
      put3(normals, i, V3{kNaN, kNaN, kNaN});
      put4(rgba, i, V4{0.0f, 0.0f, 0.0f, 0.0f});
      continue;
    }
    if (values) values[i] = sample_tsdf(r, q);
    put3(normals, i, world_normal(r, s, q));
    put4(rgba, i, blend_colors(r, q));
  }
}

void ro_cast_rays(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                  const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                  const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                  int skip_space, const uint32_t* occupied, uint32_t n_occ, const uint32_t* brick_res, float brick_size,
                  int space, const float* origins, const float* directions, uint32_t count,
                  float* positions, float* normals, float* rgba, uint32_t* steps) {
  const RM r = make_rm(tsdf, res, limit, N, inv, inv_res, cv_uv, cv_res, color, CW, CH, depth_b, quality, W, H);
  const Space s = make_space(bbox_min, bbox_max, space);
  const float sd = limit * 0.5f;
  const V3 dims = s.size;
  std::vector<V3> blo(n_occ), bhi(n_occ);
  for (uint32_t b = 0; b < n_occ; ++b) {
    uint32_t id = occupied[b];
    const uint32_t iz = id / (brick_res[0] * brick_res[1]); id %= (brick_res[0] * brick_res[1]);
    const uint32_t iy = id / brick_res[0], ix = id % brick_res[0];
    blo[b] = V3{((float)ix * brick_size) / dims.x, ((float)iy * brick_size) / dims.y, ((float)iz * brick_size) / dims.z};
    bhi[b] = V3{((float)(ix + 1) * brick_size) / dims.x, ((float)(iy + 1) * brick_size) / dims.y, ((float)(iz + 1) * brick_size) / dims.z};
  }
#pragma omp parallel for schedule(dynamic, 256)
  for (int64_t i = 0; i < (int64_t)count; ++i) {
    put3(positions, i, V3{kNaN, kNaN, kNaN});
    put3(normals, i, V3{kNaN, kNaN, kNaN});
    put4(rgba, i, V4{0.0f, 0.0f, 0.0f, 0.0f});
    if (steps) steps[i] = 0xFFFFFFFFu;
    const V3 cam = s.point(V3{origins[i * 3], origins[i * 3 + 1], origins[i * 3 + 2]});
    const V3 dir = s.direction(V3{directions[i * 3], directions[i * 3 + 1], directions[i * 3 + 2]});
    // a zero direction normalises to NaN; origins beyond 2^24 bbox sizes are not cast
    const float far = 0x1p24f;
    if (!finite3(cam) || !(fabsf(cam.x) <= far && fabsf(cam.y) <= far && fabsf(cam.z) <= far) || !finite3(dir) || !(dot3(dir, dir) > 0.0f)) continue;
    const V3 step = dir * sd;
    const V3 invd{1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z};
    const V3 invs{1.0f / step.x, 1.0f / step.y, 1.0f / step.z};
    float c0, c1;
    if (!slab(cam, invs, V3{0, 0, 0}, V3{1, 1, 1}, c0, c1) || c1 < 0.0f) continue;   // misses the unit cube ahead
    V3 sample_pos;
    uint32_t max_num_samples;
    if (skip_space) {
      float T0 = INFINITY, T1 = -INFINITY;
      for (uint32_t b = 0; b < n_occ; ++b) {
        float t0, t1;
        if (!slab(cam, invd, blo[b], bhi[b], t0, t1) || t1 < 0.0f) continue;
        T0 = gl_min(T0, gl_max(t0, 0.0f));
        T1 = gl_max(T1, t1);
      }
      if (!(T0 <= T1)) continue;                                                     // no occupied brick on the ray
      sample_pos = cam + dir * T0;
      max_num_samples = f2u_sat(ceilf((T1 - T0) / sd));
    } else {
      const float t_near = (c0 < 0.0f) ? 0.0f : c0;
      sample_pos = cam + step * t_near;
      max_num_samples = f2u_sat(ceilf(fabsf(c1 - t_near)));
    }
    float prev_density = -limit;
    uint32_t num_samples = 0;
    bool hit = false;
    while (num_samples < max_num_samples) {
      num_samples += 1;
      const float density = sample_tsdf(r, sample_pos);
      if (density > 0.0f) {
        const float ratio = prev_density / (density - prev_density);
        sample_pos = (sample_pos - step) - step * ratio;
        hit = true;
        break;
      }
      prev_density = density;
      sample_pos = sample_pos + step;
    }
    if (!hit) continue;
    put3(positions, i, s.out(sample_pos));
    put3(normals, i, world_normal(r, s, sample_pos));
    put4(rgba, i, blend_colors(r, sample_pos));
    if (steps) steps[i] = num_samples;
  }
}

}  // extern "C"
