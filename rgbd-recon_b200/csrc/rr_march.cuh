// The per-ray march of the raymarcher (tsdf_raymarch.fs:92-114 with the cube proxy and the brick depth limits made
// analytic), shared by rr_raymarch.cu and rr_query.cu so that a ray cast through rr_cast_rays and the same ray of a
// raymarched view give the same numbers.
//   * brick hull: a 3D-DDA over the brick grid visits the bricks on the ray (plus the neighbours across any edge or
//     corner the ray passes within a relative 1e-4 of, so sliver intersections are not lost) and evaluates the same
//     slab expression per occupied brick as a brute-force scan would: entry = min, exit = max.
//   * empty-space skipping inside the hull: a sample whose brick and all 26 neighbours are unoccupied reads the
//     cleared value -limit from all 8 taps, cannot be a hit, and its density is overwritten before it can be used —
//     its fetches are skipped while sample_pos += step is still replayed, so positions stay bit-identical.
//   * z-slab ownership (multi-GPU): a context samples only the steps whose z texel it owns; the composite picks the
//     smallest step index per ray.
// P is the caller's parameter block: the sample block of rr_sample.cuh plus
//   skip_space, allow_skip, occ_mask, near_occ, rb[3], brick_size, dims[3] (bbox size), z_own0, z_own1
#pragma once

#include "rr_context.h"
#include "rr_math.cuh"
#include "rr_sample.cuh"

#include <algorithm>
#include <cmath>

namespace rr {

__device__ __forceinline__ bool slab(float3 o, float3 invd, float3 lo, float3 hi, float& t0, float& t1) {
  const float ax = (lo.x - o.x) * invd.x, bx = (hi.x - o.x) * invd.x;
  const float ay = (lo.y - o.y) * invd.y, by = (hi.y - o.y) * invd.y;
  const float az = (lo.z - o.z) * invd.z, bz = (hi.z - o.z) * invd.z;
  t0 = gmax(gmax(gmin(ax, bx), gmin(ay, by)), gmin(az, bz));
  t1 = gmin(gmin(gmax(ax, bx), gmax(ay, by)), gmax(az, bz));
  return t0 <= t1;
}

template <class P>
__device__ __forceinline__ void test_brick(const P& p, int ix, int iy, int iz, float3 cam, float3 invd, float& T0, float& T1) {
  if (ix < 0 || iy < 0 || iz < 0 || ix >= p.rb[0] || iy >= p.rb[1] || iz >= p.rb[2]) return;
  if (!p.occ_mask[(iz * p.rb[1] + iy) * p.rb[0] + ix]) return;
  const float3 lo = make_float3(((float)ix * p.brick_size) / p.dims[0], ((float)iy * p.brick_size) / p.dims[1], ((float)iz * p.brick_size) / p.dims[2]);
  const float3 hi = make_float3(((float)(ix + 1) * p.brick_size) / p.dims[0], ((float)(iy + 1) * p.brick_size) / p.dims[1],
                                ((float)(iz + 1) * p.brick_size) / p.dims[2]);
  float t0, t1;
  if (!slab(cam, invd, lo, hi, t0, t1) || t1 < 0.0f) return;
  T0 = gmin(T0, gmax(t0, 0.0f));
  T1 = gmax(T1, t1);
}

// March the ray from cam (volume space) along the unit direction dir in steps of limit / 2. When the ray meets the unit
// cube (and, with skip_space, the brick hull) ahead of cam, done(num_samples, hit, sample_pos) is called once after the
// march: num_samples = the samples taken (the raymarch's tex_num_samples / 0.0027), sample_pos = the refined hit when hit.
// A callback rather than results, so that k_raymarch compiles to the code it had before the march was shared.
template <class P, class Done>
__device__ __forceinline__ void march_ray(const P& p, float3 cam, float3 dir, Done&& done) {
  const float sd = p.limit * 0.5f;
  const float3 step = dir * sd;
  const float3 invd = make_float3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);
  const float3 invs = make_float3(1.0f / step.x, 1.0f / step.y, 1.0f / step.z);
  float c0, c1;
  bool live = slab(cam, invs, make_float3(0.f, 0.f, 0.f), make_float3(1.f, 1.f, 1.f), c0, c1) && !(c1 < 0.0f);
  float3 sample_pos = cam;
  uint32_t max_num_samples = 0;
  if (live) {
    if (p.skip_space) {
      float T0 = __int_as_float(0x7f800000), T1 = __int_as_float(0xff800000);
      // 3D-DDA over the brick grid [0, rb*bsv) in volume space
      const float bsv[3] = {p.brick_size / p.dims[0], p.brick_size / p.dims[1], p.brick_size / p.dims[2]};
      const float gmaxv[3] = {bsv[0] * p.rb[0], bsv[1] * p.rb[1], bsv[2] * p.rb[2]};
      float g0, g1;
      if (slab(cam, invd, make_float3(0.f, 0.f, 0.f), make_float3(gmaxv[0], gmaxv[1], gmaxv[2]), g0, g1) && g1 >= 0.0f) {
        const float tstart = gmax(g0, 0.0f);
        const float d[3] = {dir.x, dir.y, dir.z}, oc[3] = {cam.x, cam.y, cam.z};
        int cell[3], stp[3];
        float tmax[3], tdelta[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const float e = oc[a] + d[a] * tstart;
          cell[a] = iclamp((int)floorf(e / bsv[a]), 0, p.rb[a] - 1);
          stp[a] = d[a] > 0.0f ? 1 : -1;
          if (d[a] != 0.0f) {
            const float bound = (float)(cell[a] + (d[a] > 0.0f ? 1 : 0)) * bsv[a];
            tmax[a] = (bound - oc[a]) / d[a];
            tdelta[a] = bsv[a] / fabsf(d[a]);
          } else {
            tmax[a] = __int_as_float(0x7f800000);
            tdelta[a] = __int_as_float(0x7f800000);
          }
        }
        const int max_iter = p.rb[0] + p.rb[1] + p.rb[2] + 3;
        for (int it = 0; it < max_iter; ++it) {
          test_brick(p, cell[0], cell[1], cell[2], cam, invd, T0, T1);
          const float tn = gmin(tmax[0], gmin(tmax[1], tmax[2]));
          if (tn > g1) break;
          // near an edge/corner: also test the cells across every boundary within eps of the next crossing
          const float eps = 1e-4f * fabsf(tn) + 1e-6f;
          const bool nx = (tmax[0] - tn) <= eps, ny = (tmax[1] - tn) <= eps, nz = (tmax[2] - tn) <= eps;
          if ((int)nx + (int)ny + (int)nz > 1) {
            for (int m = 1; m < 8; ++m) {
              if (((m & 1) && !nx) || ((m & 2) && !ny) || ((m & 4) && !nz)) continue;
              test_brick(p, cell[0] + ((m & 1) ? stp[0] : 0), cell[1] + ((m & 2) ? stp[1] : 0), cell[2] + ((m & 4) ? stp[2] : 0), cam, invd, T0, T1);
            }
          }
          const int ax = (tmax[0] <= tmax[1] && tmax[0] <= tmax[2]) ? 0 : ((tmax[1] <= tmax[2]) ? 1 : 2);
          if (ax == 0) { cell[0] += stp[0]; tmax[0] += tdelta[0]; }
          else if (ax == 1) { cell[1] += stp[1]; tmax[1] += tdelta[1]; }
          else { cell[2] += stp[2]; tmax[2] += tdelta[2]; }
          if (cell[0] < 0 || cell[1] < 0 || cell[2] < 0 || cell[0] >= p.rb[0] || cell[1] >= p.rb[1] || cell[2] >= p.rb[2]) break;
        }
      }
      if (T0 <= T1) {
        sample_pos = cam + dir * T0;
        max_num_samples = f2u_sat(ceilf((T1 - T0) / sd));
      } else {
        live = false;
      }
    } else {
      const float t_near = (c0 < 0.0f) ? 0.0f : c0;
      sample_pos = cam + step * t_near;
      max_num_samples = f2u_sat(ceilf(fabsf(c1 - t_near)));
    }
  }

  if (live) {
    float prev_density = -p.limit;
    float3 prev_pos = sample_pos;
    bool prev_valid = true;      // prev_density holds the density of the previous step (or the initial -limit)
    const float vbx = p.dims[0] / p.brick_size, vby = p.dims[1] / p.brick_size, vbz = p.dims[2] / p.brick_size;
    uint32_t num_samples = 0;
    bool hit = false;
    const bool sharded = (p.z_own0 > 0) || (p.z_own1 < p.Z);
    while (num_samples < max_num_samples) {
      num_samples += 1;
      bool evaluate = true;
      if (sharded) {
        const int zi = near_coord(sample_pos.z, p.Z);
        evaluate = (zi >= p.z_own0 && zi < p.z_own1);
      }
      if (evaluate && p.allow_skip) {
        const int bx = (int)floorf(sample_pos.x * vbx), by = (int)floorf(sample_pos.y * vby), bz = (int)floorf(sample_pos.z * vbz);
        if (bx >= 0 && by >= 0 && bz >= 0 && bx < p.rb[0] && by < p.rb[1] && bz < p.rb[2])
          evaluate = p.near_occ[(bz * p.rb[1] + by) * p.rb[0] + bx] != 0;
      }
      if (evaluate) {
        const float density = sample_tsdf(p, sample_pos);
        if (density > 0.0f) {
          if (!prev_valid) prev_density = sample_tsdf(p, prev_pos);
          const float ratio = prev_density / (density - prev_density);
          sample_pos = (sample_pos - step) - step * ratio;
          hit = true;
          break;
        }
        prev_density = density;
        prev_valid = true;
      } else {
        prev_valid = false;
      }
      prev_pos = sample_pos;
      sample_pos = sample_pos + step;
    }
    done(num_samples, hit, sample_pos);
  }
}

// The sample block of P (rr_sample.cuh) from the context's volume, calibration and stage images.
template <class P>
inline void set_sample_params(P& p, const rr_ctx* c) {
  p.half2 = c->cfg.store_weight == RR_VOXELS_HALF2 ? 1 : 0;
  p.tsdf = c->d_tsdf.ptr; p.X = (int)c->res[0]; p.Y = (int)c->res[1]; p.Z = (int)c->res[2];
  p.limit = c->cfg.limit;
  p.N = c->N; p.inv = c->d_inv.ptr; p.IX = (int)c->ires[0]; p.IY = (int)c->ires[1]; p.IZ = (int)c->ires[2];
  for (int i = 0; i < c->N; ++i) { p.uv[i] = c->d_uv[i].ptr; p.cx[i] = (int)c->cres[i][0]; p.cy[i] = (int)c->cres[i][1]; p.cz[i] = (int)c->cres[i][2]; }
  p.color = c->d_color; p.CW = c->CW; p.CH = c->CH;
  p.depth_b = c->d_depth_b.ptr; p.quality = c->d_quality.ptr; p.W = c->W; p.H = c->H;
}

// The march fields of P (after set_sample_params) as rr_raymarch sets them from the context's current settings and brick tables.
template <class P>
inline void set_march_params(P& p, const rr_ctx* c) {
  const float dx = c->bbox_max[0] - c->bbox_min[0], dy = c->bbox_max[1] - c->bbox_min[1], dz = c->bbox_max[2] - c->bbox_min[2];
  const bool grid_ok = c->bricks.num == c->bricks.res[0] * c->bricks.res[1] * c->bricks.res[2];
  p.skip_space = (c->cfg.skip_space && c->cfg.use_bricks && grid_ok) ? 1 : 0;   // drawF: m_skip_space && m_use_bricks
  p.occ_mask = c->d_occ_mask.ptr; p.near_occ = c->d_near_occ.ptr;
  for (int a = 0; a < 3; ++a) p.rb[a] = (int)c->bricks.res[a];
  p.brick_size = c->bricks.brick_size;
  p.dims[0] = dx; p.dims[1] = dy; p.dims[2] = dz;
  // fetch skipping needs: bricks mode (unoccupied bricks hold the cleared value), bricks of >= 8 voxels per side and a
  // march step shorter than half a brick, so a skipped sample is never the predecessor of a hit
  const float bvox_min = std::fmin(std::fmin(c->bricks.brick_size / dx * p.X, c->bricks.brick_size / dy * p.Y), c->bricks.brick_size / dz * p.Z);
  const float step_vox = p.limit * 0.5f * (float)std::max(p.X, std::max(p.Y, p.Z));
  p.allow_skip = (c->cfg.use_bricks && grid_ok && bvox_min >= 8.0f && step_vox * 2.0f <= bvox_min) ? 1 : 0;
  p.z_own0 = (int)c->slab_z0; p.z_own1 = (int)c->slab_z1;
}

}  // namespace rr
