// Depth pre-processing kernels for sm_100a: the work NetKinectArray::processTextures drives through five GLSL
// passes per sensor (framework/NetKinectArray.cpp:251-290, 311-428; glsl/pre_morph.fs, pre_depth.fs,
// pre_boundary.fs, pre_normal.fs + inc_bricks.glsl, pre_quality.fs). One launch per pass covers all sensors
// (blockIdx.z = sensor layer). The 13x13 passes stage a (32+12)x(8+12) depth tile in shared memory; brick
// occupancy counts are aggregated per warp (__match_any_sync) before one RED per distinct brick. pre_normal and pre_quality
// run as ONE launch (k_normal_quality; the separate kernels stay behind the tunable fuse_nq = 0).
// A further kernel packs depth_b / quality / silhouette into the 32-byte gather texels the integrator reads.
#include "rr_context.h"
#include "rr_math.cuh"

namespace rr {

#define TILE_X 32
#define TILE_Y 8
#define KS 6
#define SM_W (TILE_X + 2 * KS)
#define SM_H (TILE_Y + 2 * KS)
static_assert(TILE_X * TILE_Y == 256, "k_bilateral fills its 256-entry byte table with one entry per thread");

// ------------------------------------------------------------------------------------------------ pre_morph
// glsl/pre_morph.fs:73-112 dilate(kernel 1), main mode 0; mode 1 is a copy and is folded away.
__global__ void __launch_bounds__(256) k_morph(const float* __restrict__ in, float* __restrict__ out, int W, int H) {
  const int px = blockIdx.x * TILE_X + threadIdx.x, py = blockIdx.y * TILE_Y + threadIdx.y;
  if (px >= W || py >= H) return;
  const float* img = in + (size_t)blockIdx.z * W * H;
  const float min_depth = 0.5f, max_depth = 4.5f, max_dist = 0.2f;
  const float depth = img[(size_t)py * W + px];
  float result;
  if (depth > min_depth && depth < max_depth) {
    result = depth;
  } else {
    float nb[9];
#pragma unroll
    for (int y = -1; y < 2; ++y)
#pragma unroll
      for (int x = -1; x < 2; ++x)
        nb[(y + 1) * 3 + (x + 1)] = img[(size_t)iclamp(py + y, 0, H - 1) * W + iclamp(px + x, 0, W - 1)];
    float average_depth = 0.0f, num = 0.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i)
      if (nb[i] > min_depth && nb[i] < max_depth) { average_depth += nb[i]; num += 1.0f; }
    if (num == 0.0f) {
      result = 0.0f;
    } else {
      average_depth /= num;
      float new_depth = 0.0f;
      num = 0.0f;
#pragma unroll
      for (int i = 0; i < 9; ++i)
        if (nb[i] > min_depth && nb[i] < max_depth && fabsf(average_depth - nb[i]) < max_dist) { new_depth += nb[i]; num += 1.0f; }
      result = (num == 0.0f) ? 0.0f : new_depth / num;
    }
  }
  out[(size_t)blockIdx.z * W * H + (size_t)py * W + px] = result;
}

// ------------------------------------------------------------------------------------------------ pre_depth
__device__ __forceinline__ float pivot_rgb(float n) {
  return ((n > 0.04045f) ? gpow((n + 0.055f) / 1.055f, 2.4f) : n / 12.92f) * 100.0f;
}
__device__ __forceinline__ float pivot_xyz(float n) {
  return (n > 0.008856f) ? gpow(n, 1.0f / 3.0f) : (903.3f * n + 16.0f) / 116.0f;
}
// glsl/inc_color.glsl:8-46, including its redundant /255
__device__ float3 rgb_to_lab(float3 rgb) {
  float r = pivot_rgb(rgb.x / 255.0f), g = pivot_rgb(rgb.y / 255.0f), b = pivot_rgb(rgb.z / 255.0f);
  float X = (r * 0.4124f + g * 0.3576f) + b * 0.1805f;
  float Y = (r * 0.2126f + g * 0.7152f) + b * 0.0722f;
  float Z = (r * 0.0193f + g * 0.1192f) + b * 0.9505f;
  float x = pivot_xyz(X / 95.047f), y = pivot_xyz(Y / 100.000f), z = pivot_xyz(Z / 108.883f);
  return make_float3(gmax(0.0f, 116.0f * y - 16.0f), 500.0f * (x - y), 200.0f * (y - z));
}

struct DepthParams {
  float bmin[3], bmax[3];
  int filter_textures;
  int compress[RR_MAX_SENSORS];
  float scale[RR_MAX_SENSORS], near_[RR_MAX_SENSORS], scaled_near[RR_MAX_SENSORS];
};

// glsl/pre_depth.fs:129-154 main + :85-127 bilateral_filter (13x13, linear space/range kernels).
__global__ void __launch_bounds__(256) k_bilateral(const float* __restrict__ depth_in, const uint8_t* __restrict__ color,
                                                   float2* __restrict__ out_depth, float4* __restrict__ out_lab,
                                                   int W, int H, int CW, int CH,
                                                   const __grid_constant__ SensorTables st, const __grid_constant__ DepthParams dp) {
  // Tile of the 13x13 neighbourhoods. A sample the shader would skip because it lies outside the depth limits
  // (is_outside, pre_depth.fs:40-42) is stored as +inf: |inf - depth| = inf exceeds every finite range threshold, so the
  // single range comparison below also rejects it. The centre depth itself is kept in a register, untouched.
  __shared__ float tile[SM_H][SM_W];
  __shared__ float byte_lut[256];          // c / 255 of the colour fetch (tex2d_rgb8_lut)
  const int layer = blockIdx.z;
  const float* img = depth_in + (size_t)layer * W * H;
  const int bx = blockIdx.x * TILE_X, by = blockIdx.y * TILE_Y;
  const int tid = threadIdx.y * TILE_X + threadIdx.x;
  byte_lut[tid] = (float)tid / 255.0f;     // TILE_X * TILE_Y == 256 threads
  const bool compress = dp.compress[layer] != 0;
  const float cv_min = st.dmin[layer], cv_max = st.dmax[layer];
  auto decode = [&](float d) -> float {
    if (compress) d = (d < dp.scaled_near[layer]) ? 0.0f : (d * d + 0.15f * dp.scaled_near[layer]) * dp.scale[layer] + dp.near_[layer];
    return d;
  };
  for (int i = tid; i < SM_W * SM_H; i += TILE_X * TILE_Y) {
    int ty = i / SM_W, tx = i - ty * SM_W;
    const float d = decode(img[(size_t)iclamp(by + ty - KS, 0, H - 1) * W + iclamp(bx + tx - KS, 0, W - 1)]);
    tile[ty][tx] = ((d < cv_min) || (d > cv_max)) ? __int_as_float(0x7f800000) : d;
  }
  __syncthreads();
  const int px = bx + threadIdx.x, py = by + threadIdx.y;
  if (px >= W || py >= H) return;
  const float tcx = ((float)px + 0.5f) / (float)W, tcy = ((float)py + 0.5f) / (float)H;
  const float depth = decode(img[(size_t)py * W + px]);
  const float depth_norm = (depth - cv_min) / (cv_max - cv_min);
  const float3 pos_world = tex3d_xyz(st.xyz[layer], st.cx[layer], st.cy[layer], st.cz[layer], tcx, tcy, depth_norm);
  const bool in_box = pos_world.x >= dp.bmin[0] && pos_world.y >= dp.bmin[1] && pos_world.z >= dp.bmin[2] &&
                      pos_world.x <= dp.bmax[0] && pos_world.y <= dp.bmax[1] && pos_world.z <= dp.bmax[2];
  const float zc = (depth_norm <= 0.0f || depth_norm >= 1.0f) ? 1.0f : depth_norm;
  const float2 cc = tex3d_uv(st.uv[layer], st.cx[layer], st.cy[layer], st.cz[layer], tcx, tcy, zc);
  const float3 lab = rgb_to_lab(tex2d_rgb8_lut(color + (size_t)layer * CW * CH * 3, CW, CH, cc.x, cc.y, byte_lut));
  const size_t o = (size_t)layer * W * H + (size_t)py * W + px;
  out_lab[o] = make_float4(lab.x, lab.y, lab.z, 0.0f);
  if (!in_box) { out_depth[o] = make_float2(0.0f, 0.0f); return; }
  if (!dp.filter_textures) { out_depth[o] = make_float2(depth_norm, 1.0f); return; }
  const float d_dmax = depth / 4.5f;
  const float dist_range_max = 0.35f * d_dmax;
  const float dist_range_max_inv = 1.0f / dist_range_max;
  float depth_bf = 0.0f, w = 0.0f, w_range = 0.0f;
  if (depth - depth == 0.0f) {
    // finite centre (always, for real frames): one comparison per tap; the space weights 1 - |offset|/6 fold to constants
#pragma unroll
    for (int y = -KS; y <= KS; ++y) {
#pragma unroll
      for (int x = -KS; x <= KS; ++x) {
        const float depth_s = tile[threadIdx.y + KS + y][threadIdx.x + KS + x];
        const float depth_range = fabsf(depth_s - depth);
        if (depth_range > dist_range_max) continue;
        // min(depth_range, dist_range_max) == depth_range here (pre_depth.fs:112)
        const float gauss_range = 1.0f - depth_range * dist_range_max_inv;
        const float gauss_space = 1.0f - sqrtf((float)(x * x + y * y)) * (1.0f / 6.0f);
        const float w_s = gauss_space * gauss_range;
        depth_bf = fmaf(w_s, depth_s, depth_bf);
        w += w_s;
        w_range += gauss_range;
      }
    }
  } else {
    // inf / NaN centre: keep the shader's literal predicate order
#pragma unroll 1
    for (int y = -KS; y <= KS; ++y) {
#pragma unroll 1
      for (int x = -KS; x <= KS; ++x) {
        const float depth_s = decode(img[(size_t)iclamp(py + y, 0, H - 1) * W + iclamp(px + x, 0, W - 1)]);
        const float depth_range = fabsf(depth_s - depth);
        if ((depth_s < cv_min) || (depth_s > cv_max) || (depth_range > dist_range_max)) continue;
        const float gauss_range = 1.0f - gmin(depth_range, dist_range_max) * dist_range_max_inv;
        const float gauss_space = 1.0f - sqrtf((float)(x * x + y * y)) * (1.0f / 6.0f);
        const float w_s = gauss_space * gauss_range;
        depth_bf = fmaf(w_s, depth_s, depth_bf);
        w += w_s;
        w_range += gauss_range;
      }
    }
  }
  const float filtered = depth_bf / w;
  out_depth[o] = make_float2((filtered - cv_min) / (cv_max - cv_min), w_range / 169.0f);
}

// ------------------------------------------------------------------------------------------------ pre_boundary
// glsl/pre_boundary.fs:86-118 main, :37-55 get_color_diff (5x5, Lab distance, at least 8 of 16 "total_samples").
__global__ void __launch_bounds__(256) k_boundary(const float2* __restrict__ depth_rg, const float4* __restrict__ lab,
                                                  float2* __restrict__ out_depth_b, float* __restrict__ out_sil,
                                                  int W, int H, int refine) {
  const int px = blockIdx.x * TILE_X + threadIdx.x, py = blockIdx.y * TILE_Y + threadIdx.y;
  if (px >= W || py >= H) return;
  const size_t base = (size_t)blockIdx.z * W * H;
  const size_t o = base + (size_t)py * W + px;
  float2 d = depth_rg[o];
  float sil = 1.0f;
  if (d.x <= 0.0f) {
    d.y = 0.0f;
    sil = 0.0f;
  } else if (!(d.y > 0.65f)) {
    sil = 0.0f;
    const float4 c4 = lab[o];
    const float3 color = make_float3(c4.x, c4.y, c4.z);
    float total_dist = 0.0f, num = 0.0f;
    for (int y = -2; y <= 2; ++y)
      for (int x = -2; x <= 2; ++x) {
        const size_t si = base + (size_t)iclamp(py + y, 0, H - 1) * W + iclamp(px + x, 0, W - 1);
        const float2 ds = depth_rg[si];
        if (ds.x > 0.0f && ds.y > 0.65f) {
          num += 1.0f;
          const float4 s4 = lab[si];
          total_dist += length3(color - make_float3(s4.x, s4.y, s4.z));
        }
      }
    const float color_dist = (num < 16.0f * 0.5f) ? 1.0f : total_dist / num;
    if (color_dist > 0.5f || !refine) { d.x = -1.0f; d.y = 0.1f; }
    else d.y = 1.0f;
  } else {
    d.y = 0.0f;
  }
  out_depth_b[o] = d;
  out_sil[o] = sil;
}

// ------------------------------------------------------------------------------------------------ pre_normal
struct BrickParams {
  float bmin[3];
  float brick_size;
  uint32_t res[3];
  uint32_t num;
};

// glsl/pre_normal.fs:26-56 + glsl/inc_bricks.glsl:40-58 mark_brick. Counter updates are warp-aggregated:
// lanes that hit the same brick id elect one leader that issues a single RED with the group's population.
__device__ __forceinline__ void brick_add(uint32_t* __restrict__ bricks, uint32_t id, bool active) {
  const unsigned live = __ballot_sync(0xffffffffu, active);
  if (!active) return;
  const unsigned peers = __match_any_sync(live, id);
  if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(bricks + id, (uint32_t)__popc(peers));
}

__global__ void __launch_bounds__(256) k_normal(const float2* __restrict__ depth_b, float4* __restrict__ out_normal,
                                                uint32_t* __restrict__ bricks, int W, int H,
                                                const __grid_constant__ SensorTables st, const __grid_constant__ BrickParams bp) {
  const int layer = blockIdx.z;
  const int px = blockIdx.x * TILE_X + threadIdx.x, py = blockIdx.y * TILE_Y + threadIdx.y;
  const bool inside = (px < W && py < H);
  const size_t base = (size_t)layer * W * H;
  auto dep = [&](int x, int y) { return depth_b[base + (size_t)iclamp(y, 0, H - 1) * W + iclamp(x, 0, W - 1)].x; };
  auto is_outside = [](float d) { return (d <= 0.0f) || (d >= 1.0f); };
  const float4* xyz = st.xyz[layer];
  const int CX = st.cx[layer], CY = st.cy[layer], CZ = st.cz[layer];
  float depth = inside ? dep(px, py) : 0.0f;
  const bool valid = inside && !is_outside(depth);
  const float tcx = ((float)px + 0.5f) / (float)W, tcy = ((float)py + 0.5f) / (float)H;
  uint32_t id_own = 0, id_nb = 0;
  bool add_own = false, add_nb = false;
  float3 world = make_float3(0.f, 0.f, 0.f);
  if (valid) {
    world = tex3d_xyz(xyz, CX, CY, CZ, tcx, tcy, depth);
    const float3 bmin = make_float3(bp.bmin[0], bp.bmin[1], bp.bmin[2]);
    const float3 rel = (world - bmin) / bp.brick_size;
    const uint32_t ix = f2u_sat(floorf(rel.x)), iy = f2u_sat(floorf(rel.y)), iz = f2u_sat(floorf(rel.z));
    const float3 fidx = make_float3((float)ix, (float)iy, (float)iz);
    const float hb = 0.5f * bp.brick_size;
    const float3 center = (fidx * bp.brick_size + bmin) + make_float3(hb, hb, hb);
    const float3 diff = world - center;
    const float3 d_abs = make_float3(fabsf(diff.x), fabsf(diff.y), fabsf(diff.z));
    const float min_v = gmax(d_abs.x, gmax(d_abs.y, d_abs.z));
    const float cx = (d_abs.x < min_v) ? 0.0f : 1.0f, cy = (d_abs.y < min_v) ? 0.0f : 1.0f, cz = (d_abs.z < min_v) ? 0.0f : 1.0f;
    const int ox = (int)gsign(diff.x * cx), oy = (int)gsign(diff.y * cy), oz = (int)gsign(diff.z * cz);
    const int nx = iclamp((int)ix + ox, 0, (int)(bp.res[0] - 1u));
    const int ny = iclamp((int)iy + oy, 0, (int)(bp.res[1] - 1u));
    const int nz = iclamp((int)iz + oz, 0, (int)(bp.res[2] - 1u));
    id_nb = (uint32_t)nz * bp.res[1] * bp.res[0] + (uint32_t)ny * bp.res[0] + (uint32_t)nx;
    add_nb = (d_abs.x > bp.brick_size * 0.1f) && id_nb < bp.num;
    id_own = iz * bp.res[1] * bp.res[0] + iy * bp.res[0] + ix;
    add_own = id_own < bp.num;
  }
  brick_add(bricks, id_nb, add_nb);
  brick_add(bricks, id_own, add_own);
  if (!inside) return;
  const size_t o = base + (size_t)py * W + px;
  if (!valid) { out_normal[o] = make_float4(0.f, 0.f, 0.f, 0.f); return; }
  const float tsx = 1.0f / (float)W, tsy = 1.0f / (float)H;
  const float tty = tcy + tsy, tby = tcy - tsy, tlx = tcx - tsx, trx = tcx + tsx;
  float depth_t = dep(px, py + 1), depth_bb = dep(px, py - 1), depth_l = dep(px - 1, py), depth_r = dep(px + 1, py);
  depth_t = is_outside(depth_t) ? depth : depth_t;
  depth_bb = is_outside(depth_bb) ? depth : depth_bb;
  depth_l = is_outside(depth_l) ? depth : depth_l;
  depth_r = is_outside(depth_r) ? depth : depth_r;
  const float3 world_t = tex3d_xyz(xyz, CX, CY, CZ, tcx, tty, depth_t);
  const float3 world_b = tex3d_xyz(xyz, CX, CY, CZ, tcx, tby, depth_bb);
  const float3 world_l = tex3d_xyz(xyz, CX, CY, CZ, tlx, tcy, depth_l);
  const float3 world_r = tex3d_xyz(xyz, CX, CY, CZ, trx, tcy, depth_r);
  const float3 n = normalize3(cross3(world_b - world_t, world_l - world_r));
  out_normal[o] = make_float4(n.x, n.y, n.z, 0.0f);
}

// ------------------------------------------------------------------------------------------------ pre_quality
// glsl/pre_quality.fs:65-119 (13x13 support count + range weights, pow 6, 1/(6.5 d), angle^2); :115's colour loop is dead.
__global__ void __launch_bounds__(256) k_quality(const float2* __restrict__ depth_b, const float4* __restrict__ normals,
                                                 float* __restrict__ out_quality, const float* __restrict__ sil, float2* __restrict__ pairs,
                                                 int pair_pitch, uint32_t* __restrict__ flags, int W, int H,
                                                 const __grid_constant__ SensorTables st) {
  // as in k_bilateral: samples outside (0, 1) are stored as +inf so that the range comparison alone rejects them
  __shared__ float tile[SM_H][SM_W];
  const int layer = blockIdx.z;
  const size_t base = (size_t)layer * W * H;
  const int bx = blockIdx.x * TILE_X, by = blockIdx.y * TILE_Y;
  const int tid = threadIdx.y * TILE_X + threadIdx.x;
  for (int i = tid; i < SM_W * SM_H; i += TILE_X * TILE_Y) {
    int ty = i / SM_W, tx = i - ty * SM_W;
    const float d = depth_b[base + (size_t)iclamp(by + ty - KS, 0, H - 1) * W + iclamp(bx + tx - KS, 0, W - 1)].x;
    tile[ty][tx] = ((d <= 0.0f) || (d >= 1.0f)) ? __int_as_float(0x7f800000) : d;
  }
  __syncthreads();
  const int px = bx + threadIdx.x, py = by + threadIdx.y;
  if (px >= W || py >= H) return;
  const size_t o = base + (size_t)py * W + px;
  const float depth = depth_b[o].x;
  // The pair image the staged integrator tiles into shared memory (rr_integrate_staged.cu): per pixel (depth_b.x, quality
  // with the silhouette - exactly 0 or 1, pre_boundary.fs:88-108 - in the sign bit), one replicated border pixel on every
  // side so that a CLAMP_TO_EDGE footprint is pixels (e, e+1) of the padded image. quality is never negative (a product
  // of pow() results and positive divisors), so the sign bit is free; violations are counted in flags[0].
  auto emit = [&](float q) {
    out_quality[o] = q;
    if (!pairs) return;
    uint32_t bits = __float_as_uint(q);
    if ((bits >> 31) && !(q != q) && q != 0.0f) atomicAdd(flags, 1u);
    bits &= 0x7fffffffu;
    if (sil[o] >= 1.0f) bits |= 0x80000000u;
    const float2 v = make_float2(depth, __uint_as_float(bits));
    float2* img = pairs + (size_t)layer * (H + 2) * pair_pitch;
    const int xs0 = px + 1, xs1 = (px == 0) ? 0 : ((px == W - 1) ? W + 1 : -1);
    const int ys0 = py + 1, ys1 = (py == 0) ? 0 : ((py == H - 1) ? H + 1 : -1);
    img[(size_t)ys0 * pair_pitch + xs0] = v;
    if (xs1 >= 0) img[(size_t)ys0 * pair_pitch + xs1] = v;
    if (ys1 >= 0) img[(size_t)ys1 * pair_pitch + xs0] = v;
    if (xs1 >= 0 && ys1 >= 0) img[(size_t)ys1 * pair_pitch + xs1] = v;
    if (W == 1 && px == 0) {               // a one-pixel-wide image is its own left and right border
      img[(size_t)ys0 * pair_pitch + 2] = v;
      if (ys1 >= 0) img[(size_t)ys1 * pair_pitch + 2] = v;
    }
    if (H == 1 && py == 0) {
      img[(size_t)2 * pair_pitch + xs0] = v;
      if (xs1 >= 0) img[(size_t)2 * pair_pitch + xs1] = v;
      if (W == 1) img[(size_t)2 * pair_pitch + 2] = v;
    }
  };
  if ((depth <= 0.0f) || (depth >= 1.0f)) { emit(0.0f); return; }     // a NaN centre passes, as in the shader
  const float dist_range_max = 0.35f * (depth / 1.0f);
  const float dist_range_max_inv = 1.0f / dist_range_max;
  float w_range = 0.0f, border = 0.0f;
  if (depth - depth == 0.0f) {
#pragma unroll
    for (int y = 0; y <= 2 * KS; ++y) {
#pragma unroll
      for (int x = 0; x <= 2 * KS; ++x) {
        const float depth_range = fabsf(tile[threadIdx.y + y][threadIdx.x + x] - depth);
        if (depth_range > dist_range_max) { border += 1.0f; continue; }
        w_range += 1.0f - depth_range * dist_range_max_inv;
      }
    }
  } else {
#pragma unroll 1
    for (int y = -KS; y <= KS; ++y) {
#pragma unroll 1
      for (int x = -KS; x <= KS; ++x) {
        const float depth_s = depth_b[base + (size_t)iclamp(py + y, 0, H - 1) * W + iclamp(px + x, 0, W - 1)].x;
        const float depth_range = fabsf(depth_s - depth);
        if ((depth_s <= 0.0f) || (depth_s >= 1.0f) || (depth_range > dist_range_max)) { border += 1.0f; continue; }
        w_range += 1.0f - gmin(depth_range, dist_range_max) * dist_range_max_inv;
      }
    }
  }
  const float lateral_quality = 1.0f - border / 169.0f;
  float q = gpow(lateral_quality, 6.0f);
  q *= gpow(w_range / 169.0f, 6.0f);
  q /= depth * 6.5f;
  const float tcx = ((float)px + 0.5f) / (float)W, tcy = ((float)py + 0.5f) / (float)H;
  const float4 n4 = normals[o];
  const float3 world_pos = tex3d_xyz(st.xyz[layer], st.cx[layer], st.cy[layer], st.cz[layer], tcx, tcy, depth);
  const float3 cam = make_float3(st.cam[layer][0], st.cam[layer][1], st.cam[layer][2]);
  const float angle = dot3(normalize3(cam - world_pos), make_float3(n4.x, n4.y, n4.z));
  q *= gpow(angle, 2.0f);
  emit(q);
}

// ------------------------------------------------------------------------------------------------ pre_normal + pre_quality
// The two passes in one launch: pre_normal.fs is per pixel over depth_b's 4-neighbourhood, which pre_quality.fs's 13x13 tile
// already holds (its +inf code for a sample outside (0, 1) is pre_normal's is_outside), the normal feeds pre_quality's angle term
// from registers, and the centre's world position (the same tex3d_xyz of the same coordinates in both shaders) is fetched once.
// The four neighbour fetches are issued ahead of the 169-tap loop, whose arithmetic hides their latency. Every value is
// computed by the expressions of k_normal / k_quality above: bit-identical stage images and brick counters.
__global__ void __launch_bounds__(256) k_normal_quality(const float2* __restrict__ depth_b, float4* __restrict__ out_normal,
                                                        uint32_t* __restrict__ bricks, float* __restrict__ out_quality,
                                                        const float* __restrict__ sil, float2* __restrict__ pairs, int pair_pitch,
                                                        uint32_t* __restrict__ flags, int W, int H,
                                                        const __grid_constant__ SensorTables st, const __grid_constant__ BrickParams bp) {
  __shared__ float tile[SM_H][SM_W];
  const int layer = blockIdx.z;
  const size_t base = (size_t)layer * W * H;
  const int bx = blockIdx.x * TILE_X, by = blockIdx.y * TILE_Y;
  const int tid = threadIdx.y * TILE_X + threadIdx.x;
  for (int i = tid; i < SM_W * SM_H; i += TILE_X * TILE_Y) {
    int ty = i / SM_W, tx = i - ty * SM_W;
    const float d = depth_b[base + (size_t)iclamp(by + ty - KS, 0, H - 1) * W + iclamp(bx + tx - KS, 0, W - 1)].x;
    tile[ty][tx] = ((d <= 0.0f) || (d >= 1.0f)) ? __int_as_float(0x7f800000) : d;
  }
  __syncthreads();
  const int px = bx + threadIdx.x, py = by + threadIdx.y;
  const bool inside = (px < W && py < H);
  const size_t o = base + (size_t)(inside ? py : 0) * W + (inside ? px : 0);
  const float depth = inside ? depth_b[o].x : 0.0f;
  const bool valid = inside && !((depth <= 0.0f) || (depth >= 1.0f));          // a NaN centre is valid, as in both shaders
  const float4* xyz = st.xyz[layer];
  const int CX = st.cx[layer], CY = st.cy[layer], CZ = st.cz[layer];
  const float tcx = ((float)px + 0.5f) / (float)W, tcy = ((float)py + 0.5f) / (float)H;
  // ---- pre_normal.fs:26-56 + inc_bricks.glsl:40-58 (k_normal) ----
  uint32_t id_own = 0, id_nb = 0;
  bool add_own = false, add_nb = false;
  float3 world = make_float3(0.f, 0.f, 0.f);
  if (valid) {
    world = tex3d_xyz(xyz, CX, CY, CZ, tcx, tcy, depth);
    const float3 bmin = make_float3(bp.bmin[0], bp.bmin[1], bp.bmin[2]);
    const float3 rel = (world - bmin) / bp.brick_size;
    const uint32_t ix = f2u_sat(floorf(rel.x)), iy = f2u_sat(floorf(rel.y)), iz = f2u_sat(floorf(rel.z));
    const float3 fidx = make_float3((float)ix, (float)iy, (float)iz);
    const float hb = 0.5f * bp.brick_size;
    const float3 center = (fidx * bp.brick_size + bmin) + make_float3(hb, hb, hb);
    const float3 diff = world - center;
    const float3 d_abs = make_float3(fabsf(diff.x), fabsf(diff.y), fabsf(diff.z));
    const float min_v = gmax(d_abs.x, gmax(d_abs.y, d_abs.z));
    const float cx = (d_abs.x < min_v) ? 0.0f : 1.0f, cy = (d_abs.y < min_v) ? 0.0f : 1.0f, cz = (d_abs.z < min_v) ? 0.0f : 1.0f;
    const int ox = (int)gsign(diff.x * cx), oy = (int)gsign(diff.y * cy), oz = (int)gsign(diff.z * cz);
    const int nx = iclamp((int)ix + ox, 0, (int)(bp.res[0] - 1u));
    const int ny = iclamp((int)iy + oy, 0, (int)(bp.res[1] - 1u));
    const int nz = iclamp((int)iz + oz, 0, (int)(bp.res[2] - 1u));
    id_nb = (uint32_t)nz * bp.res[1] * bp.res[0] + (uint32_t)ny * bp.res[0] + (uint32_t)nx;
    add_nb = (d_abs.x > bp.brick_size * 0.1f) && id_nb < bp.num;
    id_own = iz * bp.res[1] * bp.res[0] + iy * bp.res[0] + ix;
    add_own = id_own < bp.num;
  }
  brick_add(bricks, id_nb, add_nb);
  brick_add(bricks, id_own, add_own);
  if (!inside) return;
  auto emit = [&](float q) {
    out_quality[o] = q;
    if (!pairs) return;
    uint32_t bits = __float_as_uint(q);
    if ((bits >> 31) && !(q != q) && q != 0.0f) atomicAdd(flags, 1u);
    bits &= 0x7fffffffu;
    if (sil[o] >= 1.0f) bits |= 0x80000000u;
    const float2 v = make_float2(depth, __uint_as_float(bits));
    float2* img = pairs + (size_t)layer * (H + 2) * pair_pitch;
    const int xs0 = px + 1, xs1 = (px == 0) ? 0 : ((px == W - 1) ? W + 1 : -1);
    const int ys0 = py + 1, ys1 = (py == 0) ? 0 : ((py == H - 1) ? H + 1 : -1);
    img[(size_t)ys0 * pair_pitch + xs0] = v;
    if (xs1 >= 0) img[(size_t)ys0 * pair_pitch + xs1] = v;
    if (ys1 >= 0) img[(size_t)ys1 * pair_pitch + xs0] = v;
    if (xs1 >= 0 && ys1 >= 0) img[(size_t)ys1 * pair_pitch + xs1] = v;
    if (W == 1 && px == 0) {
      img[(size_t)ys0 * pair_pitch + 2] = v;
      if (ys1 >= 0) img[(size_t)ys1 * pair_pitch + 2] = v;
    }
    if (H == 1 && py == 0) {
      img[(size_t)2 * pair_pitch + xs0] = v;
      if (xs1 >= 0) img[(size_t)2 * pair_pitch + xs1] = v;
      if (W == 1) img[(size_t)2 * pair_pitch + 2] = v;
    }
  };
  if (!valid) { out_normal[o] = make_float4(0.f, 0.f, 0.f, 0.f); emit(0.0f); return; }
  const float tsx = 1.0f / (float)W, tsy = 1.0f / (float)H;
  const float tty = tcy + tsy, tby = tcy - tsy, tlx = tcx - tsx, trx = tcx + tsx;
  const int cyi = threadIdx.y + KS, cxi = threadIdx.x + KS;
  const float inf = __int_as_float(0x7f800000);
  float depth_t = tile[cyi + 1][cxi], depth_bb = tile[cyi - 1][cxi], depth_l = tile[cyi][cxi - 1], depth_r = tile[cyi][cxi + 1];
  depth_t = (depth_t == inf) ? depth : depth_t;            // is_outside(neighbour) ? depth : neighbour
  depth_bb = (depth_bb == inf) ? depth : depth_bb;
  depth_l = (depth_l == inf) ? depth : depth_l;
  depth_r = (depth_r == inf) ? depth : depth_r;
  const float3 world_t = tex3d_xyz(xyz, CX, CY, CZ, tcx, tty, depth_t);
  const float3 world_b = tex3d_xyz(xyz, CX, CY, CZ, tcx, tby, depth_bb);
  const float3 world_l = tex3d_xyz(xyz, CX, CY, CZ, tlx, tcy, depth_l);
  const float3 world_r = tex3d_xyz(xyz, CX, CY, CZ, trx, tcy, depth_r);
  // ---- pre_quality.fs:65-119 (k_quality) ----
  const float dist_range_max = 0.35f * (depth / 1.0f);
  const float dist_range_max_inv = 1.0f / dist_range_max;
  float w_range = 0.0f, border = 0.0f;
  if (depth - depth == 0.0f) {
#pragma unroll
    for (int y = 0; y <= 2 * KS; ++y) {
#pragma unroll
      for (int x = 0; x <= 2 * KS; ++x) {
        const float depth_range = fabsf(tile[threadIdx.y + y][threadIdx.x + x] - depth);
        if (depth_range > dist_range_max) { border += 1.0f; continue; }
        w_range += 1.0f - depth_range * dist_range_max_inv;
      }
    }
  } else {
#pragma unroll 1
    for (int y = -KS; y <= KS; ++y) {
#pragma unroll 1
      for (int x = -KS; x <= KS; ++x) {
        const float depth_s = depth_b[base + (size_t)iclamp(py + y, 0, H - 1) * W + iclamp(px + x, 0, W - 1)].x;
        const float depth_range = fabsf(depth_s - depth);
        if ((depth_s <= 0.0f) || (depth_s >= 1.0f) || (depth_range > dist_range_max)) { border += 1.0f; continue; }
        w_range += 1.0f - gmin(depth_range, dist_range_max) * dist_range_max_inv;
      }
    }
  }
  const float3 n = normalize3(cross3(world_b - world_t, world_l - world_r));
  out_normal[o] = make_float4(n.x, n.y, n.z, 0.0f);
  const float lateral_quality = 1.0f - border / 169.0f;
  float q = gpow(lateral_quality, 6.0f);
  q *= gpow(w_range / 169.0f, 6.0f);
  q /= depth * 6.5f;
  const float3 cam = make_float3(st.cam[layer][0], st.cam[layer][1], st.cam[layer][2]);
  const float angle = dot3(normalize3(cam - world), n);
  q *= gpow(angle, 2.0f);
  emit(q);
}

// ------------------------------------------------------------------------------------------------ gather texels
// Entry (ex, ey) in [0,W]x[0,H] serves the bilinear footprint whose unclamped lower-left texel is (ex-1, ey-1):
//   .lo = depth_b.x at (x0,y0) (x1,y0) (x0,y1) (x1,y1);  .hi = quality at the same taps with the silhouette
// (exactly 0 or 1, pre_boundary.fs:88-108) in the sign bit. quality is never negative (a product of pow() results
// and positive divisors), so the sign bit is free; violations are counted in flags[0].
__global__ void __launch_bounds__(256) k_pack_gather(const float2* __restrict__ depth_b, const float* __restrict__ quality,
                                                     const float* __restrict__ sil, float4* __restrict__ gather,
                                                     uint32_t* __restrict__ flags, int W, int H) {
  const int ex = blockIdx.x * TILE_X + threadIdx.x, ey = blockIdx.y * TILE_Y + threadIdx.y;
  if (ex > W || ey > H) return;
  const size_t base = (size_t)blockIdx.z * W * H;
  const int x0 = iclamp(ex - 1, 0, W - 1), x1 = iclamp(ex, 0, W - 1);
  const int y0 = iclamp(ey - 1, 0, H - 1), y1 = iclamp(ey, 0, H - 1);
  const size_t i00 = base + (size_t)y0 * W + x0, i10 = base + (size_t)y0 * W + x1;
  const size_t i01 = base + (size_t)y1 * W + x0, i11 = base + (size_t)y1 * W + x1;
  auto enc = [&](size_t i) -> float {
    const float q = quality[i];
    uint32_t b = __float_as_uint(q);
    if ((b >> 31) && !(q != q) && q != 0.0f) atomicAdd(flags, 1u);
    b &= 0x7fffffffu;
    if (sil[i] >= 1.0f) b |= 0x80000000u;
    return __uint_as_float(b);
  };
  const size_t go = (((size_t)blockIdx.z * (H + 1) + ey) * (W + 1) + ex) * 2;
  gather[go] = make_float4(depth_b[i00].x, depth_b[i10].x, depth_b[i01].x, depth_b[i11].x);
  gather[go + 1] = make_float4(enc(i00), enc(i10), enc(i01), enc(i11));
}

// ------------------------------------------------------------------------------------------------ host launcher
int launch_preprocess(rr_ctx* c, int filter_textures, int use_processed_depth, int refine) {
  const int N = c->N, W = c->W, H = c->H;
  const dim3 blk(TILE_X, TILE_Y, 1);
  const dim3 grd((W + TILE_X - 1) / TILE_X, (H + TILE_Y - 1) / TILE_Y, N);
  const SensorTables st = sensor_tables(c);
  cudaStream_t s = c->stream;
  RR_TRY_RC(staged_prepare(c));            // decides which integrator the frame set is packed for (no-op unless settings changed)
  timer_begin(c, "1preprocess");

  timer_begin(c, "morph");
  k_morph<<<grd, blk, 0, s>>>(c->d_depth_raw, c->d_morph.ptr, W, H);
  RR_LAUNCH_CHECK(c, "k_morph");
  timer_end(c, "morph");

  timer_begin(c, "bilateral");
  DepthParams dp{};
  for (int a = 0; a < 3; ++a) { dp.bmin[a] = c->bbox_min[a]; dp.bmax[a] = c->bbox_max[a]; }
  dp.filter_textures = filter_textures;
  for (int i = 0; i < N; ++i) {
    // NetKinectArray.cpp:345-351: compress, scale = far - near, near, scaled_near = scale / 255
    dp.compress[i] = c->depth_format == RR_DEPTH_U8 ? 1 : 0;
    dp.near_[i] = c->depth_near[i];
    dp.scale[i] = c->depth_far[i] - c->depth_near[i];
    dp.scaled_near[i] = dp.scale[i] / 255.0f;
  }
  k_bilateral<<<grd, blk, 0, s>>>(use_processed_depth ? c->d_morph.ptr : c->d_depth_raw, c->d_color, c->d_depth.ptr, c->d_lab.ptr,
                                  W, H, c->CW, c->CH, st, dp);
  RR_LAUNCH_CHECK(c, "k_bilateral");
  timer_end(c, "bilateral");

  timer_begin(c, "boundary");
  k_boundary<<<grd, blk, 0, s>>>(c->d_depth.ptr, c->d_lab.ptr, c->d_depth_b.ptr, c->d_sil.ptr, W, H, refine);
  RR_LAUNCH_CHECK(c, "k_boundary");
  timer_end(c, "boundary");

  BrickParams bp{};
  for (int a = 0; a < 3; ++a) { bp.bmin[a] = c->bbox_min[a]; bp.res[a] = c->bricks.res[a]; }
  bp.brick_size = c->bricks.brick_size;
  bp.num = c->bricks.num;
  // The staged integrator reads the pair image k_quality writes on its way out; the 32-byte gather texels of the direct
  // kernels (dense mode, configurations the staged kernel declines) cost one more pass and are built only when needed.
  const bool staged = staged_selected(c);
  c->sti.lists_key = 0;                    // the item lists describe the previous pair image
  c->gather_packed = false;
  if (tunables().fuse_nq) {
    timer_begin(c, "quality");
    k_normal_quality<<<grd, blk, 0, s>>>(c->d_depth_b.ptr, c->d_normal.ptr, c->d_counters.ptr, c->d_quality.ptr, c->d_sil.ptr, c->d_pairs.ptr, c->pair_pitch,
                                         c->d_flags.ptr, W, H, st, bp);
    RR_LAUNCH_CHECK(c, "k_normal_quality");
  } else {
    timer_begin(c, "normal");
    k_normal<<<grd, blk, 0, s>>>(c->d_depth_b.ptr, c->d_normal.ptr, c->d_counters.ptr, W, H, st, bp);
    RR_LAUNCH_CHECK(c, "k_normal");
    timer_end(c, "normal");
    timer_begin(c, "quality");
    k_quality<<<grd, blk, 0, s>>>(c->d_depth_b.ptr, c->d_normal.ptr, c->d_quality.ptr, c->d_sil.ptr, c->d_pairs.ptr, c->pair_pitch, c->d_flags.ptr, W, H, st);
    RR_LAUNCH_CHECK(c, "k_quality");
  }
  if (!staged) RR_TRY_RC(launch_pack_gather(c));
  timer_end(c, "quality");

  timer_end(c, "1preprocess");
  return RR_OK;
}

int launch_pack_gather(rr_ctx* c) {
  const dim3 blk(TILE_X, TILE_Y, 1);
  const dim3 grd_g((c->W + 1 + TILE_X - 1) / TILE_X, (c->H + 1 + TILE_Y - 1) / TILE_Y, c->N);
  k_pack_gather<<<grd_g, blk, 0, c->stream>>>(c->d_depth_b.ptr, c->d_quality.ptr, c->d_sil.ptr, c->d_gather.ptr, c->d_flags.ptr, c->W, c->H);
  RR_LAUNCH_CHECK(c, "k_pack_gather");
  c->gather_packed = true;
  return RR_OK;
}

}  // namespace rr
