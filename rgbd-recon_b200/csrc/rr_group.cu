// rr_group: one process, several GPUs (SURVEY.md §8e). The reference has no multi-GPU path; its single GL context does the
// whole of kinect_client.cpp:572-617 per frame. Here the TSDF volume is split into contiguous z-slabs, one rr_ctx per device:
//   * a frame set goes host -> the ingest device (member 0) -> every other member by peer copies over NVLink, down a binary
//     tree of members (cudaMemcpyPeerAsync on the members' copy streams, double-buffered like rr_stage_frames: the copies
//     of frame set i+1 overlap the kernels of frame set i);
//   * pre-processing and the brick tables are replicated (identical on every member, no exchange), integration is per slab
//     (plus a halo recomputed locally, rr_integrate);
//   * a view is marched per slab; ONE kernel on the display device (member 0) composites it, reading the other members'
//     first-hit keys (4 bytes per pixel and member) and only the winner's colour / depth / sample count through peer
//     memory - the exchange happens inside the kernel, pixel by pixel, instead of gathering whole record images.
// In one process no collective library is needed: the "broadcast" is N-1 peer copies, the "gather" a kernel's loads.
// The multi-process form of the same path (one rank per GPU, NCCL) is what bench.py drives through rrpy/multigpu.py.
#include "rr_context.h"

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

struct rr_group {
  std::vector<rr_ctx*> m;
  std::vector<int> dev;
  std::vector<char> peer;              // member 0's kernels may load from member i's memory
  std::string error;
  // fallback for members member 0 cannot address: their view is copied into these (device 0) before compositing
  struct FallbackView { rr::DeviceArray<uint32_t> step; rr::DeviceArray<float4> rgba; rr::DeviceArray<float> zbuf, nsamp; };
  std::vector<FallbackView> fallback;  // per member
  size_t f_pixels = 0;
  std::vector<cudaEvent_t> ev_view;    // member i's view (or its fallback copy) is complete
  std::vector<cudaEvent_t> ev_copied[2];   // [slot][i]: member i has copied its parent's frame slot `slot` (the parent may overwrite it)
  std::vector<uint32_t> bounds;        // slab boundaries [n + 1]
};

namespace rr {

struct PeerViews {
  const uint32_t* step[RR_MAX_GROUP];
  const float4* rgba[RR_MAX_GROUP];
  const float* zbuf[RR_MAX_GROUP];
  const float* nsamp[RR_MAX_GROUP];
  int n;
};

// tsdf_raymarch.fs:92-142 finds ONE first hit per ray; with the ray's samples split over slabs that is the member whose
// first hit has the smallest step index (lowest member on ties, as k_composite). Member 0's images are also the output.
__global__ void __launch_bounds__(256) k_composite_peers(const __grid_constant__ PeerViews pv, int n, float4* __restrict__ rgba,
                                                         float* __restrict__ depth, uint32_t* __restrict__ step, float* __restrict__ nsamp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t keys[RR_MAX_GROUP];
#pragma unroll
  for (int p = 0; p < RR_MAX_GROUP; ++p) keys[p] = p < pv.n ? pv.step[p][i] : 0xffffffffu;      // all loads in flight at once
  int best = 0;
  uint32_t best_step = keys[0];
#pragma unroll
  for (int p = 1; p < RR_MAX_GROUP; ++p)
    if (keys[p] < best_step) { best_step = keys[p]; best = p; }
  if (best != 0) {                     // member 0 wins: its images already are the output
    const float4 c = pv.rgba[best][i];
    const float d = pv.zbuf[best][i], s = pv.nsamp[best][i];
    rgba[i] = c; depth[i] = d; step[i] = best_step; nsamp[i] = s;
  }
}

}  // namespace rr

namespace {

int gfail(rr_group* g, int code, const std::string& msg) {
  if (g) g->error = msg;
  return code;
}
int member_fail(rr_group* g, size_t i, int code) {
  return gfail(g, code, "member " + std::to_string(i) + " (device " + std::to_string(g->dev[i]) + "): " + rr_last_error(g->m[i]));
}
int gcheck(rr_group* g, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return RR_OK;
  return gfail(g, RR_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

}  // namespace

#define RR_G_REQUIRE(g, cond, msg) do { if (!(cond)) return gfail((g), RR_ERR_INVALID, (msg)); } while (0)
#define RR_G_ALL(g, call)                                                    \
  do {                                                                       \
    for (size_t i__ = 0; i__ < (g)->m.size(); ++i__) {                       \
      rr_ctx* ctx = (g)->m[i__];                                             \
      const int rc__ = (call);                                               \
      if (rc__ != RR_OK) return member_fail((g), i__, rc__);                 \
    }                                                                        \
  } while (0)
#define RR_G_TRY(g, expr) do { const int rc__ = gcheck((g), (expr), #expr); if (rc__ != RR_OK) return rc__; } while (0)
#define RR_G_TRY_RC(expr) do { const int rc__ = (expr); if (rc__ != RR_OK) return rc__; } while (0)

extern "C" {

int rr_group_create(rr_group** out, const int* devices, int n_devices, int num_sensors, int depth_w, int depth_h, int color_w, int color_h) {
  if (!out || !devices || n_devices < 1 || n_devices > RR_MAX_GROUP) return RR_ERR_INVALID;
  *out = nullptr;
  rr_group* g = new rr_group();
  for (int i = 0; i < n_devices; ++i) {
    rr_ctx* c = nullptr;
    const int rc = rr_create(&c, devices[i], num_sensors, depth_w, depth_h, color_w, color_h);
    if (rc != RR_OK) {
      for (rr_ctx* m : g->m) rr_destroy(m);
      delete g;
      return rc;
    }
    g->m.push_back(c); g->dev.push_back(devices[i]);
  }
  // member 0 composites: let its kernels address the other members' memory where the hardware allows it
  g->peer.assign(n_devices, 0);
  g->peer[0] = 1;
  cudaSetDevice(devices[0]);
  for (int i = 1; i < n_devices; ++i) {
    if (devices[i] == devices[0]) { g->peer[i] = 1; continue; }
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, devices[0], devices[i]) == cudaSuccess && can) {
      const cudaError_t e = cudaDeviceEnablePeerAccess(devices[i], 0);
      if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) g->peer[i] = 1;
    }
    cudaGetLastError();
  }
  // Frame sets travel down a binary tree of members (member i copies from member (i - 1) / 2, so no device serves more than
  // two copies of a set): peer access in both directions along every edge, so that the copies go device to device over
  // NVLink (without peer access cudaMemcpyPeerAsync stages through host memory)
  for (int i = 1; i < n_devices; ++i) {
    const int a = devices[i], b = devices[(i - 1) / 2];
    if (a == b) continue;
    int can = 0;
    cudaSetDevice(a);
    if (cudaDeviceCanAccessPeer(&can, a, b) == cudaSuccess && can) cudaDeviceEnablePeerAccess(b, 0);
    cudaGetLastError();
    cudaSetDevice(b);
    if (cudaDeviceCanAccessPeer(&can, b, a) == cudaSuccess && can) cudaDeviceEnablePeerAccess(a, 0);
    cudaGetLastError();
  }
  g->ev_view.assign(n_devices, nullptr);
  g->ev_copied[0].assign(n_devices, nullptr); g->ev_copied[1].assign(n_devices, nullptr);
  for (int i = 0; i < n_devices; ++i) {
    cudaSetDevice(devices[i]);
    cudaEventCreateWithFlags(&g->ev_view[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&g->ev_copied[0][i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&g->ev_copied[1][i], cudaEventDisableTiming);
  }
  g->fallback = std::vector<rr_group::FallbackView>(n_devices);
  *out = g;
  return RR_OK;
}

void rr_group_destroy(rr_group* g) {
  if (!g) return;
  for (size_t i = 0; i < g->m.size(); ++i) {
    cudaSetDevice(g->dev[i]);
    cudaStreamSynchronize(g->m[i]->stream);
    cudaStreamSynchronize(g->m[i]->copy_stream);
    if (g->ev_view[i]) cudaEventDestroy(g->ev_view[i]);
    for (int b = 0; b < 2; ++b) if (g->ev_copied[b][i]) cudaEventDestroy(g->ev_copied[b][i]);
  }
  cudaSetDevice(g->dev[0]);
  g->fallback.clear();
  for (rr_ctx* c : g->m) rr_destroy(c);
  delete g;
}

int rr_group_size(const rr_group* g) { return g ? (int)g->m.size() : 0; }
rr_ctx* rr_group_member(rr_group* g, int i) { return (g && i >= 0 && i < (int)g->m.size()) ? g->m[i] : nullptr; }
const char* rr_group_last_error(const rr_group* g) { return g ? g->error.c_str() : "null group"; }

int rr_group_synchronize(rr_group* g) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_synchronize(ctx));
  return RR_OK;
}

/* ---- replicated setup ------------------------------------------------------------------------------------------ */
int rr_group_set_bbox(rr_group* g, const float bbox_min[3], const float bbox_max[3]) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_set_bbox(ctx, bbox_min, bbox_max));
  return RR_OK;
}
int rr_group_calib_upload(rr_group* g, int sensor, const float* cv_xyz, const float* cv_uv, const uint32_t res[3], const float depth_limits[2]) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_calib_upload(ctx, sensor, cv_xyz, cv_uv, res, depth_limits));
  return RR_OK;
}
int rr_group_calib_upload_inv(rr_group* g, int sensor, const float* cv_xyz_inv, const uint32_t res[3]) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_calib_upload_inv(ctx, sensor, cv_xyz_inv, res));
  return RR_OK;
}
int rr_group_set_frame_format(rr_group* g, int color_format, int depth_format, const float* near_far) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_set_frame_format(ctx, color_format, depth_format, near_far));
  return RR_OK;
}
int rr_group_set_timing(rr_group* g, int level) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_set_timing(ctx, level));
  return RR_OK;
}

int rr_group_set_slabs(rr_group* g, const uint32_t* z_bounds) {
  if (!g) return RR_ERR_INVALID;
  RR_G_REQUIRE(g, z_bounds, "rr_group_set_slabs: null bounds");
  const size_t n = g->m.size();
  uint32_t res[3];
  if (rr_get_volume_res(g->m[0], res) != RR_OK) return member_fail(g, 0, RR_ERR_INVALID);
  RR_G_REQUIRE(g, z_bounds[0] == 0 && z_bounds[n] == res[2], "rr_group_set_slabs: the slabs must tile [0, Z)");
  for (size_t i = 0; i < n; ++i) RR_G_REQUIRE(g, z_bounds[i] < z_bounds[i + 1], "rr_group_set_slabs: empty or unordered slab");
  for (size_t i = 0; i < n; ++i) {
    const int rc = rr_set_slab(g->m[i], z_bounds[i], z_bounds[i + 1]);
    if (rc != RR_OK) return member_fail(g, i, rc);
  }
  g->bounds.assign(z_bounds, z_bounds + n + 1);
  return RR_OK;
}

int rr_group_get_slabs(const rr_group* g, uint32_t* z_bounds) {
  if (!g || !z_bounds || g->bounds.size() != g->m.size() + 1) return RR_ERR_INVALID;
  std::memcpy(z_bounds, g->bounds.data(), g->bounds.size() * sizeof(uint32_t));
  return RR_OK;
}

int rr_group_configure(rr_group* g, const rr_config* cfg) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_configure(ctx, cfg));
  // equal-thickness slabs to start with (the remainder spread over the first members); rr_group_balance_slabs refines them
  uint32_t res[3];
  if (rr_get_volume_res(g->m[0], res) != RR_OK) return member_fail(g, 0, RR_ERR_INVALID);
  const uint32_t n = (uint32_t)g->m.size();
  RR_G_REQUIRE(g, res[2] >= n, "rr_group_configure: fewer z slices than devices");
  std::vector<uint32_t> b(n + 1, 0);
  for (uint32_t i = 0; i < n; ++i) b[i + 1] = b[i] + res[2] / n + (i < res[2] % n ? 1u : 0u);
  return rr_group_set_slabs(g, b.data());
}

// Slabs of (nearly) equal integrate cost from the occupied bricks of the last fused frame set: occupied bricks cluster
// around the captured subject, so equal-thickness slabs leave the outer members idle. Cost of slice z = X*Y (the clear
// stream) + compute_to_fill * (voxels of occupied bricks in the slice). Every member holds the same brick tables, so the
// boundaries follow from member 0's alone. Synchronises; call it now and then, not per frame.
int rr_group_balance_slabs(rr_group* g, float compute_to_fill) {
  if (!g) return RR_ERR_INVALID;
  rr_ctx* c0 = g->m[0];
  uint32_t res[3], nb = 0, n_occ = 0;
  if (rr_get_volume_res(c0, res) != RR_OK || rr_get_brick_info(c0, nullptr, nullptr, &nb) != RR_OK) return member_fail(g, 0, RR_ERR_INVALID);
  const uint32_t n = (uint32_t)g->m.size(), Z = res[2];
  if (n == 1 || nb == 0) return RR_OK;
  std::vector<uint32_t> occ(nb);
  std::vector<int32_t> ranges((size_t)nb * 6);
  int rc = rr_download_bricks(c0, nullptr, occ.data(), &n_occ);
  if (rc == RR_OK) rc = rr_get_brick_ranges(c0, ranges.data());
  if (rc != RR_OK) return member_fail(g, 0, rc);
  if (compute_to_fill <= 0.0f) compute_to_fill = 45.0f;
  std::vector<double> cost(Z, (double)res[0] * res[1]);
  for (uint32_t k = 0; k < n_occ; ++k) {
    const int32_t* r = ranges.data() + (size_t)occ[k] * 6;
    const double area = (double)(r[1] - r[0]) * (r[3] - r[2]);
    for (int z = std::max(0, r[4]); z < std::min((int)Z, r[5]); ++z) cost[z] += (double)compute_to_fill * area;
  }
  std::vector<double> cum(Z + 1, 0.0);
  for (uint32_t z = 0; z < Z; ++z) cum[z + 1] = cum[z] + cost[z];
  // A member also integrates a halo on either side of its slab (rr_integrate), which weighs heavily on thin slabs: the cost
  // of a slab is the cost of slab + halo, and the boundaries minimise the largest one (bisection on the bound, greedy fill).
  const uint32_t h = (uint32_t)std::ceil(c0->cfg.limit * (float)Z) + 2u;
  auto slab_cost = [&](uint32_t z0, uint32_t z1) { return cum[std::min(Z, z1 + h)] - cum[z0 > h ? z0 - h : 0u]; };
  auto fill = [&](double bound, std::vector<uint32_t>& out) {
    out.assign(1, 0u);
    while (out.back() < Z) {
      if (out.size() > n) return false;
      const uint32_t z0 = out.back();
      uint32_t z1 = z0 + 1;
      while (z1 < Z && slab_cost(z0, z1 + 1) <= bound) ++z1;
      out.push_back(z1);
    }
    return true;
  };
  double lo = 0.0, hi = cum[Z];
  std::vector<uint32_t> b;
  for (int it = 0; it < 60; ++it) {
    const double mid = 0.5 * (lo + hi);
    if (fill(mid, b)) hi = mid; else lo = mid;
  }
  fill(hi, b);
  while (b.size() - 1 < n) {             // fewer slabs than members (tiny volumes): split the thickest
    size_t k = 0;
    for (size_t i = 0; i + 1 < b.size(); ++i) if (b[i + 1] - b[i] > b[k + 1] - b[k]) k = i;
    if (b[k + 1] - b[k] < 2) return gfail(g, RR_ERR_INVALID, "rr_group_balance_slabs: fewer z slices than devices");
    b.insert(b.begin() + (long)k + 1, (b[k] + b[k + 1]) / 2);
  }
  return rr_group_set_slabs(g, b.data());
}

/* ---- per frame ------------------------------------------------------------------------------------------------- */
// member c takes the frame set member s has just staged (the same back slot parity everywhere: members are only ever
// staged and swapped together)
// member `self` is about to overwrite its back slot t: its children in the tree must have finished copying the frame set that
// slot held (waiting on an event that was never recorded is a no-op)
static int wait_for_children(rr_group* g, size_t self, int t) {
  rr_ctx* c = g->m[self];
  for (size_t child = 2 * self + 1; child <= 2 * self + 2 && child < g->m.size(); ++child)
    RR_G_TRY(g, cudaStreamWaitEvent(c->copy_stream, g->ev_copied[t][child], 0));
  return RR_OK;
}

static int stage_from_peer(rr_group* g, size_t self, bool color, size_t cb, size_t db) {
  rr_ctx* c = g->m[self];
  rr_ctx* s = g->m[(self - 1) / 2];
  RR_G_TRY(g, cudaSetDevice(c->device));
  const int t = c->cur_slot ^ 1, ts = s->cur_slot ^ 1;
  if (c->free_recorded[t]) RR_G_TRY(g, cudaStreamWaitEvent(c->copy_stream, c->ev_free[t], 0));
  RR_G_TRY_RC(wait_for_children(g, self, t));
  RR_G_TRY(g, cudaStreamWaitEvent(c->copy_stream, s->ev_staged, 0));
  void* dd = c->depth_format == RR_DEPTH_U8 ? (void*)c->d_depth_packed[t].ptr : (void*)c->d_depth_slot[t].ptr;
  const void* sd = s->depth_format == RR_DEPTH_U8 ? (const void*)s->d_depth_packed[ts].ptr : (const void*)s->d_depth_slot[ts].ptr;
  RR_G_TRY(g, cudaMemcpyPeerAsync(dd, c->device, sd, s->device, db, c->copy_stream));
  if (color) {
    void* dc = c->color_format != RR_COLOR_RGB8 ? (void*)c->d_color_packed[t].ptr : (void*)c->d_color_slot[t].ptr;
    const void* sc = s->color_format != RR_COLOR_RGB8 ? (const void*)s->d_color_packed[ts].ptr : (const void*)s->d_color_slot[ts].ptr;
    RR_G_TRY(g, cudaMemcpyPeerAsync(dc, c->device, sc, s->device, cb, c->copy_stream));
  }
  c->staged_color = color;
  RR_G_TRY(g, cudaEventRecord(c->ev_staged, c->copy_stream));
  RR_G_TRY(g, cudaEventRecord(g->ev_copied[ts][self], c->copy_stream));
  c->staged = true;
  return RR_OK;
}

int rr_group_stage_frames(rr_group* g, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes) {
  if (!g) return RR_ERR_INVALID;
  rr_ctx* c0 = g->m[0];
  // the ingest device's back slot was the source of its children's copies two frame sets ago: they must have drained before
  // it is overwritten (per slot, so this host->device copy overlaps the deeper levels' copies of the previous frame set)
  RR_G_TRY(g, cudaSetDevice(c0->device));
  int rc = wait_for_children(g, 0, c0->cur_slot ^ 1);
  if (rc != RR_OK) return rc;
  rc = rr_stage_frames(c0, color, color_bytes, depth, depth_bytes);
  if (rc != RR_OK) return member_fail(g, 0, rc);
  // down the tree: a member's copy waits for its parent's (ev_staged of the parent), ascending order issues parents first
  for (size_t i = 1; i < g->m.size(); ++i) {
    rc = stage_from_peer(g, i, color != nullptr, color_bytes, depth_bytes);
    if (rc != RR_OK) return rc;
  }
  return RR_OK;
}

int rr_group_swap_frames(rr_group* g) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_swap_frames(ctx));
  return RR_OK;
}
int rr_group_stage_sync(rr_group* g) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_stage_sync(g->m[0]);          // the host buffers are read by the ingest device only
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}
int rr_group_upload_frames(rr_group* g, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_group_stage_frames(g, color, color_bytes, depth, depth_bytes);
  return rc == RR_OK ? rr_group_swap_frames(g) : rc;
}
int rr_group_bricks_clear(rr_group* g) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_bricks_clear(ctx));
  return RR_OK;
}
int rr_group_preprocess(rr_group* g, int filter_textures, int use_processed_depth, int refine_boundary) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_preprocess(ctx, filter_textures, use_processed_depth, refine_boundary));
  return RR_OK;
}
int rr_group_bricks_update(rr_group* g, uint32_t* out_num_occupied, float* out_ratio) {
  if (!g) return RR_ERR_INVALID;
  for (size_t i = 1; i < g->m.size(); ++i) {
    const int rc = rr_bricks_update(g->m[i], nullptr, nullptr);
    if (rc != RR_OK) return member_fail(g, i, rc);
  }
  const int rc = rr_bricks_update(g->m[0], out_num_occupied, out_ratio);       // identical on every member
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}
int rr_group_integrate(rr_group* g) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_integrate(ctx));
  return RR_OK;
}
int rr_group_fuse_frame(rr_group* g, int filter_textures, int use_processed_depth, int refine_boundary) {
  if (!g) return RR_ERR_INVALID;
  RR_G_ALL(g, rr_fuse_frame(ctx, filter_textures, use_processed_depth, refine_boundary));
  return RR_OK;
}
int rr_group_bricks_count(rr_group* g, uint32_t* out_num_occupied, float* out_ratio) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_bricks_count(g->m[0], out_num_occupied, out_ratio);
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

int rr_group_raymarch(rr_group* g, const rr_view* view, float* out_rgba, float* out_depth) {
  if (!g) return RR_ERR_INVALID;
  RR_G_REQUIRE(g, view && view->viewport[2] > 0 && view->viewport[3] > 0, "rr_group_raymarch: bad view");
  const size_t n = g->m.size();
  if (n == 1) {
    const int rc = rr_raymarch(g->m[0], view, out_rgba, out_depth);
    return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
  }
  const size_t px = (size_t)view->viewport[2] * view->viewport[3];
  rr_ctx* c0 = g->m[0];
  // every member marches the samples of its own slab (rr_set_slab) into its own view images
  RR_G_ALL(g, rr_raymarch(ctx, view, nullptr, nullptr));
  rr::PeerViews pv{};
  pv.n = (int)n;
  for (size_t i = 0; i < n; ++i) {
    rr_ctx* c = g->m[i];
    if (i > 0 && !g->peer[i]) {
      // no peer addressing between the two devices: copy the member's view to the display device first
      rr_group::FallbackView& f = g->fallback[i];
      if (g->f_pixels < px || !f.step.ptr) {
        RR_G_TRY(g, cudaSetDevice(c0->device));
        int rc = f.step.allocate(c0, px, "group view steps");
        if (rc == RR_OK) rc = f.rgba.allocate(c0, px, "group view rgba");
        if (rc == RR_OK) rc = f.zbuf.allocate(c0, px, "group view depth");
        if (rc == RR_OK) rc = f.nsamp.allocate(c0, px, "group view samples");
        if (rc != RR_OK) return member_fail(g, 0, rc);
      }
      RR_G_TRY(g, cudaSetDevice(c->device));
      RR_G_TRY(g, cudaMemcpyPeerAsync(f.step.ptr, c0->device, c->d_step.ptr, c->device, px * sizeof(uint32_t), c->stream));
      RR_G_TRY(g, cudaMemcpyPeerAsync(f.rgba.ptr, c0->device, c->d_rgba.ptr, c->device, px * sizeof(float4), c->stream));
      RR_G_TRY(g, cudaMemcpyPeerAsync(f.zbuf.ptr, c0->device, c->d_zbuf.ptr, c->device, px * sizeof(float), c->stream));
      RR_G_TRY(g, cudaMemcpyPeerAsync(f.nsamp.ptr, c0->device, c->d_nsamples.ptr, c->device, px * sizeof(float), c->stream));
      pv.step[i] = f.step.ptr; pv.rgba[i] = f.rgba.ptr; pv.zbuf[i] = f.zbuf.ptr; pv.nsamp[i] = f.nsamp.ptr;
    } else {
      pv.step[i] = c->d_step.ptr; pv.rgba[i] = c->d_rgba.ptr; pv.zbuf[i] = c->d_zbuf.ptr; pv.nsamp[i] = c->d_nsamples.ptr;
    }
    if (i > 0) {
      RR_G_TRY(g, cudaSetDevice(c->device));
      RR_G_TRY(g, cudaEventRecord(g->ev_view[i], c->stream));
    }
  }
  bool grew = false;
  for (size_t i = 1; i < n; ++i) grew = grew || !g->peer[i];
  if (grew) g->f_pixels = std::max(g->f_pixels, px);
  RR_G_TRY(g, cudaSetDevice(c0->device));
  for (size_t i = 1; i < n; ++i) RR_G_TRY(g, cudaStreamWaitEvent(c0->stream, g->ev_view[i], 0));
  rr::timer_begin(c0, "composite");
  rr::k_composite_peers<<<(unsigned)((px + 255) / 256), 256, 0, c0->stream>>>(pv, (int)px, c0->d_rgba.ptr, c0->d_zbuf.ptr, c0->d_step.ptr, c0->d_nsamples.ptr);
  ++c0->launches;
  RR_G_TRY(g, cudaGetLastError());
  rr::timer_end(c0, "composite");
  // the other members must not start their next view (overwriting the images the kernel reads) before it has finished
  RR_G_TRY(g, cudaEventRecord(g->ev_view[0], c0->stream));
  for (size_t i = 1; i < n; ++i) {
    RR_G_TRY(g, cudaSetDevice(g->dev[i]));
    RR_G_TRY(g, cudaStreamWaitEvent(g->m[i]->stream, g->ev_view[0], 0));
  }
  RR_G_TRY(g, cudaSetDevice(c0->device));
  const int rc = rr::view_download(c0, out_rgba, out_depth, "rr_group_raymarch");
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

int rr_group_fill_colors(rr_group* g, float* out_rgba) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_fill_colors(g->m[0], out_rgba);            // on the composited view of the display device
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

/* ---- the same compositing across processes (one process per GPU): the peers' view images through CUDA IPC --------------- */
int ensure_view(rr_ctx* c, int w, int h);      // rr_api.cu (same linkage block)

int rr_view_export(rr_ctx* c, int width, int height, void* out_handle) {
  if (!c) return RR_ERR_INVALID;
  if (!out_handle || width <= 0 || height <= 0) return rr::fail(c, RR_ERR_INVALID, "rr_view_export: bad arguments");
  if (cudaSetDevice(c->device) != cudaSuccess) return rr::check(c, cudaGetLastError(), "rr_view_export");
  RR_TRY_RC(ensure_view(c, width, height));
  cudaIpcMemHandle_t h[4];
  static_assert(sizeof(h) == RR_VIEW_HANDLE_BYTES, "four IPC handles");
  void* ptrs[4] = {c->d_step.ptr, c->d_rgba.ptr, c->d_zbuf.ptr, c->d_nsamples.ptr};
  for (int i = 0; i < 4; ++i) {
    const cudaError_t e = cudaIpcGetMemHandle(&h[i], ptrs[i]);
    if (e != cudaSuccess) return rr::check(c, e, "rr_view_export: cudaIpcGetMemHandle");
  }
  std::memcpy(out_handle, h, sizeof(h));
  return RR_OK;
}

int rr_composite_peers(rr_ctx* c, const void* peer_handles, int n_peers, int width, int height, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  if (n_peers < 0 || n_peers >= RR_MAX_GROUP || (n_peers > 0 && !peer_handles) || width != c->view_w || height != c->view_h || !c->d_step.ptr)
    return rr::fail(c, RR_ERR_INVALID, "rr_composite_peers: march this context's own view at this size first; at most 15 peers");
  if (cudaSetDevice(c->device) != cudaSuccess) return rr::check(c, cudaGetLastError(), "rr_composite_peers");
  rr::PeerViews pv{};
  pv.n = n_peers + 1;
  pv.step[0] = c->d_step.ptr; pv.rgba[0] = c->d_rgba.ptr; pv.zbuf[0] = c->d_zbuf.ptr; pv.nsamp[0] = c->d_nsamples.ptr;
  for (int p = 0; p < n_peers; ++p) {
    const std::string key(static_cast<const char*>(peer_handles) + (size_t)p * RR_VIEW_HANDLE_BYTES, RR_VIEW_HANDLE_BYTES);
    const rr_ctx::IpcView* v = nullptr;
    for (const auto& o : c->ipc_views) if (o.key == key) { v = &o; break; }
    if (!v) {
      cudaIpcMemHandle_t h[4];
      std::memcpy(h, key.data(), sizeof(h));
      void* ptrs[4] = {nullptr, nullptr, nullptr, nullptr};
      for (int i = 0; i < 4; ++i) {
        const cudaError_t e = cudaIpcOpenMemHandle(&ptrs[i], h[i], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
          for (int k = 0; k < i; ++k) cudaIpcCloseMemHandle(ptrs[k]);
          return rr::check(c, e, "rr_composite_peers: cudaIpcOpenMemHandle (handles come from rr_view_export in ANOTHER process)");
        }
      }
      c->ipc_views.push_back({key, (uint32_t*)ptrs[0], (float4*)ptrs[1], (float*)ptrs[2], (float*)ptrs[3]});
      v = &c->ipc_views.back();
    }
    pv.step[p + 1] = v->step; pv.rgba[p + 1] = v->rgba; pv.zbuf[p + 1] = v->zbuf; pv.nsamp[p + 1] = v->nsamp;
  }
  const size_t px = (size_t)width * height;
  rr::timer_begin(c, "composite");
  rr::k_composite_peers<<<(unsigned)((px + 255) / 256), 256, 0, c->stream>>>(pv, (int)px, c->d_rgba.ptr, c->d_zbuf.ptr, c->d_step.ptr, c->d_nsamples.ptr);
  RR_LAUNCH_CHECK(c, "k_composite_peers");
  rr::timer_end(c, "composite");
  return rr::view_download(c, out_rgba, out_depth, "rr_composite_peers");
}

// Member 0 receives every other member's owned slices by peer copies (one volume over NVLink per call), so that it holds
// the whole volume. Member 0's integrate and raymarch read only its slab and halo, and the halo slices equal the owners'
// bit for bit (integration is pure), so overwriting its unowned slices changes nothing it computes later. The caller works
// on member 0's stream and synchronises it before returning: the copies read the members' volumes, which must not
// integrate again before the copies are done.
// need_calib: refuse unless member 0 has every sensor's calibration volumes (the mesh's colours and normals read them).
static int group_gather_volume(rr_group* g, const std::string& who, bool need_calib) {
  RR_G_REQUIRE(g, g->bounds.size() == g->m.size() + 1, who + ": configure the group first");
  rr_ctx* c0 = g->m[0];
  for (size_t i = 0; i < g->m.size(); ++i) {
    rr_ctx* c = g->m[i];
    if (!c->configured || !c->volume_integrated)
      return gfail(g, RR_ERR_INVALID, who + ": nothing has been integrated into the current volume");
  }
  for (int s = 0; need_calib && s < c0->N; ++s)
    RR_G_REQUIRE(g, c0->have_calib[s] && c0->have_inv[s], who + ": upload every sensor's calibration volumes first");
  const size_t plane = (size_t)c0->res[0] * c0->res[1];
  for (size_t i = 1; i < g->m.size(); ++i) {
    rr_ctx* c = g->m[i];
    RR_G_TRY(g, cudaSetDevice(c->device));
    RR_G_TRY(g, cudaEventRecord(g->ev_view[i], c->stream));
    RR_G_TRY(g, cudaSetDevice(c0->device));
    RR_G_TRY(g, cudaStreamWaitEvent(c0->stream, g->ev_view[i], 0));
    const size_t z0 = g->bounds[i], z1 = g->bounds[i + 1];
    if (z1 > z0)
      RR_G_TRY(g, cudaMemcpyPeerAsync(c0->d_tsdf.ptr + plane * z0, c0->device, c->d_tsdf.ptr + plane * z0, c->device, plane * (z1 - z0) * sizeof(float), c0->stream));
  }
  c0->clear.valid = false;      // member 0's volume was written outside an integrate: its next integrate clears the whole slab
  RR_G_TRY(g, cudaSetDevice(c0->device));
  return RR_OK;
}

int rr_group_extract_mesh(rr_group* g, uint32_t* out_num_vertices, uint32_t* out_num_triangles) {
  if (!g) return RR_ERR_INVALID;
  rr_ctx* c0 = g->m[0];
  RR_TRY_RC(group_gather_volume(g, "rr_group_extract_mesh", true));
  const int rc = rr::launch_extract_mesh(c0, out_num_vertices, out_num_triangles);
  RR_G_TRY(g, cudaStreamSynchronize(c0->stream));
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

// The same gather, then member 0 labels the whole volume; read the parts with rr_download_parts(rr_group_member(g, 0), ...).
int rr_group_label_parts(rr_group* g, uint32_t* out_num_parts) {
  if (!g) return RR_ERR_INVALID;
  RR_G_REQUIRE(g, out_num_parts, "rr_group_label_parts: null count pointer");
  RR_TRY_RC(group_gather_volume(g, "rr_group_label_parts", false));
  const int rc = rr::launch_label_parts(g->m[0], rr::label_dest(g->m[0]), out_num_parts);
  RR_G_TRY(g, cudaStreamSynchronize(g->m[0]->stream));
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

// The same gather, then member 0 tracks the whole volume against its tracked labelling; read the tracks with
// rr_download_part_tracks(rr_group_member(g, 0), ...), reset them with rr_reset_part_tracks on member 0.
int rr_group_track_parts(rr_group* g, uint32_t min_voxels, uint32_t* out_num_parts, uint32_t* out_num_ended) {
  if (!g) return RR_ERR_INVALID;
  RR_G_REQUIRE(g, out_num_parts && out_num_ended, "rr_group_track_parts: null count pointer");
  RR_G_REQUIRE(g, min_voxels >= 1, "rr_group_track_parts: min_voxels must be at least 1");
  RR_TRY_RC(group_gather_volume(g, "rr_group_track_parts", false));
  const int rc = rr::launch_track_parts(g->m[0], min_voxels, out_num_parts, out_num_ended);
  RR_G_TRY(g, cudaStreamSynchronize(g->m[0]->stream));
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

// Right after rr_group_extract_mesh member 0 holds the gathered whole volume and the mesh: it simplifies, with no peer traffic.
int rr_group_simplify_mesh(rr_group* g, uint32_t cluster_voxels, uint32_t* out_num_vertices, uint32_t* out_num_triangles) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_simplify_mesh(g->m[0], cluster_voxels, out_num_vertices, out_num_triangles);
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

// Pre-processing is replicated on every member (rr_group_preprocess / rr_group_fuse_frame), so member 0's stage images are
// the whole frame set's: the cloud is extracted there, with no peer traffic.
int rr_group_extract_points(rr_group* g, uint32_t sensor_mask, uint32_t* out_num_points) {
  if (!g) return RR_ERR_INVALID;
  const int rc = rr_extract_points(g->m[0], sensor_mask, out_num_points);
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

// Queries: member 0 takes the caller's inputs, every other member peer-copies them from member 0 and evaluates what its
// slab owns (the halo covers the gradient and refinement taps), and one kernel on member 0 picks each entry's result from
// the members' arrays through peer memory. No volume moves.
static int group_query(rr_group* g, bool rays, int space, const float* a, const float* b, uint32_t count, float* out_a,
                       float* normals, float* rgba, uint32_t* steps) {
  const char* who = rays ? "rr_group_cast_rays" : "rr_group_sample_points";
  const size_t n = g->m.size();
  rr_ctx* c0 = g->m[0];
  if (n == 1) {
    const int rc = rays ? rr_cast_rays(c0, space, a, b, count, out_a, normals, rgba, steps) : rr_sample_points(c0, space, a, count, out_a, normals, rgba);
    return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
  }
  if (count == 0 && (space == RR_QUERY_WORLD || space == RR_QUERY_VOLUME)) return RR_OK;
  RR_G_REQUIRE(g, g->bounds.size() == n + 1, std::string(who) + ": configure the group first");
  for (size_t i = 0; i < n; ++i) {
    const int rc = rr::query_check(g->m[i], space, count, a && (!rays || b), false, who);
    if (rc != RR_OK) return member_fail(g, i, rc);
  }
  for (size_t i = 1; i < n; ++i)
    if (!g->peer[i])
      return gfail(g, RR_ERR_UNSUPPORTED, std::string(who) + ": member 0's device cannot address member " + std::to_string(i) + "'s memory");
  RR_G_TRY(g, cudaSetDevice(c0->device));
  int rc = rr::query_upload(c0, a, b, count);
  if (rc != RR_OK) return member_fail(g, 0, rc);
  RR_G_TRY(g, cudaEventRecord(g->ev_view[0], c0->stream));
  const size_t bytes = (size_t)count * (rays ? 6 : 3) * sizeof(float);
  for (size_t i = 0; i < n; ++i) {
    rr_ctx* c = g->m[i];
    RR_G_TRY(g, cudaSetDevice(c->device));
    if (i > 0) {
      rc = rr::query_reserve(c, count);
      if (rc != RR_OK) return member_fail(g, i, rc);
      RR_G_TRY(g, cudaStreamWaitEvent(c->stream, g->ev_view[0], 0));
      // the directions follow the origins at offset 3 * count in both members' input arrays
      RR_G_TRY(g, cudaMemcpyPeerAsync(c->d_q_in.ptr, c->device, c0->d_q_in.ptr, c0->device, bytes, c->stream));
    }
    rc = rays ? rr::launch_cast_rays(c, space, count) : rr::launch_sample_points(c, space, count);
    if (rc != RR_OK) return member_fail(g, i, rc);
    if (i > 0) RR_G_TRY(g, cudaEventRecord(g->ev_view[i], c->stream));
  }
  RR_G_TRY(g, cudaSetDevice(c0->device));
  for (size_t i = 1; i < n; ++i) RR_G_TRY(g, cudaStreamWaitEvent(c0->stream, g->ev_view[i], 0));
  rc = rr::launch_query_composite(g->m.data(), (int)n, rays, space, count);
  // the download synchronises member 0's stream: the composite has read the members' arrays before the call returns
  if (rc == RR_OK) rc = rr::query_download(c0, count, rays, out_a, normals, rgba, steps);
  return rc == RR_OK ? RR_OK : member_fail(g, 0, rc);
}

int rr_group_sample_points(rr_group* g, int space, const float* points, uint32_t count, float* values, float* normals, float* rgba) {
  if (!g) return RR_ERR_INVALID;
  return group_query(g, false, space, points, nullptr, count, values, normals, rgba, nullptr);
}

int rr_group_cast_rays(rr_group* g, int space, const float* origins, const float* directions, uint32_t count,
                       float* positions, float* normals, float* rgba, uint32_t* steps) {
  if (!g) return RR_ERR_INVALID;
  return group_query(g, true, space, origins, directions, count, positions, normals, rgba, steps);
}

// The whole volume, assembled from the slices each member owns. out: float32 [Z][Y][X], as rr_download_tsdf returns it
// (half2 voxels: the tsdf half widened to float).
int rr_group_download_tsdf(rr_group* g, float* out) {
  if (!g || !out) return RR_ERR_INVALID;
  uint32_t res[3];
  if (rr_get_volume_res(g->m[0], res) != RR_OK) return member_fail(g, 0, RR_ERR_INVALID);
  RR_G_REQUIRE(g, g->bounds.size() == g->m.size() + 1, "rr_group_download_tsdf: configure the group first");
  const size_t plane = (size_t)res[0] * res[1];
  for (size_t i = 0; i < g->m.size(); ++i) {
    rr_ctx* c = g->m[i];
    RR_G_TRY(g, cudaSetDevice(c->device));
    const size_t z0 = g->bounds[i], z1 = g->bounds[i + 1];
    RR_G_TRY(g, cudaMemcpyAsync(out + plane * z0, c->d_tsdf.ptr + plane * z0, plane * (z1 - z0) * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  }
  const int rc = rr_group_synchronize(g);
  if (rc != RR_OK || g->m[0]->cfg.store_weight != RR_VOXELS_HALF2) return rc;
  const size_t n = plane * res[2];
  for (size_t i = 0; i < n; ++i) {
    uint32_t u;
    std::memcpy(&u, out + i, sizeof(u));
    const __half h = __ushort_as_half((unsigned short)(u & 0xffffu));
    out[i] = __half2float(h);
  }
  return RR_OK;
}

}  // extern "C"
