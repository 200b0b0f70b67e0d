// C ABI of librr_b200.so (include/rgbd_recon_b200.h): context lifetime, uploads, settings, read-back, timing.
// There is no CPU fallback: without a CUDA device rr_create fails with RR_ERR_NO_DEVICE.
#include "rr_context.h"

#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

namespace rr {

int fail(rr_ctx* c, int code, const std::string& msg) {
  if (c) {
    std::lock_guard<std::mutex> lock(c->error_mutex);
    c->error = msg;
  }
  return code;
}

int check(rr_ctx* c, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return RR_OK;
  return fail(c, RR_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

void drop_frame_graphs(rr_ctx* c) {
  if (c->frame_graphs.empty()) return;
  cudaStreamSynchronize(c->stream);
  for (auto& g : c->frame_graphs) cudaGraphExecDestroy(g.exec);
  c->frame_graphs.clear();
}

static bool timer_is_top(const char* name) { return name[0] >= '0' && name[0] <= '9'; }   // "1preprocess", "2integrate", "3recon"

void timer_begin(rr_ctx* c, const char* name) {
  if (c->timing == 0 || (c->timing == 1 && !timer_is_top(name))) return;
  StageTimer& t = c->timers[name];
  if (t.used >= StageTimer::kMaxPending) {
    // fold the pending intervals (long since complete) into the running sum and reuse their events
    for (size_t i = 0; i < t.used; ++i) {
      float ms = 0.0f;
      if (cudaEventSynchronize(t.end[i]) == cudaSuccess && cudaEventElapsedTime(&ms, t.beg[i], t.end[i]) == cudaSuccess) {
        t.folded_ms += ms; ++t.folded_n; t.last_ms = ms;
      }
    }
    cudaGetLastError();
    t.used = 0;
  }
  if (t.used == t.beg.size()) {
    cudaEvent_t b, e;
    cudaEventCreate(&b); cudaEventCreate(&e);
    t.beg.push_back(b); t.end.push_back(e);
  }
  cudaEventRecord(t.beg[t.used], c->stream);
  t.open = true;
}

void timer_end(rr_ctx* c, const char* name) {
  if (c->timing == 0 || (c->timing == 1 && !timer_is_top(name))) return;
  auto it = c->timers.find(name);
  if (it == c->timers.end() || !it->second.open) return;
  StageTimer& t = it->second;
  cudaEventRecord(t.end[t.used], c->stream);
  ++t.used;
  t.open = false;
}

SensorTables sensor_tables(const rr_ctx* c) {
  SensorTables st{};
  for (int i = 0; i < c->N; ++i) {
    st.xyz[i] = c->d_xyz[i].ptr; st.uv[i] = c->d_uv[i].ptr;
    st.cx[i] = (int)c->cres[i][0]; st.cy[i] = (int)c->cres[i][1]; st.cz[i] = (int)c->cres[i][2];
    st.dmin[i] = c->dlim[i][0]; st.dmax[i] = c->dlim[i][1];
    for (int a = 0; a < 3; ++a) st.cam[i][a] = c->cam_pos[i][a];
  }
  return st;
}

// The read-back of a rendered view: rgba and / or depth of the current view, then one synchronise if either was asked for.
int view_download(rr_ctx* c, float* out_rgba, float* out_depth, const char* what) {
  const size_t n = (size_t)c->view_w * c->view_h;
  if (out_rgba) RR_TRY_RC(check(c, cudaMemcpyAsync(out_rgba, c->d_rgba.ptr, n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream), what));
  if (out_depth) RR_TRY_RC(check(c, cudaMemcpyAsync(out_depth, c->d_zbuf.ptr, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream), what));
  if (out_rgba || out_depth) RR_TRY_RC(check(c, cudaStreamSynchronize(c->stream), what));
  return RR_OK;
}

__global__ void k_pad_xyz(const float* __restrict__ src, float4* __restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = make_float4(src[i * 3], src[i * 3 + 1], src[i * 3 + 2], 0.0f);
}

__global__ void k_unpad3(const float4* __restrict__ src, float* __restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float4 v = src[i]; dst[i * 3] = v.x; dst[i * 3 + 1] = v.y; dst[i * 3 + 2] = v.z; }
}

}  // namespace rr

using namespace rr;

#define RR_REQUIRE(c, cond, msg) do { if (!(cond)) return fail((c), RR_ERR_INVALID, (msg)); } while (0)
#define RR_TRY(expr) do { int rc__ = (expr); if (rc__ != RR_OK) return rc__; } while (0)
#define RR_SET_DEVICE(c) do { cudaError_t e__ = cudaSetDevice((c)->device); if (e__ != cudaSuccess) return check((c), e__, "cudaSetDevice"); } while (0)

extern "C" {

int rr_version(void) { return 100; }

int rr_create(rr_ctx** out, int device, int num_sensors, int depth_w, int depth_h, int color_w, int color_h) {
  if (!out) return RR_ERR_INVALID;
  *out = nullptr;
  if (num_sensors < 1 || num_sensors > RR_MAX_SENSORS || depth_w < 1 || depth_h < 1 || color_w < 1 || color_h < 1) return RR_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return RR_ERR_NO_DEVICE;
  rr_ctx* c = new (std::nothrow) rr_ctx();
  if (!c) return RR_ERR_INVALID;
  c->device = device; c->N = num_sensors; c->W = depth_w; c->H = depth_h; c->CW = color_w; c->CH = color_h;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return RR_ERR_CUDA;
  }
  if (cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || c->num_sms < 1) c->num_sms = 148;
  const size_t px = (size_t)c->N * c->W * c->H;
  int rc = RR_OK;
  for (int b = 0; b < 2; ++b) {
    if (rc == RR_OK) rc = c->d_depth_slot[b].allocate(c, px, "depth");
    if (rc == RR_OK) rc = c->d_color_slot[b].allocate(c, (size_t)c->N * c->CW * c->CH * 3, "color");
    if (rc == RR_OK) rc = check(c, cudaEventCreateWithFlags(&c->ev_free[b], cudaEventDisableTiming), "event");
  }
  if (rc == RR_OK) rc = check(c, cudaEventCreateWithFlags(&c->ev_staged, cudaEventDisableTiming), "event");
  if (rc == RR_OK) rc = check(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking), "copy stream");
  c->d_depth_raw = c->d_depth_slot[0].ptr; c->d_color = c->d_color_slot[0].ptr;
  if (rc == RR_OK) rc = c->d_morph.allocate(c, px, "morph");
  if (rc == RR_OK) rc = c->d_depth.allocate(c, px, "depth rg");
  if (rc == RR_OK) rc = c->d_lab.allocate(c, px, "lab");
  if (rc == RR_OK) rc = c->d_depth_b.allocate(c, px, "depth_b");
  if (rc == RR_OK) rc = c->d_sil.allocate(c, px, "silhouette");
  if (rc == RR_OK) rc = c->d_normal.allocate(c, px, "normal");
  if (rc == RR_OK) rc = c->d_quality.allocate(c, px, "quality");
  if (rc == RR_OK) rc = c->d_gather.allocate(c, (size_t)c->N * (c->W + 1) * (c->H + 1) * 2, "gather");
  c->pair_pitch = (c->W + 3) & ~1;
  if (rc == RR_OK) rc = c->d_pairs.allocate(c, (size_t)c->N * (c->H + 2) * c->pair_pitch, "pair image");
  if (rc == RR_OK) rc = c->d_flags.allocate(c, 4, "flags");
  if (rc == RR_OK) rc = c->d_num_occ.allocate(c, 1, "num_occ");
  if (rc == RR_OK) rc = c->d_work.allocate(c, 8, "work counters");
  if (rc == RR_OK) rc = check(c, cudaMallocHost((void**)&c->pinned, sizeof(rr::PinnedScalars)), "pinned scalars");
  if (rc == RR_OK) {
    cudaMemsetAsync(c->d_flags.ptr, 0, 4 * sizeof(uint32_t), c->stream);
    cudaMemsetAsync(c->d_work.ptr, 0, 8 * sizeof(uint32_t), c->stream);
    cudaMemsetAsync(c->d_pairs.ptr, 0, (size_t)c->N * (c->H + 2) * c->pair_pitch * sizeof(float2), c->stream);
    cudaMemsetAsync(c->d_num_occ.ptr, 0, sizeof(uint32_t), c->stream);
    for (int b = 0; b < 2; ++b) {
      cudaMemsetAsync(c->d_color_slot[b].ptr, 0, (size_t)c->N * c->CW * c->CH * 3, c->stream);
      cudaMemsetAsync(c->d_depth_slot[b].ptr, 0, px * sizeof(float), c->stream);
    }
    c->pinned->num_occ = 0;
    rc = check(c, cudaStreamSynchronize(c->stream), "create sync");
  }
  if (rc != RR_OK) { rr_destroy(c); return rc; }
  *out = c;
  return RR_OK;
}

void rr_destroy(rr_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  drop_frame_graphs(c);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (int b = 0; b < 2; ++b) if (c->ev_free[b]) cudaEventDestroy(c->ev_free[b]);
  if (c->ev_staged) cudaEventDestroy(c->ev_staged);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (auto& v : c->ipc_views) { cudaIpcCloseMemHandle(v.step); cudaIpcCloseMemHandle(v.rgba); cudaIpcCloseMemHandle(v.zbuf); cudaIpcCloseMemHandle(v.nsamp); }
  cudaGetLastError();
  if (c->pinned) cudaFreeHost(c->pinned);
  for (auto& kv : c->timers) {
    for (cudaEvent_t e : kv.second.beg) cudaEventDestroy(e);
    for (cudaEvent_t e : kv.second.end) cudaEventDestroy(e);
  }
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;                    // the device arrays free their memory, on the context's device (current since the top)
}

const char* rr_last_error(const rr_ctx* c) {
  if (!c) return "null context";
  // a copy per calling thread: the text stays valid for the caller while another thread's call fails
  thread_local std::string text;
  {
    std::lock_guard<std::mutex> lock(const_cast<rr_ctx*>(c)->error_mutex);
    text = c->error;
  }
  return text.c_str();
}

int rr_synchronize(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaStreamSynchronize(c->copy_stream), "synchronize (copy stream)"));
  return check(c, cudaStreamSynchronize(c->stream), "synchronize");
}

void* rr_stream(rr_ctx* c) { return c ? (void*)c->stream : nullptr; }

int rr_set_bbox(rr_ctx* c, const float bmin[3], const float bmax[3]) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, bmin && bmax, "rr_set_bbox: null pointer");
  for (int a = 0; a < 3; ++a) {
    RR_REQUIRE(c, bmax[a] > bmin[a], "rr_set_bbox: empty box");
    c->bbox_min[a] = bmin[a]; c->bbox_max[a] = bmax[a];
  }
  c->have_bbox = true;
  c->configured = false;
  return RR_OK;
}

int rr_calib_upload(rr_ctx* c, int sensor, const float* cv_xyz, const float* cv_uv, const uint32_t res[3], const float dl[2]) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, sensor >= 0 && sensor < c->N, "rr_calib_upload: sensor index out of range");
  RR_REQUIRE(c, cv_xyz && cv_uv && res && dl, "rr_calib_upload: null pointer");
  RR_REQUIRE(c, res[0] >= 2 && res[1] >= 2 && res[2] >= 2, "rr_calib_upload: volume needs >= 2 voxels per axis");
  RR_SET_DEVICE(c);
  const size_t n = (size_t)res[0] * res[1] * res[2];
  RR_TRY(c->d_xyz[sensor].allocate(c, n, "cv_xyz"));
  RR_TRY(c->d_uv[sensor].allocate(c, n, "cv_uv"));
  DeviceArray<float> staging;
  RR_TRY(staging.allocate(c, n * 3, "cv_xyz staging"));
  cudaMemcpyAsync(staging.ptr, cv_xyz, n * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream);
  k_pad_xyz<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(staging.ptr, c->d_xyz[sensor].ptr, n);
  ++c->launches;
  cudaMemcpyAsync(c->d_uv[sensor].ptr, cv_uv, n * 2 * sizeof(float), cudaMemcpyHostToDevice, c->stream);
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "calib upload"));
  for (int a = 0; a < 3; ++a) c->cres[sensor][a] = res[a];
  c->dlim[sensor][0] = dl[0]; c->dlim[sensor][1] = dl[1];
  host_frustum(cv_xyz, res, c->planes[sensor], c->cam_pos[sensor]);
  for (int a = 0; a < 3; ++a) { c->xyz_min[sensor][a] = cv_xyz[a]; c->xyz_max[sensor][a] = cv_xyz[a]; }
  for (size_t i = 0; i < n; ++i)
    for (int a = 0; a < 3; ++a) {
      const float v = cv_xyz[i * 3 + a];
      if (v < c->xyz_min[sensor][a]) c->xyz_min[sensor][a] = v;
      if (v > c->xyz_max[sensor][a]) c->xyz_max[sensor][a] = v;
    }
  c->have_calib[sensor] = true;
  return RR_OK;
}

// All sensors share one inverse-volume resolution (CalibVolumes::getVolumeRes): a new one reallocates d_inv, and is refused
// with `refusal` while another sensor's inverse volume is loaded.
static int ensure_inv(rr_ctx* c, int sensor, const uint32_t res[3], const char* refusal) {
  if (c->d_inv.ptr && c->ires[0] == res[0] && c->ires[1] == res[1] && c->ires[2] == res[2]) return RR_OK;
  for (int i = 0; i < c->N; ++i) RR_REQUIRE(c, !c->have_inv[i] || i == sensor, refusal);
  RR_TRY(c->d_inv.allocate(c, (size_t)res[0] * res[1] * res[2] * c->N, "cv_xyz_inv"));
  for (int a = 0; a < 3; ++a) c->ires[a] = res[a];
  for (int i = 0; i < c->N; ++i) c->have_inv[i] = false;
  return RR_OK;
}

int rr_calib_upload_inv(rr_ctx* c, int sensor, const float* inv, const uint32_t res[3]) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, sensor >= 0 && sensor < c->N, "rr_calib_upload_inv: sensor index out of range");
  RR_REQUIRE(c, inv && res && res[0] && res[1] && res[2], "rr_calib_upload_inv: null pointer or empty volume");
  RR_SET_DEVICE(c);
  const size_t n = (size_t)res[0] * res[1] * res[2];
  RR_TRY(ensure_inv(c, sensor, res, "rr_calib_upload_inv: all sensors must share one inverse-volume resolution (CalibVolumes::getVolumeRes)"));
  RR_TRY(check(c, cudaMemcpyAsync(c->d_inv.ptr + n * sensor, inv, n * sizeof(float4), cudaMemcpyHostToDevice, c->stream), "inv upload"));
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "inv upload sync"));
  c->have_inv[sensor] = true;
  c->sti.dirty = true;
  return RR_OK;
}

int rr_get_camera_positions(const rr_ctx* c, float* out) {
  if (!c || !out) return RR_ERR_INVALID;
  for (int i = 0; i < c->N; ++i) for (int a = 0; a < 3; ++a) out[i * 3 + a] = c->cam_pos[i][a];
  return RR_OK;
}

int rr_get_frustum_planes(const rr_ctx* c, int sensor, float* out) {
  if (!c || !out || sensor < 0 || sensor >= c->N || !c->have_calib[sensor]) return RR_ERR_INVALID;
  std::memcpy(out, c->planes[sensor], sizeof(float) * 24);
  return RR_OK;
}

int rr_configure(rr_ctx* c, const rr_config* cfg) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, cfg, "rr_configure: null config");
  RR_REQUIRE(c, c->have_bbox, "rr_configure: call rr_set_bbox first");
  RR_REQUIRE(c, cfg->voxel_size > 0.0f && cfg->brick_size > 0.0f && cfg->limit > 0.0f, "rr_configure: sizes and limit must be positive");
  RR_REQUIRE(c, cfg->store_weight >= RR_VOXELS_F32 && cfg->store_weight <= RR_VOXELS_HALF2, "rr_configure: unknown voxel format (store_weight must be 0, 1 or 2)");
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "configure sync"));
  uint32_t res[3];
  host_volume_res(c->bbox_min, c->bbox_max, cfg->voxel_size, res);
  RR_REQUIRE(c, res[0] && res[1] && res[2], "rr_configure: empty volume");
  // The kernels index voxels with 32-bit arithmetic (march_column / march_staged offsets, sample_tsdf's z0 * X * Y): a
  // volume of 2^31 voxels or more (about 1290^3; 8 GB of R32F, which HBM would hold) is refused instead of wrapping.
  if ((unsigned long long)res[0] * res[1] * res[2] >= (1ull << 31))
    return fail(c, RR_ERR_UNSUPPORTED, "rr_configure: volumes of 2^31 voxels or more are not supported (32-bit voxel indices)");
  const float bs = host_adjust_brick_size(cfg->voxel_size, cfg->brick_size);
  RR_REQUIRE(c, bs > 0.0f, "rr_configure: brick size rounds to zero voxels");
  const bool new_volume = !c->configured || res[0] != c->res[0] || res[1] != c->res[1] || res[2] != c->res[2] ||
                          (cfg->store_weight == RR_VOXELS_F32_WEIGHT) != (c->d_weight.ptr != nullptr);
  const bool new_bricks = new_volume || bs != c->bricks.brick_size;
  // the staged integrator's tables depend on the volume, the brick grid, bricks mode and the voxel format; plain setters
  // (limit, min_voxels, skip_space) keep them, and the next integrate needs no synchronising rebuild
  const bool restage = new_bricks || cfg->use_bricks != c->cfg.use_bricks || cfg->store_weight != c->cfg.store_weight;
  if (new_volume) {
    const size_t nvox = (size_t)res[0] * res[1] * res[2];
    RR_TRY(c->d_tsdf.allocate(c, nvox, "tsdf volume"));
    RR_TRY(c->d_weight.allocate(c, cfg->store_weight == RR_VOXELS_F32_WEIGHT ? nvox : 0, "weight volume"));
    for (int a = 0; a < 3; ++a) c->res[a] = res[a];
    c->slab_z0 = 0; c->slab_z1 = res[2];
  }
  // the incremental clear knows nothing about a new allocation, a new brick grid or a volume last written in another mode
  if (new_bricks || !c->configured || cfg->store_weight != c->cfg.store_weight || cfg->use_bricks != c->cfg.use_bricks) c->clear.valid = false;
  if (new_volume || cfg->store_weight != c->cfg.store_weight) {   // a new volume allocation as far as extraction goes
    c->volume_integrated = false;
    c->mesh_valid = false;
    c->parts_valid = false;
    c->simp_valid = false;
    track_reset(c);                // labels of another grid or voxel format are not comparable
    ++c->volume_epoch;
  }
  if (new_volume) {   // the label and row arrays are sized by the volume
    c->d_parts_labels[0].release();
    c->d_parts_labels[1].release();
    c->d_parts_rows.release();
  }
  if (new_bricks) {
    c->mesh_rows_ok = false;
    uint32_t rb[3];
    const uint32_t nb = host_divide_box(c->bbox_min, c->bbox_max, bs, res, rb, &c->h_ranges);
    c->bricks.brick_size = bs; c->bricks.num = nb;
    for (int a = 0; a < 3; ++a) c->bricks.res[a] = rb[a];
    RR_TRY(c->d_ranges.allocate(c, (size_t)nb * 6, "brick ranges"));
    RR_TRY(c->d_counters.allocate(c, (size_t)nb + RR_CLASS_COUNTERS, "brick counters"));
    RR_TRY(c->d_occupied.allocate(c, nb, "occupied list"));
    RR_TRY(c->d_near_occ.allocate(c, nb, "near-occupied mask"));
    RR_TRY(c->d_occ_mask.allocate(c, nb, "occupied mask"));
    RR_TRY(c->d_written.allocate(c, 2 * (size_t)nb, "written bricks"));
    // per-axis candidate bricks of every voxel index (bricks may overlap by a voxel, or leave a gap)
    c->mask_words = (int)((res[0] + 31) / 32);
    c->fused_ok = rb[0] <= 32767 && rb[1] <= 32767 && rb[2] <= 32767;
    std::vector<int16_t> cand[3];
    for (int a = 0; a < 3 && c->fused_ok; ++a) {
      cand[a].assign((size_t)res[a] * 2, (int16_t)-1);
      const size_t stride = (a == 0) ? 1 : (a == 1 ? rb[0] : (size_t)rb[0] * rb[1]);
      for (uint32_t i = 0; i < rb[a] && c->fused_ok; ++i) {
        const int32_t* r = c->h_ranges.data() + (size_t)i * stride * 6 + 2 * a;
        for (int32_t v = r[0]; v < r[1]; ++v) {
          int16_t* slot = cand[a].data() + (size_t)v * 2;
          if (slot[0] < 0) slot[0] = (int16_t)i;
          else if (slot[1] < 0) slot[1] = (int16_t)i;
          else c->fused_ok = false;     // three bricks share a voxel on one axis: use the unfused path
        }
      }
    }
    RR_TRY(c->d_rowmask.allocate(c, (size_t)rb[2] * rb[1] * c->mask_words, "row masks"));
    RR_TRY(c->d_rowany.allocate(c, (size_t)rb[2] * rb[1], "row flags"));
    RR_TRY(c->d_cand_y.allocate(c, (size_t)res[1] * 2, "cand y"));
    RR_TRY(c->d_cand_z.allocate(c, (size_t)res[2] * 2, "cand z"));
    if (c->fused_ok) {
      cudaMemcpyAsync(c->d_cand_y.ptr, cand[1].data(), cand[1].size() * sizeof(int16_t), cudaMemcpyHostToDevice, c->stream);
      cudaMemcpyAsync(c->d_cand_z.ptr, cand[2].data(), cand[2].size() * sizeof(int16_t), cudaMemcpyHostToDevice, c->stream);
    }
    cudaMemsetAsync(c->d_rowmask.ptr, 0, (size_t)rb[2] * rb[1] * c->mask_words * sizeof(uint32_t), c->stream);
    cudaMemsetAsync(c->d_rowany.ptr, 0, (size_t)rb[2] * rb[1], c->stream);
    cudaMemcpyAsync(c->d_ranges.ptr, c->h_ranges.data(), (size_t)nb * 6 * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    cudaMemsetAsync(c->d_counters.ptr, 0, ((size_t)nb + RR_CLASS_COUNTERS) * sizeof(uint32_t), c->stream);
    cudaMemsetAsync(c->d_near_occ.ptr, 0, nb, c->stream);
    cudaMemsetAsync(c->d_occ_mask.ptr, 0, nb, c->stream);
    cudaMemsetAsync(c->d_written.ptr, 0, 2 * (size_t)nb, c->stream);
    cudaMemsetAsync(c->d_num_occ.ptr, 0, sizeof(uint32_t), c->stream);
    c->pinned->num_occ = 0;
    RR_TRY(check(c, cudaStreamSynchronize(c->stream), "brick table upload"));
  }
  c->cfg = *cfg;
  c->configured = true;
  if (restage) c->sti.dirty = true;
  return RR_OK;
}

int rr_get_volume_res(const rr_ctx* c, uint32_t res[3]) {
  if (!c || !res || !c->configured) return RR_ERR_INVALID;
  for (int a = 0; a < 3; ++a) res[a] = c->res[a];
  return RR_OK;
}

int rr_get_brick_info(const rr_ctx* c, uint32_t rb[3], float* bs, uint32_t* nb) {
  if (!c || !c->configured) return RR_ERR_INVALID;
  if (rb) for (int a = 0; a < 3; ++a) rb[a] = c->bricks.res[a];
  if (bs) *bs = c->bricks.brick_size;
  if (nb) *nb = c->bricks.num;
  return RR_OK;
}

int rr_get_brick_ranges(const rr_ctx* c, int32_t* out) {
  if (!c || !out || !c->configured) return RR_ERR_INVALID;
  std::memcpy(out, c->h_ranges.data(), c->h_ranges.size() * sizeof(int32_t));
  return RR_OK;
}

int rr_set_slab(rr_ctx* c, uint32_t z0, uint32_t z1) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, c->configured, "rr_set_slab: call rr_configure first");
  RR_REQUIRE(c, z0 <= z1 && z1 <= c->res[2], "rr_set_slab: slab outside the volume");
  c->slab_z0 = z0; c->slab_z1 = z1;
  c->clear.valid = false;
  return RR_OK;
}

static size_t color_bytes_of(const rr_ctx* c) {
  if (c->color_format == RR_COLOR_DXT1) return (size_t)c->N * c->CW * c->CH / 2;       // 8 bytes per 4x4 block
  if (c->color_format == RR_COLOR_DXT5) return (size_t)c->N * c->CW * c->CH;           // 16 bytes per 4x4 block
  return (size_t)c->N * c->CW * c->CH * 3;
}
static size_t depth_bytes_of(const rr_ctx* c) {
  return (size_t)c->N * c->W * c->H * (c->depth_format == RR_DEPTH_U8 ? 1 : sizeof(float));
}

static int check_frame_sizes(rr_ctx* c, const void* color, size_t cb, const void* depth, size_t db) {
  RR_REQUIRE(c, depth && db == depth_bytes_of(c), "rr_upload_frames: depth must be [N][H][W] in the format of rr_set_frame_format (default float32)");
  RR_REQUIRE(c, !color || cb == color_bytes_of(c), "rr_upload_frames: colour must be [N] layers in the format of rr_set_frame_format (default uint8 [CH][CW][3])");
  return RR_OK;
}

int rr_set_frame_format(rr_ctx* c, int color_format, int depth_format, const float* near_far) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, color_format == RR_COLOR_RGB8 || color_format == RR_COLOR_DXT1 || color_format == RR_COLOR_DXT5, "rr_set_frame_format: unknown colour format");
  RR_REQUIRE(c, depth_format == RR_DEPTH_F32 || depth_format == RR_DEPTH_U8, "rr_set_frame_format: unknown depth format");
  RR_REQUIRE(c, color_format == RR_COLOR_RGB8 || ((c->CW % 4) == 0 && (c->CH % 4) == 0), "rr_set_frame_format: DXT1 / DXT5 need colour width and height that are multiples of 4");
  RR_REQUIRE(c, depth_format != RR_DEPTH_U8 || near_far, "rr_set_frame_format: 8-bit depth needs the per-sensor (near, far) range");
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaStreamSynchronize(c->copy_stream), "format sync"));
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "format sync"));
  c->staged = false;
  c->color_format = color_format; c->depth_format = depth_format;
  for (int b = 0; b < 2; ++b) {
    // sized for the larger block format (DXT5, 16 bytes per 4x4 block), so a later format switch needs no reallocation
    if (color_format != RR_COLOR_RGB8 && !c->d_color_packed[b].ptr) RR_TRY(c->d_color_packed[b].allocate(c, (size_t)c->N * c->CW * c->CH, "packed colour"));
    if (depth_format == RR_DEPTH_U8 && !c->d_depth_packed[b].ptr) RR_TRY(c->d_depth_packed[b].allocate(c, (size_t)c->N * c->W * c->H, "packed depth"));
  }
  for (int i = 0; i < c->N; ++i) {
    c->depth_near[i] = near_far ? near_far[2 * i] : 0.0f;
    c->depth_far[i] = near_far ? near_far[2 * i + 1] : 0.0f;
  }
  return RR_OK;
}

int rr_stage_frames(rr_ctx* c, const void* color, size_t cb, const void* depth, size_t db) {
  if (!c) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  RR_TRY(check_frame_sizes(c, color, cb, depth, db));
  const int t = c->cur_slot ^ 1;
  // the slot may still be read by kernels launched while it was current
  if (c->free_recorded[t]) RR_TRY(check(c, cudaStreamWaitEvent(c->copy_stream, c->ev_free[t], 0), "stage wait"));
  void* dd = c->depth_format == RR_DEPTH_U8 ? (void*)c->d_depth_packed[t].ptr : (void*)c->d_depth_slot[t].ptr;
  void* dc = c->color_format != RR_COLOR_RGB8 ? (void*)c->d_color_packed[t].ptr : (void*)c->d_color_slot[t].ptr;
  RR_TRY(check(c, cudaMemcpyAsync(dd, depth, db, cudaMemcpyHostToDevice, c->copy_stream), "depth upload"));
  if (color) RR_TRY(check(c, cudaMemcpyAsync(dc, color, cb, cudaMemcpyHostToDevice, c->copy_stream), "colour upload"));
  c->staged_color = color != nullptr;
  RR_TRY(check(c, cudaEventRecord(c->ev_staged, c->copy_stream), "stage record"));
  c->staged = true;
  return RR_OK;
}

int rr_swap_frames(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->staged, "rr_swap_frames: no staged frame set (call rr_stage_frames first)");
  RR_SET_DEVICE(c);
  const int old = c->cur_slot, t = old ^ 1;
  RR_TRY(check(c, cudaEventRecord(c->ev_free[old], c->stream), "swap record"));
  c->free_recorded[old] = true;
  RR_TRY(check(c, cudaStreamWaitEvent(c->stream, c->ev_staged, 0), "swap wait"));
  c->cur_slot = t;
  c->d_depth_raw = c->d_depth_slot[t].ptr; c->d_color = c->d_color_slot[t].ptr;
  c->staged = false;
  // packed layers (DXT1 colour, 8-bit depth) are expanded here, once, behind the staged copy
  const int keep_color = c->color_format;
  if (!c->staged_color) c->color_format = RR_COLOR_RGB8;      // no colour was staged: nothing to decode
  const int rc = launch_unpack_frames(c, t);
  c->color_format = keep_color;
  return rc;
}

int rr_stage_sync(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  return check(c, cudaStreamSynchronize(c->copy_stream), "stage sync");
}

int rr_upload_frames(rr_ctx* c, const void* color, size_t cb, const void* depth, size_t db) {
  if (!c) return RR_ERR_INVALID;
  if (c->staged) RR_TRY(rr_swap_frames(c));     // a frame set staged earlier is superseded, but its slot must be released in order
  RR_TRY(rr_stage_frames(c, color, cb, depth, db));
  return rr_swap_frames(c);
}

int rr_upload_frames_device(rr_ctx* c, const void* color, size_t cb, const void* depth, size_t db) {
  if (!c) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  RR_TRY(check_frame_sizes(c, color, cb, depth, db));
  // already on this GPU (e.g. the output of an NCCL broadcast ordered before the context's stream): straight into the
  // current slot, on the compute stream
  const int t = c->cur_slot;
  void* dd = c->depth_format == RR_DEPTH_U8 ? (void*)c->d_depth_packed[t].ptr : (void*)c->d_depth_slot[t].ptr;
  void* dc = c->color_format != RR_COLOR_RGB8 ? (void*)c->d_color_packed[t].ptr : (void*)c->d_color_slot[t].ptr;
  RR_TRY(check(c, cudaMemcpyAsync(dd, depth, db, cudaMemcpyDeviceToDevice, c->stream), "depth upload"));
  if (color) RR_TRY(check(c, cudaMemcpyAsync(dc, color, cb, cudaMemcpyDeviceToDevice, c->stream), "colour upload"));
  const int keep_color = c->color_format;
  if (!color) c->color_format = RR_COLOR_RGB8;
  const int rc = launch_unpack_frames(c, t);
  c->color_format = keep_color;
  return rc;
}

static int require_ready(rr_ctx* c, bool need_inv) {
  RR_REQUIRE(c, c->configured, "call rr_configure first");
  for (int i = 0; i < c->N; ++i) {
    RR_REQUIRE(c, c->have_calib[i], "missing forward calibration volume (rr_calib_upload)");
    if (need_inv) RR_REQUIRE(c, c->have_inv[i], "missing inverse calibration volume (rr_calib_upload_inv / rr_calib_invert)");
  }
  return RR_OK;
}

int rr_bricks_clear(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->configured, "rr_bricks_clear: call rr_configure first");
  RR_SET_DEVICE(c);
  return launch_bricks_clear(c);
}

int rr_preprocess(rr_ctx* c, int filter_textures, int use_processed_depth, int refine_boundary) {
  if (!c) return RR_ERR_INVALID;
  RR_TRY(require_ready(c, false));
  RR_SET_DEVICE(c);
  RR_TRY(launch_preprocess(c, filter_textures, use_processed_depth, refine_boundary));
  c->preprocessed = true;
  return RR_OK;
}

int rr_bricks_update(rr_ctx* c, uint32_t* out_num, float* out_ratio) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->configured, "rr_bricks_update: call rr_configure first");
  RR_SET_DEVICE(c);
  RR_TRY(launch_bricks_update(c));
  if (out_num || out_ratio) {
    RR_TRY(check(c, cudaStreamSynchronize(c->stream), "bricks update sync"));
    if (out_num) *out_num = c->pinned->num_occ;
    if (out_ratio) *out_ratio = float(c->pinned->num_occ) / float(c->bricks.num);
  }
  return RR_OK;
}

int rr_integrate(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  RR_TRY(require_ready(c, true));
  RR_SET_DEVICE(c);
  return launch_integrate(c);
}

static int frame_direct(rr_ctx* c, int f, int p, int r) {
  RR_TRY(launch_bricks_clear(c));
  RR_TRY(launch_preprocess(c, f, p, r));
  RR_TRY(launch_bricks_update(c));
  return launch_integrate(c);
}

int rr_fuse_frame(rr_ctx* c, int filter_textures, int use_processed_depth, int refine_boundary) {
  if (!c) return RR_ERR_INVALID;
  RR_TRY(require_ready(c, true));
  RR_SET_DEVICE(c);
  const int f = filter_textures ? 1 : 0, p = use_processed_depth ? 1 : 0, r = refine_boundary ? 1 : 0;
  RR_TRY(staged_prepare(c));       // table rebuilds synchronise: never inside a capture
  c->preprocessed = true;          // every path below pre-processes (direct, captured or replayed)
  // capture needs a launch sequence without allocations or event timers: the z table exists (first frame ran direct)
  // and stage timing is off
  const bool ready = rr::tunables().graph != 0 && !c->graphs_broken && c->timing == 0 && c->d_ztab.ptr &&
                     c->ztab_Z == (int)c->res[2] && c->ztab_IZ == (int)c->ires[2];
  if (!ready) return frame_direct(c, f, p, r);
  // a graph captured with the incremental clear must not run while the volume needs the whole slab cleared, nor the other
  // way round: whether the integrate clears incrementally is part of the key
  const int inc = rr::clear_incremental(c) ? 1 : 0;
  const uint64_t key = ((uint64_t)rr::tunables().generation << 8) | (uint64_t)(inc << 4 | c->cur_slot << 3 | f << 2 | p << 1 | r);
  for (auto& g : c->frame_graphs)
    if (g.key == key) {
      c->launches += g.launches;
      c->volume_integrated = true;                 // the captured frame ends with the integrate launch_integrate recorded
      ++c->volume_epoch;
      c->clear = g.clear;
      std::memcpy(c->last_integrate, g.last, sizeof(g.last));
      c->mesh_rows_ok = mesh_rows_usable(c);
      return check(c, cudaGraphLaunch(g.exec, c->stream), "frame graph launch");
    }
  if (c->frame_graphs.size() >= 16) drop_frame_graphs(c);          // stale tunable generations
  const uint64_t l0 = c->launches;
  // a capture runs nothing: what launch_integrate records on the host while capturing must not survive a failed capture
  const rr::ClearState clear0 = c->clear;
  uint32_t last0[8];
  std::memcpy(last0, c->last_integrate, sizeof(last0));
  if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    c->graphs_broken = true;
    return frame_direct(c, f, p, r);
  }
  const int rc = frame_direct(c, f, p, r);
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
  cudaGraphExec_t exec = nullptr;
  if (rc == RR_OK && e == cudaSuccess && graph) e = cudaGraphInstantiate(&exec, graph, 0);
  if (graph) cudaGraphDestroy(graph);
  const uint64_t captured = c->launches - l0;
  c->launches = l0;
  if (rc != RR_OK || e != cudaSuccess || !exec) {
    cudaGetLastError();
    c->graphs_broken = true;
    c->clear = clear0;
    std::memcpy(c->last_integrate, last0, sizeof(last0));
    return frame_direct(c, f, p, r);
  }
  c->frame_graphs.push_back({key, exec, captured, c->clear, {}});
  std::memcpy(c->frame_graphs.back().last, c->last_integrate, sizeof(c->last_integrate));
  c->launches += captured;
  return check(c, cudaGraphLaunch(exec, c->stream), "frame graph launch");
}

int rr_bricks_count(rr_ctx* c, uint32_t* out_num, float* out_ratio) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->configured, "rr_bricks_count: call rr_configure first");
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "bricks count sync"));
  if (out_num) *out_num = c->pinned->num_occ;
  if (out_ratio) *out_ratio = float(c->pinned->num_occ) / float(c->bricks.num);
  return RR_OK;
}

int ensure_view(rr_ctx* c, int w, int h) {
  if (w == c->view_w && h == c->view_h) return RR_OK;
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "raymarch resize sync"));
  RR_TRY(c->d_rgba.allocate(c, (size_t)w * h, "view rgba"));
  RR_TRY(c->d_zbuf.allocate(c, (size_t)w * h, "view depth"));
  RR_TRY(c->d_nsamples.allocate(c, (size_t)w * h, "view samples"));
  RR_TRY(c->d_pos.allocate(c, (size_t)w * h, "view positions"));
  RR_TRY(c->d_step.allocate(c, (size_t)w * h, "view steps"));
  RR_TRY(c->d_point_keys.allocate(c, (size_t)w * h, "point keys"));
  c->view_w = w; c->view_h = h;
  return RR_OK;
}

int rr_raymarch(rr_ctx* c, const rr_view* view, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, view, "rr_raymarch: null view");
  RR_TRY(require_ready(c, true));
  RR_REQUIRE(c, view->viewport[2] > 0 && view->viewport[3] > 0, "rr_raymarch: empty viewport");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, view->viewport[2], view->viewport[3]));
  RR_TRY(launch_raymarch(c, view));
  return view_download(c, out_rgba, out_depth, "rr_raymarch");
}

static int draw_points_common(rr_ctx* c, const rr_view* view, int mode, float limit, float* out_rgba, float* out_depth, const char* who) {
  RR_REQUIRE(c, view, "draw points: null view");
  RR_REQUIRE(c, view->viewport[2] > 0 && view->viewport[3] > 0, "draw points: empty viewport");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, view->viewport[2], view->viewport[3]));
  RR_TRY(launch_draw_points(c, view, mode, limit));
  return view_download(c, out_rgba, out_depth, who);
}

int rr_draw_points(rr_ctx* c, const rr_view* view, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  for (int i = 0; i < c->N; ++i) RR_REQUIRE(c, c->have_calib[i], "rr_draw_points: upload every sensor's calibration volumes first");
  return draw_points_common(c, view, 0, 0.0f, out_rgba, out_depth, "rr_draw_points");
}

int rr_draw_calibs(rr_ctx* c, const rr_view* view, int active_kinect, float tsdf_limit, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  RR_TRY(require_ready(c, true));
  RR_REQUIRE(c, active_kinect >= 0 && active_kinect < c->N, "rr_draw_calibs: no such sensor");
  RR_REQUIRE(c, tsdf_limit > 0.0f, "rr_draw_calibs: the limit must be positive");
  return draw_points_common(c, view, 1, tsdf_limit, out_rgba, out_depth, "rr_draw_calibs");
}

int rr_draw_trigrid(rr_ctx* c, const rr_view* view, float min_length, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, view, "rr_draw_trigrid: null view");
  RR_REQUIRE(c, view->viewport[2] > 0 && view->viewport[3] > 0, "rr_draw_trigrid: empty viewport");
  RR_REQUIRE(c, min_length > 0.0f, "rr_draw_trigrid: min_length must be positive");
  for (int i = 0; i < c->N; ++i) RR_REQUIRE(c, c->have_calib[i], "rr_draw_trigrid: upload every sensor's calibration volumes first");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, view->viewport[2], view->viewport[3]));
  RR_TRY(launch_draw_trigrid(c, view, min_length));
  return view_download(c, out_rgba, out_depth, "rr_draw_trigrid");
}

int rr_fill_colors(rr_ctx* c, float* out_rgba) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->d_rgba.ptr && c->view_w > 0 && c->view_h > 0, "rr_fill_colors: no view yet (rr_raymarch / rr_composite / rr_upload_view first)");
  RR_SET_DEVICE(c);
  RR_TRY(launch_fill_colors(c));
  if (out_rgba) {
    RR_TRY(check(c, cudaMemcpyAsync(out_rgba, c->d_filled.ptr, (size_t)c->view_w * c->view_h * sizeof(float4), cudaMemcpyDeviceToHost, c->stream), "filled colour download"));
    RR_TRY(check(c, cudaStreamSynchronize(c->stream), "fill sync"));
  }
  return RR_OK;
}

int rr_upload_view(rr_ctx* c, int width, int height, const float* rgba, const float* depth) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, width > 0 && height > 0 && rgba && depth, "rr_upload_view: bad arguments");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, width, height));
  const size_t n = (size_t)width * height;
  RR_TRY(check(c, cudaMemcpyAsync(c->d_rgba.ptr, rgba, n * sizeof(float4), cudaMemcpyHostToDevice, c->stream), "view upload"));
  RR_TRY(check(c, cudaMemcpyAsync(c->d_zbuf.ptr, depth, n * sizeof(float), cudaMemcpyHostToDevice, c->stream), "view upload"));
  return check(c, cudaStreamSynchronize(c->stream), "view upload sync");
}

int rr_raymarch_partial(rr_ctx* c, const rr_view* view, void* d_records) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, view && d_records, "rr_raymarch_partial: null pointer");
  RR_TRY(require_ready(c, true));
  RR_REQUIRE(c, view->viewport[2] > 0 && view->viewport[3] > 0, "rr_raymarch_partial: empty viewport");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, view->viewport[2], view->viewport[3]));
  RR_TRY(launch_raymarch(c, view));
  return launch_pack_partial(c, (float4*)d_records);
}

int rr_partial_keys(rr_ctx* c, const void* d_records, int rank, void* d_keys) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, d_records && d_keys && rank >= 0 && rank < 256 && c->view_w > 0, "rr_partial_keys: bad arguments (march a view first; ranks 0..255)");
  RR_SET_DEVICE(c);
  return launch_partial_keys(c, (const float4*)d_records, rank, (long long*)d_keys);
}

int rr_partial_keep_winners(rr_ctx* c, void* d_records, const void* d_keys_min, int rank) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, d_records && d_keys_min && rank >= 0 && rank < 256 && c->view_w > 0, "rr_partial_keep_winners: bad arguments");
  RR_SET_DEVICE(c);
  return launch_partial_keep(c, (float4*)d_records, (const long long*)d_keys_min, rank);
}

int rr_composite(rr_ctx* c, const void* d_records, int n_parts, int width, int height, float* out_rgba, float* out_depth) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, d_records && n_parts >= 1 && width > 0 && height > 0, "rr_composite: bad arguments");
  RR_SET_DEVICE(c);
  RR_TRY(ensure_view(c, width, height));
  timer_begin(c, "composite");
  RR_TRY(launch_composite(c, (const float4*)d_records, n_parts));
  timer_end(c, "composite");
  return view_download(c, out_rgba, out_depth, "rr_composite");
}

int rr_calib_invert(rr_ctx* c, int sensor, const uint32_t out_res[3], float* host_out, int keep) {
  if (!c) return RR_ERR_INVALID;
  drop_frame_graphs(c);
  RR_REQUIRE(c, sensor >= 0 && sensor < c->N && c->have_calib[sensor], "rr_calib_invert: upload the sensor's cv_xyz first");
  RR_REQUIRE(c, c->have_bbox, "rr_calib_invert: call rr_set_bbox first");
  RR_REQUIRE(c, out_res && out_res[0] && out_res[1] && out_res[2], "rr_calib_invert: empty output resolution");
  RR_SET_DEVICE(c);
  const size_t n = (size_t)out_res[0] * out_res[1] * out_res[2];
  DeviceArray<float4> own;     // the output when it is not kept
  float4* d_out = nullptr;
  if (keep) {
    RR_TRY(ensure_inv(c, sensor, out_res, "rr_calib_invert: all sensors must share one inverse-volume resolution"));
    d_out = c->d_inv.ptr + n * sensor;
  } else {
    RR_TRY(own.allocate(c, n, "inverse volume"));
    d_out = own.ptr;
  }
  RR_TRY(launch_calib_invert(c, sensor, out_res, d_out));
  if (host_out) RR_TRY(check(c, cudaMemcpyAsync(host_out, d_out, n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream), "inverse download"));
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "invert sync"));
  if (keep) { c->have_inv[sensor] = true; c->sti.dirty = true; }
  return RR_OK;
}

static int download(rr_ctx* c, void* dst, const void* src, size_t bytes, const char* what) {
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream), what));
  return check(c, cudaStreamSynchronize(c->stream), what);
}

// binary16 -> binary32, exact (host side of the half2 voxel downloads)
static float half_bits_to_float(uint16_t h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16, exp = (h >> 10) & 31u, man = h & 1023u;
  uint32_t u;
  if (exp == 0) {
    if (man == 0) {
      u = sign;
    } else {                                   // subnormal half: normalise
      int e = -1;
      uint32_t m = man;
      do { ++e; m <<= 1; } while (!(m & 1024u));
      u = sign | ((uint32_t)(127 - 15 - e) << 23) | ((m & 1023u) << 13);
    }
  } else if (exp == 31) {
    u = sign | 0x7f800000u | (man << 13);
  } else {
    u = sign | ((exp + 112u) << 23) | (man << 13);
  }
  float f;
  std::memcpy(&f, &u, sizeof(f));
  return f;
}

// half2 voxels are 4 bytes like R32F ones: download raw, then widen the chosen half in place
static int download_half2(rr_ctx* c, float* out, int which) {
  const size_t n = (size_t)c->res[0] * c->res[1] * c->res[2];
  RR_TRY(download(c, out, c->d_tsdf.ptr, n * sizeof(float), "voxel download"));
  for (size_t i = 0; i < n; ++i) {
    uint32_t u;
    std::memcpy(&u, out + i, sizeof(u));
    out[i] = half_bits_to_float((uint16_t)(which ? (u >> 16) : (u & 0xffffu)));
  }
  return RR_OK;
}

int rr_download_tsdf(rr_ctx* c, float* out) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out && c->configured, "rr_download_tsdf: not configured or null pointer");
  if (c->cfg.store_weight == RR_VOXELS_HALF2) return download_half2(c, out, 0);
  return download(c, out, c->d_tsdf.ptr, (size_t)c->res[0] * c->res[1] * c->res[2] * sizeof(float), "tsdf download");
}

int rr_download_weight(rr_ctx* c, float* out) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out && c->configured, "rr_download_weight: not configured or null pointer");
  if (c->cfg.store_weight == RR_VOXELS_HALF2) return download_half2(c, out, 1);
  RR_REQUIRE(c, c->d_weight.ptr, "rr_download_weight: store_weight is off");
  return download(c, out, c->d_weight.ptr, (size_t)c->res[0] * c->res[1] * c->res[2] * sizeof(float), "weight download");
}

int rr_download_stage(rr_ctx* c, int stage, float* out) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out, "rr_download_stage: null pointer");
  const size_t px = (size_t)c->N * c->W * c->H;
  switch (stage) {
    case RR_STAGE_MORPH: return download(c, out, c->d_morph.ptr, px * sizeof(float), "stage download");
    case RR_STAGE_DEPTH: return download(c, out, c->d_depth.ptr, px * sizeof(float2), "stage download");
    case RR_STAGE_DEPTH_B: return download(c, out, c->d_depth_b.ptr, px * sizeof(float2), "stage download");
    case RR_STAGE_SILHOUETTE: return download(c, out, c->d_sil.ptr, px * sizeof(float), "stage download");
    case RR_STAGE_QUALITY: return download(c, out, c->d_quality.ptr, px * sizeof(float), "stage download");
    case RR_STAGE_LAB:
    case RR_STAGE_NORMAL: {
      RR_SET_DEVICE(c);
      DeviceArray<float> tmp;
      RR_TRY(tmp.allocate(c, px * 3, "stage staging"));
      k_unpad3<<<(unsigned)((px + 255) / 256), 256, 0, c->stream>>>(stage == RR_STAGE_LAB ? c->d_lab.ptr : c->d_normal.ptr, tmp.ptr, px);
      ++c->launches;
      return download(c, out, tmp.ptr, px * 3 * sizeof(float), "stage download");
    }
    default: return fail(c, RR_ERR_INVALID, "rr_download_stage: unknown stage");
  }
}

int rr_download_bricks(rr_ctx* c, uint32_t* counters, uint32_t* occupied, uint32_t* num_occupied) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->configured, "rr_download_bricks: call rr_configure first");
  RR_SET_DEVICE(c);
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "bricks download sync"));
  uint32_t n = 0;
  RR_TRY(download(c, &n, c->d_num_occ.ptr, sizeof(uint32_t), "count download"));
  if (counters) RR_TRY(download(c, counters, c->d_counters.ptr, c->bricks.num * sizeof(uint32_t), "counters download"));
  if (occupied && n) RR_TRY(download(c, occupied, c->d_occupied.ptr, n * sizeof(uint32_t), "occupied download"));
  if (num_occupied) *num_occupied = n;
  return RR_OK;
}

int rr_download_num_samples(rr_ctx* c, float* out) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out && c->d_nsamples.ptr, "rr_download_num_samples: no raymarch yet");
  return download(c, out, c->d_nsamples.ptr, (size_t)c->view_w * c->view_h * sizeof(float), "samples download");
}

int rr_download_hit_positions(rr_ctx* c, float* out) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out && c->d_pos.ptr, "rr_download_hit_positions: no raymarch yet");
  return download(c, out, c->d_pos.ptr, (size_t)c->view_w * c->view_h * sizeof(float4), "positions download");
}

int rr_extract_mesh(rr_ctx* c, uint32_t* out_num_vertices, uint32_t* out_num_triangles) {
  if (!c) return RR_ERR_INVALID;
  RR_TRY(require_ready(c, true));
  RR_REQUIRE(c, c->volume_integrated, "rr_extract_mesh: nothing has been integrated into the current volume");
  RR_REQUIRE(c, c->slab_z0 == 0 && c->slab_z1 == c->res[2],
             "rr_extract_mesh: this context holds only its z-slab (rr_set_slab); extract through rr_group_extract_mesh");
  RR_SET_DEVICE(c);
  return launch_extract_mesh(c, out_num_vertices, out_num_triangles);
}

int rr_label_parts(rr_ctx* c, uint32_t* out_num_parts) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out_num_parts, "rr_label_parts: null count pointer");
  RR_REQUIRE(c, c->configured && c->volume_integrated, "rr_label_parts: nothing has been integrated into the current volume");
  RR_REQUIRE(c, c->slab_z0 == 0 && c->slab_z1 == c->res[2],
             "rr_label_parts: this context holds only its z-slab (rr_set_slab); label through rr_group_label_parts");
  RR_SET_DEVICE(c);
  return launch_label_parts(c, label_dest(c), out_num_parts);
}

int rr_track_parts(rr_ctx* c, uint32_t min_voxels, uint32_t* out_num_parts, uint32_t* out_num_ended) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out_num_parts && out_num_ended, "rr_track_parts: null count pointer");
  RR_REQUIRE(c, min_voxels >= 1, "rr_track_parts: min_voxels must be at least 1");
  RR_REQUIRE(c, c->configured && c->volume_integrated, "rr_track_parts: nothing has been integrated into the current volume");
  RR_REQUIRE(c, c->slab_z0 == 0 && c->slab_z1 == c->res[2],
             "rr_track_parts: this context holds only its z-slab (rr_set_slab); track through rr_group_track_parts");
  RR_SET_DEVICE(c);
  return launch_track_parts(c, min_voxels, out_num_parts, out_num_ended);
}

int rr_download_part_tracks(rr_ctx* c, uint32_t* track_ids, uint32_t* prev_parts, uint32_t* overlaps, uint32_t* ended) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->track_valid, "rr_download_part_tracks: nothing tracked in the current volume (rr_track_parts first)");
  RR_SET_DEVICE(c);
  return track_download(c, track_ids, prev_parts, overlaps, ended);
}

int rr_reset_part_tracks(rr_ctx* c) {
  if (!c) return RR_ERR_INVALID;
  track_reset(c);
  return RR_OK;
}

int rr_download_parts(rr_ctx* c, uint32_t* voxels, int32_t* boxes, float* centroids, uint32_t* labels) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->parts_valid, "rr_download_parts: nothing labelled in the current volume (rr_label_parts first)");
  RR_SET_DEVICE(c);
  return parts_download(c, voxels, boxes, centroids, labels);
}

int rr_download_mesh_parts(rr_ctx* c, uint32_t* vertex_parts, uint32_t* triangle_parts) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->mesh_valid && c->parts_valid && c->mesh_epoch == c->parts_epoch,
             "rr_download_mesh_parts: needs a mesh and a labelling of the same volume state (rr_extract_mesh and rr_label_parts "
             "with no integrate in between)");
  RR_SET_DEVICE(c);
  return mesh_parts_download(c, vertex_parts, triangle_parts);
}

int rr_simplify_mesh(rr_ctx* c, uint32_t cluster_voxels, uint32_t* out_num_vertices, uint32_t* out_num_triangles) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out_num_vertices && out_num_triangles, "rr_simplify_mesh: null count pointer");
  RR_REQUIRE(c, cluster_voxels >= 1, "rr_simplify_mesh: cluster_voxels must be at least 1");
  RR_REQUIRE(c, c->mesh_valid && c->mesh_epoch == c->volume_epoch,
             "rr_simplify_mesh: no mesh of the current volume state (rr_extract_mesh after the last integrate first)");
  RR_SET_DEVICE(c);
  return launch_simplify_mesh(c, cluster_voxels, out_num_vertices, out_num_triangles);
}

int rr_download_simplified_mesh(rr_ctx* c, float* positions, float* normals, float* rgba, uint32_t* triangles, uint32_t* sources) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->simp_valid, "rr_download_simplified_mesh: nothing simplified in the current volume (rr_simplify_mesh first)");
  RR_SET_DEVICE(c);
  return simplified_download(c, positions, normals, rgba, triangles, sources);
}

}  // extern "C"

// The checks rr_sample_points / rr_cast_rays share with their group forms (whole_volume = false: a group member, which
// holds only its slab). RR_OK: go ahead with count > 0 entries.
int rr::query_check(rr_ctx* c, int space, uint32_t count, bool have_inputs, bool whole_volume, const char* who) {
  const std::string w(who);
  RR_REQUIRE(c, space == RR_QUERY_WORLD || space == RR_QUERY_VOLUME, w + ": space must be RR_QUERY_WORLD or RR_QUERY_VOLUME");
  RR_REQUIRE(c, have_inputs, w + ": null inputs");
  if (count >= (1u << 31)) return fail(c, RR_ERR_UNSUPPORTED, w + ": 2^31 or more entries are not supported");
  RR_TRY(require_ready(c, true));
  RR_REQUIRE(c, c->volume_integrated, w + ": nothing has been integrated into the current volume");
  if (whole_volume)
    RR_REQUIRE(c, c->slab_z0 == 0 && c->slab_z1 == c->res[2], w + ": this context holds only its z-slab (rr_set_slab); use the group form");
  return RR_OK;
}

extern "C" {

int rr_sample_points(rr_ctx* c, int space, const float* points, uint32_t count, float* values, float* normals, float* rgba) {
  if (!c) return RR_ERR_INVALID;
  if (count == 0 && (space == RR_QUERY_WORLD || space == RR_QUERY_VOLUME)) return RR_OK;
  RR_TRY(query_check(c, space, count, points != nullptr, true, "rr_sample_points"));
  RR_SET_DEVICE(c);
  RR_TRY(query_upload(c, points, nullptr, count));
  RR_TRY(launch_sample_points(c, space, count));
  return query_download(c, count, false, values, normals, rgba, nullptr);
}

int rr_cast_rays(rr_ctx* c, int space, const float* origins, const float* directions, uint32_t count,
                 float* positions, float* normals, float* rgba, uint32_t* steps) {
  if (!c) return RR_ERR_INVALID;
  if (count == 0 && (space == RR_QUERY_WORLD || space == RR_QUERY_VOLUME)) return RR_OK;
  RR_TRY(query_check(c, space, count, origins && directions, true, "rr_cast_rays"));
  RR_SET_DEVICE(c);
  RR_TRY(query_upload(c, origins, directions, count));
  RR_TRY(launch_cast_rays(c, space, count));
  return query_download(c, count, true, positions, normals, rgba, steps);
}

int rr_extract_points(rr_ctx* c, uint32_t sensor_mask, uint32_t* out_num_points) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, out_num_points, "rr_extract_points: null count pointer");
  RR_REQUIRE(c, (sensor_mask >> c->N) == 0, "rr_extract_points: sensor mask names a sensor at or above the sensor count");
  *out_num_points = 0;
  if (sensor_mask == 0) {
    c->cloud_n = 0;
    c->cloud_valid = true;
    return RR_OK;
  }
  for (int i = 0; i < c->N; ++i)
    if ((sensor_mask >> i) & 1u) RR_REQUIRE(c, c->have_calib[i], "rr_extract_points: missing forward calibration volume (rr_calib_upload)");
  RR_REQUIRE(c, c->preprocessed, "rr_extract_points: no stage images yet (rr_preprocess / rr_fuse_frame first)");
  RR_SET_DEVICE(c);
  return launch_extract_points(c, sensor_mask, out_num_points);
}

int rr_download_points(rr_ctx* c, float* positions, float* normals, float* colors, float* quality, uint32_t* pixels) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->cloud_valid, "rr_download_points: nothing extracted yet (rr_extract_points first)");
  RR_SET_DEVICE(c);
  return cloud_download(c, positions, normals, colors, quality, pixels);
}

int rr_download_mesh(rr_ctx* c, float* positions, float* normals, float* rgba, uint32_t* triangles) {
  if (!c) return RR_ERR_INVALID;
  RR_REQUIRE(c, c->mesh_valid, "rr_download_mesh: no mesh extracted from the current volume (rr_extract_mesh first)");
  RR_SET_DEVICE(c);
  const size_t nv = c->mesh_nv, nt = c->mesh_nt;
  if (positions && nv) RR_TRY(check(c, cudaMemcpyAsync(positions, c->d_mesh_pos.ptr, nv * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream), "mesh download"));
  if (normals && nv) RR_TRY(check(c, cudaMemcpyAsync(normals, c->d_mesh_nrm.ptr, nv * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream), "mesh download"));
  if (rgba && nv) RR_TRY(check(c, cudaMemcpyAsync(rgba, c->d_mesh_rgba.ptr, nv * sizeof(float4), cudaMemcpyDeviceToHost, c->stream), "mesh download"));
  if (triangles && nt) RR_TRY(check(c, cudaMemcpyAsync(triangles, c->d_mesh_tri.ptr, nt * 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "mesh download"));
  return check(c, cudaStreamSynchronize(c->stream), "mesh download sync");
}

int rr_set_timing(rr_ctx* c, int level) {
  if (!c) return RR_ERR_INVALID;
  c->timing = level < 0 ? 0 : (level > 2 ? 2 : level);
  return RR_OK;
}

int rr_get_stage_ms(rr_ctx* c, const char* name, float* ms) {
  if (!c || !name || !ms) return RR_ERR_INVALID;
  auto it = c->timers.find(name);
  RR_REQUIRE(c, it != c->timers.end() && (it->second.used > 0 || it->second.folded_n > 0), "rr_get_stage_ms: stage has not run with timing enabled");
  if (it->second.used == 0) { *ms = it->second.last_ms; return RR_OK; }
  RR_SET_DEVICE(c);
  const size_t i = it->second.used - 1;
  RR_TRY(check(c, cudaEventSynchronize(it->second.end[i]), "stage timer sync"));
  return check(c, cudaEventElapsedTime(ms, it->second.beg[i], it->second.end[i]), "stage timer");
}

int rr_get_stage_stats(rr_ctx* c, const char* name, float* total_ms, uint32_t* count) {
  if (!c || !name || !total_ms || !count) return RR_ERR_INVALID;
  *total_ms = 0.0f; *count = 0;
  auto it = c->timers.find(name);
  if (it == c->timers.end()) return RR_OK;
  RR_SET_DEVICE(c);
  StageTimer& t = it->second;
  for (size_t i = 0; i < t.used; ++i) {
    float ms = 0.0f;
    RR_TRY(check(c, cudaEventSynchronize(t.end[i]), "stage timer sync"));
    RR_TRY(check(c, cudaEventElapsedTime(&ms, t.beg[i], t.end[i]), "stage timer"));
    *total_ms += ms;
  }
  *total_ms += (float)t.folded_ms;
  *count = (uint32_t)t.used + t.folded_n;
  t.used = 0; t.folded_ms = 0.0; t.folded_n = 0;
  return RR_OK;
}

uint64_t rr_launch_count(const rr_ctx* c) { return c ? c->launches : 0; }

int rr_integrator_info(rr_ctx* c, uint32_t* out) {
  if (!c || !out) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  RR_TRY(staged_prepare(c));
  const auto& s = c->sti;
  std::memset(out, 0, 16 * sizeof(uint32_t));
  out[0] = staged_selected(c) ? 1u : 0u;
  out[1] = (uint32_t)s.T; out[2] = (uint32_t)s.BX; out[3] = (uint32_t)s.BY; out[4] = (uint32_t)s.BZ;
  out[5] = (uint32_t)s.cy; out[6] = (uint32_t)s.cz; out[7] = (uint32_t)s.n_yc; out[8] = (uint32_t)s.n_zc;
  out[9] = s.n_oversize; out[10] = s.smem_bytes; out[11] = (uint32_t)s.cwarps; out[12] = (uint32_t)s.fwarps; out[14] = s.n_slots; out[15] = s.slot_bytes;
  if (s.d_err.ptr) {
    uint32_t e[4] = {0, 0, 0, 0};
    RR_TRY(check(c, cudaStreamSynchronize(c->stream), "integrator info sync"));
    RR_TRY(check(c, cudaMemcpy(e, s.d_err.ptr, sizeof(e), cudaMemcpyDeviceToHost), "integrator flags"));
    out[13] = (e[0] ? 1u : 0u) | (e[1] ? 2u : 0u);
    if (out[13]) c->clear.valid = false;       // an item may have been left out: clear the whole slab next time
  }
  return RR_OK;
}

int rr_integrator_last(const rr_ctx* c, uint32_t* out) {
  if (!c || !out) return RR_ERR_INVALID;
  std::memcpy(out, c->last_integrate, sizeof(c->last_integrate));
  return RR_OK;
}

int rr_integrator_cleared(rr_ctx* c, uint32_t* out) {
  if (!c || !out) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  out[0] = 0;
  if (c->last_integrate[0] != 1 || c->last_integrate[5] != 2 || !c->d_work.ptr) return RR_OK;
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "integrator cleared sync"));
  return check(c, cudaMemcpy(out, c->d_work.ptr + 6, sizeof(uint32_t), cudaMemcpyDeviceToHost), "cleared bricks");
}

int rr_integrator_profile(rr_ctx* c, uint64_t* out) {
  if (!c || !out) return RR_ERR_INVALID;
  RR_SET_DEVICE(c);
  std::memset(out, 0, 16 * sizeof(uint64_t));
  if (!c->sti.d_err.ptr) return RR_OK;
  RR_TRY(check(c, cudaStreamSynchronize(c->stream), "integrator profile sync"));
  RR_TRY(check(c, cudaMemcpy(out, c->sti.d_err.ptr + 4, 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost), "integrator profile"));
  RR_TRY(check(c, cudaMemset(c->sti.d_err.ptr + 4, 0, 16 * sizeof(uint64_t)), "integrator profile reset"));
  return RR_OK;
}

int rr_set_tunable(const char* name, int value) {
  if (!name) return RR_ERR_INVALID;
  Tunables& t = tunables();
  const std::string n(name);
  if (n == "fused") t.fused = value;
  else if (n == "zchunk") t.zchunk = value;
  else if (n == "fill_rows") t.fill_rows = value;
  else if (n == "fill_warps") t.fill_warps = value;
  else if (n == "ctas") t.ctas = value;
  else if (n == "threads") t.threads = value;
  else if (n == "chunk") t.chunk = value;
  else if (n == "brick_grid") t.brick_grid = value;
  else if (n == "ldg256") t.ldg256 = value;
  else if (n == "graph") t.graph = value;
  else if (n == "staged") t.staged = value;
  else if (n == "stage_zchunk") t.stage_zchunk = value;
  else if (n == "stage_ychunk") t.stage_ychunk = value;
  else if (n == "stage_tile") t.stage_tile = value;
  else if (n == "stage_fill_rows") t.stage_fill_rows = value;
  else if (n == "stage_debug") t.stage_debug = value;
  else if (n == "stage_fill_depth") t.stage_fill_depth = value;
  else if (n == "stage_fill_lsu") t.stage_fill_lsu = value;
  else if (n == "stage_tail_cap") t.stage_tail_cap = value;
  else if (n == "stage_ctas") t.stage_ctas = value;
  else if (n == "stage_cwarps") t.stage_cwarps = value;
  else if (n == "stage_bulk_fill") t.stage_bulk_fill = value;
  else if (n == "trigrid_pool") t.trigrid_pool = value;
  else if (n == "fuse_nq") t.fuse_nq = value;
  else return RR_ERR_INVALID;
  ++t.generation;              // captured frame graphs bake the launch shapes in: stale keys never match again
  return RR_OK;
}

}  // extern "C"
