// Internal state behind the opaque rr_ctx of include/rgbd_recon_b200.h. One context = one GPU, one stream.
//
// Device memory layout (all allocations live for the context's lifetime; sized for 180 GB HBM3e, nothing is paged):
//   frames     depth float[N][H][W], colour uint8[N][CH][CW][3]                       (written by rr_upload_frames)
//   calib      per sensor cv_xyz as float4[Z][Y][X] (xyz padded to 16 B so a corner is one LDG.128),
//              cv_uv float2[Z][Y][X]; cv_xyz_inv float4[N][IZ][IY][IX] in one allocation
//   stages     morph float, depth float2, lab float4, depth_b float2, silhouette float, normal float4, quality float,
//              each [N][H][W]
//   gather     float4[N][H+1][W+1][2]: per bilinear footprint (i0,j0) the four depth_b.x taps and the four quality
//              taps (silhouette in the sign bit) = one 32-byte sector per voxel-sensor lookup in the integrator
//   bricks     uint32 counters[nb], occupied[nb], count; int32 ranges[nb][6]; uint8 near_occupied[nb], occ_mask[nb];
//              uint32 rowmask[nbz][nby][ceil(X/32)], uint8 rowany[nbz][nby], int16 cand_y[Y][2], cand_z[Z][2]
//   pairs      float2[N][H+2][pitch]: (depth_b.x, quality with the silhouette in the sign bit) per pixel, one replicated
//              border pixel on every side (CLAMP_TO_EDGE) - the image the staged integrator tiles into shared memory by TMA
//   footprints uint32[bricks * y-chunks * z-chunks][N]: origin of the pair-image tile each work item of the staged
//              integrator needs per sensor (fixed by calibration + brick grid, built once by k_footprints)
//   volume     tsdf float[Z][Y][X] (+ weight float[Z][Y][X] when rr_config.store_weight)
#pragma once

#include <cuda.h>            // CUtensorMap (types only; the encoder is fetched with cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rgbd_recon_b200.h"

#define RR_MAX_SENSORS 8
#define RR_MAX_GROUP 16           // members of an rr_group

namespace rr {

struct SensorTables {            // passed to kernels by value (__grid_constant__)
  const float4* xyz[RR_MAX_SENSORS];
  const float2* uv[RR_MAX_SENSORS];
  int cx[RR_MAX_SENSORS], cy[RR_MAX_SENSORS], cz[RR_MAX_SENSORS];
  float dmin[RR_MAX_SENSORS], dmax[RR_MAX_SENSORS];
  float cam[RR_MAX_SENSORS][3];
};

struct BrickGrid {
  float brick_size;
  uint32_t res[3];
  uint32_t num;
};

#define RR_CLASS_COUNTERS 16      // >= RR_MAX_SENSORS + 1

struct StageTimer {            // one CUDA-event pair per recorded interval; summed and recycled by rr_get_stage_stats
  std::vector<cudaEvent_t> beg, end;
  size_t used = 0;             // intervals recorded since the last reset / fold
  bool open = false;
  // O(1) state for callers that only ever ask for the mean at exit (TimerDatabase::mean): once kMaxPending intervals are
  // pending they are folded into a running sum, so the event vectors stop growing
  static constexpr size_t kMaxPending = 256;
  double folded_ms = 0.0;
  uint32_t folded_n = 0;
  float last_ms = 0.0f;        // the newest folded interval (rr_get_stage_ms right after a fold)
};

// A device array of the context that grows on demand to the size of a result (reserve, defined below rr_ctx); freed by the
// context's destructor, on the context's device.
template <typename T>
struct DeviceArray {
  T* ptr = nullptr;
  size_t cap = 0;              // in elements
  DeviceArray() = default;
  DeviceArray(const DeviceArray&) = delete;
  DeviceArray& operator=(const DeviceArray&) = delete;
  ~DeviceArray() { cudaFree(ptr); }
  int reserve(rr_ctx* c, size_t need, const char* what);
  void release() { cudaFree(ptr); ptr = nullptr; cap = 0; }
};

// Host scalars that device-to-host copies land in, one slot per reader: num_occ is filled by an asynchronous copy in
// rr_bricks_update and read by a later call, so no other copy may reuse its slot.
struct PinnedScalars {
  uint32_t num_occ;
  uint32_t cloud_count;
  uint32_t parts_count;
  unsigned long long mesh_totals[2];   // vertices, triangles
};

}  // namespace rr

struct rr_ctx {
  int device = 0;
  int N = 0, W = 0, H = 0, CW = 0, CH = 0;
  cudaStream_t stream = nullptr;
  std::string error;           // text of the last failing call; written under error_mutex (a reader thread may stage frames)
  std::mutex error_mutex;
  uint64_t launches = 0;
  int num_sms = 148;           // multiprocessors of the device (persistent kernels launch one CTA per SM)
  int timing = 0;              // 0 off, 1 top-level stages, 2 every pass
  std::map<std::string, rr::StageTimer> timers;

  // calibration
  float bbox_min[3] = {0, 0, 0}, bbox_max[3] = {0, 0, 0};
  bool have_bbox = false;
  float4* d_xyz[RR_MAX_SENSORS] = {};
  float2* d_uv[RR_MAX_SENSORS] = {};
  uint32_t cres[RR_MAX_SENSORS][3] = {};
  float dlim[RR_MAX_SENSORS][2] = {};
  float cam_pos[RR_MAX_SENSORS][3] = {};
  float planes[RR_MAX_SENSORS][6][4] = {};
  float xyz_min[RR_MAX_SENSORS][3] = {}, xyz_max[RR_MAX_SENSORS][3] = {};   // bounding box of the cv_xyz samples
  bool have_calib[RR_MAX_SENSORS] = {};
  float4* d_inv = nullptr;
  uint32_t ires[3] = {0, 0, 0};
  bool have_inv[RR_MAX_SENSORS] = {};

  // frames + stages. Two device frame slots (the reference's double PBO, double_pixel_buffer.cpp): d_depth_raw / d_color
  // alias the CURRENT slot (read by the kernels); rr_stage_frames copies into the other one on copy_stream.
  float* d_depth_raw = nullptr;
  uint8_t* d_color = nullptr;
  float* d_depth_slot[2] = {nullptr, nullptr};
  uint8_t* d_color_slot[2] = {nullptr, nullptr};
  int cur_slot = 0;
  bool staged = false;                       // the other slot holds a frame set that has not been swapped in yet
  bool staged_color = false;                 // ... and it came with colour
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_staged = nullptr;           // recorded on copy_stream after the staged copies
  cudaEvent_t ev_free[2] = {nullptr, nullptr};   // recorded on stream when a slot stops being current
  bool free_recorded[2] = {false, false};
  // compressed ingest (rr_set_frame_format): packed layers per slot, expanded by launch_unpack_frames at the swap
  int color_format = 0, depth_format = 0;
  uint8_t* d_color_packed[2] = {nullptr, nullptr};
  uint8_t* d_depth_packed[2] = {nullptr, nullptr};
  float depth_near[RR_MAX_SENSORS] = {}, depth_far[RR_MAX_SENSORS] = {};
  float* d_morph = nullptr;
  float2* d_depth = nullptr;
  float4* d_lab = nullptr;
  float2* d_depth_b = nullptr;
  float* d_sil = nullptr;
  float4* d_normal = nullptr;
  float* d_quality = nullptr;
  float4* d_gather = nullptr;
  bool gather_packed = false;      // d_gather holds the texels of the last rr_preprocess (k_pack_gather ran for it)
  float2* d_pairs = nullptr;       // [N][H+2][pair_pitch]
  int pair_pitch = 0;              // W+2 rounded up to even (TMA strides are multiples of 16 bytes)
  uint32_t* d_flags = nullptr;     // [0] pack-encoding violation counter

  // settings + bricks + volume
  rr_config cfg{};
  bool configured = false;
  uint32_t res[3] = {0, 0, 0};
  uint32_t slab_z0 = 0, slab_z1 = 0;
  rr::BrickGrid bricks{};
  std::vector<int32_t> h_ranges;
  int32_t* d_ranges = nullptr;
  uint32_t* d_counters = nullptr;  // [bricks.num] voxels seen per brick, then RR_CLASS_COUNTERS item-class counters of the staged integrator
  uint32_t* d_occupied = nullptr;
  uint32_t* d_num_occ = nullptr;
  uint8_t* d_near_occ = nullptr;
  uint8_t* d_occ_mask = nullptr;
  // fused clear+integrate support: per brick row (bz, by) the x bitmask of voxels inside occupied bricks, a byte that
  // says whether the row has any, and per voxel y / z index the (at most two) brick indices whose range contains it
  uint32_t* d_rowmask = nullptr;   // [nbz][nby][mask_words]
  uint8_t* d_rowany = nullptr;     // [nbz][nby]
  int16_t* d_cand_y = nullptr;     // [Y][2], -1 = none
  int16_t* d_cand_z = nullptr;     // [Z][2]
  uint32_t* d_work = nullptr;      // [4] work-item counters of the persistent fused kernel
  bool work_fresh = false;         // k_bricks_update has reset them and no integrate launch has drawn from them since
  int mask_words = 0;
  float4* d_ztab = nullptr;        // [Z] (k0, k1, g, 1-g) of the z filter tap against the inverse volume (k_build_ztab)
  int ztab_Z = 0, ztab_IZ = 0;
  bool fused_ok = false;           // brick table is separable with <= 2 bricks per voxel and axis
  // rr_fuse_frame: captured launch sequences, keyed by (frame slot, pre-process flags, tunable generation)
  struct FrameGraph { uint64_t key; cudaGraphExec_t exec; uint64_t launches; };
  std::vector<FrameGraph> frame_graphs;
  // view images of other processes' contexts opened through CUDA IPC (rr_composite_peers); key = the 256-byte handle blob
  struct IpcView { std::string key; uint32_t* step; float4* rgba; float* zbuf; float* nsamp; };
  std::vector<IpcView> ipc_views;
  bool graphs_broken = false;      // a capture failed once: stay on direct launches
  // the last launch_integrate (rr_integrator_last): path (0 none, 1 staged, 2 fused, 3 k_fill + k_integrate_bricks, 4 dense),
  // sensors, voxel mode, CTA threads or consumer warps, repairs (bit 0 stale item lists declined, bit 1 gather packed late)
  uint32_t last_integrate[8] = {};
  // staged (TMA) integrator, rr_integrate_staged.cu. `dirty` is set by everything its tables depend on (inverse volumes,
  // volume / brick grid, bricks mode, voxel format, tunables); they are rebuilt lazily by the next integrate or pre-process call.
  struct StagedIntegrator {
    bool dirty = true;             // tables below do not match the current calibration / configuration
    bool ok = false;               // the configuration fits the staged kernel
    unsigned generation = 0;       // key of the tunables the tables were built for (staged_key)
    int cy = 0, cz = 0, n_yc = 0, n_zc = 0;   // work item = brick x y-chunk x z-chunk (voxels per chunk, chunks per brick)
    int BX = 0, BY = 0, BZ = 0;    // inverse-volume box staged per item (coarse texels)
    int T = 0;                     // pair-image tile edge staged per item and sensor (pixels, even)
    int cwarps = 0, fwarps = 0;    // consumer / fill warps per CTA
    uint32_t inv_bytes = 0, tile_bytes = 0, inv_span = 0, smem_bytes = 0, fill_src_bytes = 0, fill_src_off = 0, tables_off = 0;
    uint32_t slot_bytes = 0, n_slots = 0, slots_off = 0;   // ring of per-sensor operand slots (inverse-volume box + tile)
    uint2* d_fp = nullptr;         // [items][N]: tile origin tx0 | ty0 << 16, footprint rectangle inside the tile (bit 7 of .y: exceeds the tile)
    uint32_t n_oversize = 0;       // (item, sensor) pairs of the whole brick grid whose footprint exceeds the tile
    uint2* d_list = nullptr;       // [N + 1][list_stride]: this frame's occupied items by cost class (item, verdict), k_bricks_update
    unsigned tables = 0;           // bumped by every table rebuild
    uint64_t lists_key = 0;        // staged_lists_key() the lists were classified for; 0: no valid lists (cleared by a table
                                   // rebuild, rr_bricks_clear and rr_preprocess, whose new pair image the verdicts do not describe)
    uint32_t list_stride = 0;
    float2* d_zr = nullptr;        // [items][N]: exact range of pos_calib.z over the item (k_footprints)
    uint32_t* d_err = nullptr;     // [4] device-side consistency flags (must stay 0)
    CUtensorMap map_inv, map_pairs;
  } sti;
  rr::PinnedScalars* pinned = nullptr;   // one cudaMallocHost allocation for the context's lifetime
  float* d_tsdf = nullptr;
  float* d_weight = nullptr;

  // raymarch outputs
  int view_w = 0, view_h = 0;
  float4* d_rgba = nullptr;
  float* d_zbuf = nullptr;
  float* d_nsamples = nullptr;
  float4* d_pos = nullptr;         // hit position in volume space (w = 1 on a hit)
  uint32_t* d_step = nullptr;      // step index of the hit, 0xFFFFFFFF = none (multi-GPU compositing key)
  unsigned long long* d_point_keys = nullptr;   // rr_draw_points / rr_draw_calibs: per pixel (depth bits << 32 | vertex id), atomicMin

  // rr_draw_trigrid (rr_trigrid.cu): vertex records, pass-1 depth bits, per-pixel fragment lists (grown on demand)
  rr::DeviceArray<float4> d_tg_verts;
  rr::DeviceArray<uint32_t> d_tg_depth, d_tg_head;
  rr::DeviceArray<float4> d_tg_frag_rgba, d_tg_frag_pos;
  rr::DeviceArray<uint2> d_tg_frag_link;
  rr::DeviceArray<uint32_t> d_tg_count;

  // surface extraction (rr_mesh.cu)
  bool volume_integrated = false;  // an integrate has run into the current volume allocation
  bool mesh_rows_ok = false;       // rowany / cand_y / cand_z are the tables the last integrate cleared the volume by
  bool mesh_table = false;         // the case table is in this device's constant memory
  bool mesh_valid = false;         // the d_mesh_* arrays hold an extraction of the current volume allocation (of mesh_epoch)
  uint32_t mesh_nv = 0, mesh_nt = 0;
  rr::DeviceArray<unsigned long long> d_mesh_rows;   // per row: counts and offsets of vertices, triangles
  rr::DeviceArray<uint8_t> d_mesh_scratch;           // CUB scan storage
  rr::DeviceArray<unsigned long long> d_mesh_keys;   // [V] edge key = linear index of the lower corner * 3 + axis
  rr::DeviceArray<float> d_mesh_pos, d_mesh_nrm;     // [V][3]
  rr::DeviceArray<float4> d_mesh_rgba;               // [V]
  rr::DeviceArray<uint32_t> d_mesh_tri;              // [T][3]

  // queries (rr_query.cu): inputs (points [n][3], or origins [n][3] then directions [n][3]) and per-entry results
  rr::DeviceArray<float> d_q_in, d_q_val, d_q_pos, d_q_nrm;
  rr::DeviceArray<float4> d_q_rgba;
  rr::DeviceArray<uint32_t> d_q_step;

  // point-cloud export (rr_cloud.cu): per depth pixel a keep flag, then its exclusive scan; per kept point the outputs
  bool preprocessed = false;       // an rr_preprocess / rr_fuse_frame has defined the stage images
  bool cloud_valid = false;        // the d_cloud_* arrays hold the last extraction (cloud_n points)
  uint32_t cloud_n = 0;
  rr::DeviceArray<uint32_t> d_cloud_flags;           // [2][N * W * H + 1]: flags, offsets
  rr::DeviceArray<uint8_t> d_cloud_scratch;          // CUB scan storage
  rr::DeviceArray<float> d_cloud_pos, d_cloud_nrm, d_cloud_rgb, d_cloud_q;
  rr::DeviceArray<uint32_t> d_cloud_pix;

  // connected parts (rr_parts.cu). The volume epoch advances with every integrate and every new volume allocation; the
  // mesh and the labelling record the epoch they were computed from, so rr_download_mesh_parts pairs only those of one state.
  uint64_t volume_epoch = 0, mesh_epoch = 0, parts_epoch = 0;
  bool parts_valid = false;        // d_parts_* hold the last labelling (parts_n parts)
  uint32_t parts_n = 0;
  rr::DeviceArray<uint32_t> d_parts_labels;          // [Z][Y][X]: union-find forest, then part labels
  rr::DeviceArray<uint32_t> d_parts_rows;            // [2][rows + 1]: roots per row, their offsets
  rr::DeviceArray<uint8_t> d_parts_scratch;          // CUB scan storage
  rr::DeviceArray<uint32_t> d_parts_voxels;          // per part
  rr::DeviceArray<int32_t> d_parts_boxes;            // [P][6]
  rr::DeviceArray<unsigned long long> d_parts_sums;  // [P][3]
  rr::DeviceArray<float> d_parts_centroids;          // [P][3]
  rr::DeviceArray<uint32_t> d_mesh_parts;            // [V] vertex parts, then [T] triangle parts

  // colour hole filling (rr_colorfill.cu): atlas right of column W, squeezed copy, filled colour
  int fill_w = 0, fill_h = 0;
  float4* d_fill_fc = nullptr; float* d_fill_fd = nullptr;
  float4* d_fill_sc = nullptr; float* d_fill_sd = nullptr;
  float4* d_filled = nullptr;
};

namespace rr {

// launch-shape knobs of the integrator, process-wide (rr_set_tunable / environment RR_*)
struct Tunables {
  int fused = 1;        // one persistent clear+integrate kernel (0: k_fill + k_integrate_bricks)
  int zchunk = 13;      // voxels of a brick's z extent per compute item
  int fill_rows = 16;   // voxel rows per fill item
  int fill_warps = 2;   // warps of a CTA that start on fill items
  int ctas = 2;         // resident CTAs per SM
  int threads = 512;    // CTA size (register budget): 512 (64 registers) or 384 (85 registers)
  int chunk = 1;        // compute items a CTA draws at a time (0: one z-chunk of one brick)
  int brick_grid = 6;   // grid multiple of the unfused brick kernel
  int ldg256 = 1;       // gather texels with one 256-bit load (0: two 128-bit loads)
  int graph = 1;        // rr_fuse_frame replays a captured CUDA graph (0: direct launches)
  int staged = 1;       // bricks mode uses the TMA-staged integrator when the configuration fits (0: direct kernels)
  int stage_zchunk = 13; // staged integrator: voxels of a brick's z extent per work item
  int stage_ychunk = 0; // ... and of its y extent (0: chosen so that an item's columns fill the consumer threads)
  int stage_tile = 0;   // pair-image tile edge in pixels (0: chosen from the footprint statistics and the smem budget)
  int stage_fill_rows = 16;   // voxel rows per fill item
  int stage_cwarps = 0; // consumer warps per CTA: 0 = 22 up to four sensors (80 registers), 11 = half of that at 144 registers
  int stage_bulk_fill = 4;    // KB of cleared voxels in shared memory, the source of the clear's TMA bulk stores
  int stage_fill_depth = 0;   // bulk-store groups a clear lane may leave pending (-1: unbounded)
 int stage_tail_cap = 2;     // items in flight per CTA towards the end of the item list (0: the ring's capacity throughout)
  int stage_ctas = 0;         // CTAs of the staged integrator (0: one per SM)
  int stage_fill_lsu = 0;     // 1: rows without occupied bricks are cleared by per-lane stores instead of bulk stores
  int fuse_nq = 1;            // pre_normal + pre_quality in one launch (k_normal_quality; 0: the two kernels)
  int trigrid_pool = 64;      // rr_draw_trigrid: initial capacity of the fragment pool, in fragments per 16 view pixels (it grows on demand)
  int stage_debug = 0;  // measurement only, results are WRONG: bit 0 skips the clear stream, bit 1 the brick evaluation
  unsigned generation = 0;   // bumped by every rr_set_tunable (invalidates captured graphs)
};
Tunables& tunables();

int fail(rr_ctx* c, int code, const std::string& msg);
int check(rr_ctx* c, cudaError_t e, const char* what);
void timer_begin(rr_ctx* c, const char* name);
void timer_end(rr_ctx* c, const char* name);
SensorTables sensor_tables(const rr_ctx* c);

// kernels' host launchers (one translation unit each)
int launch_preprocess(rr_ctx* c, int filter_textures, int use_processed_depth, int refine);
int launch_pack_gather(rr_ctx* c);    // the gather texels of the direct integrators from the last pre-process's stage images
int launch_bricks_clear(rr_ctx* c);
int launch_bricks_update(rr_ctx* c);
int launch_integrate(rr_ctx* c);
int launch_raymarch(rr_ctx* c, const rr_view* v);
int launch_pack_partial(rr_ctx* c, float4* d_rec);
int launch_composite(rr_ctx* c, const float4* d_rec, int n_parts);
int launch_partial_keys(rr_ctx* c, const float4* d_rec, int rank, long long* d_keys);
int launch_partial_keep(rr_ctx* c, float4* d_rec, const long long* d_keys_min, int rank);
int launch_fill_colors(rr_ctx* c);
int launch_draw_points(rr_ctx* c, const rr_view* v, int mode, float calib_limit);   // rr_points.cu
int launch_draw_trigrid(rr_ctx* c, const rr_view* v, float min_length);             // rr_trigrid.cu
int launch_extract_mesh(rr_ctx* c, uint32_t* out_nv, uint32_t* out_nt);   // rr_mesh.cu: the whole volume, ignoring the slab
bool mesh_rows_usable(const rr_ctx* c);   // the last integrate cleared everything outside the occupied bricks of the row tables
// rr_query.cu: rr_sample_points / rr_cast_rays. query_upload copies the inputs (b: the directions, NULL for points) into
// d_q_in, the launchers evaluate the context's own slab (a group member evaluates only what it owns), query_download
// copies the requested results out and synchronises once.
int query_check(rr_ctx* c, int space, uint32_t count, bool have_inputs, bool whole_volume, const char* who);   // rr_api.cu
int query_reserve(rr_ctx* c, uint32_t count);
int query_upload(rr_ctx* c, const float* a, const float* b, uint32_t count);
int launch_sample_points(rr_ctx* c, int space, uint32_t count);
int launch_cast_rays(rr_ctx* c, int space, uint32_t count);
int launch_query_composite(rr_ctx* const* members, int n, bool rays, int space, uint32_t count);   // on member 0's stream
int query_download(rr_ctx* c, uint32_t count, bool rays, float* values_or_positions, float* normals, float* rgba, uint32_t* steps);
// rr_cloud.cu: rr_extract_points over the sensors of `mask` (checked by the caller); cloud_download copies the last extraction
// out and synchronises once
int launch_extract_points(rr_ctx* c, uint32_t mask, uint32_t* out_n);
int cloud_download(rr_ctx* c, float* positions, float* normals, float* colors, float* quality, uint32_t* pixels);
// rr_parts.cu: rr_label_parts over the whole volume, ignoring the slab; the downloads copy out and synchronise once
int launch_label_parts(rr_ctx* c, uint32_t* out_num_parts);
int parts_download(rr_ctx* c, uint32_t* voxels, int32_t* boxes, float* centroids, uint32_t* labels);
int mesh_parts_download(rr_ctx* c, uint32_t* vertex_parts, uint32_t* triangle_parts);   // the mesh and labelling of one epoch
int launch_unpack_frames(rr_ctx* c, int slot);
int launch_calib_invert(rr_ctx* c, int sensor, const uint32_t out_res[3], float4* d_out);
int staged_prepare(rr_ctx* c);        // (re)builds the staged integrator's tables when dirty; RR_OK also when it declines
void staged_release(rr_ctx* c);
bool staged_selected(const rr_ctx* c); // after staged_prepare: the next bricks-mode integrate runs the staged kernel
uint64_t staged_lists_key(const rr_ctx* c);   // what the item lists depend on besides the frame: table rebuild, limit
void drop_frame_graphs(rr_ctx* c);

// host geometry (rr_host_geom.cpp)
void host_frustum(const float* cv_xyz, const uint32_t res[3], float planes[6][4], float cam[3]);
void host_volume_res(const float bmin[3], const float bmax[3], float voxel_size, uint32_t res[3]);
float host_adjust_brick_size(float voxel_size, float size);
uint32_t host_divide_box(const float bmin[3], const float bmax[3], float brick_size, const uint32_t res[3],
                         uint32_t res_bricks[3], std::vector<int32_t>* ranges);

}  // namespace rr

#define RR_TRY_RC(expr) do { int rc__ = (expr); if (rc__ != RR_OK) return rc__; } while (0)

#define RR_LAUNCH_CHECK(c, what)                                   \
  do {                                                             \
    ++(c)->launches;                                               \
    cudaError_t e__ = cudaGetLastError();                          \
    if (e__ != cudaSuccess) return rr::check((c), e__, (what));    \
  } while (0)

// Grows to `need` elements plus 1/8 slack; a queued kernel or copy may still read the old memory, so the stream drains first.
template <typename T>
int rr::DeviceArray<T>::reserve(rr_ctx* c, size_t need, const char* what) {
  if (need <= cap) return RR_OK;
  if (ptr) {
    RR_TRY_RC(rr::check(c, cudaStreamSynchronize(c->stream), what));
    release();
  }
  const size_t n = need + need / 8 + 1;
  RR_TRY_RC(rr::check(c, cudaMalloc((void**)&ptr, n * sizeof(T)), what));
  cap = n;
  return RR_OK;
}
