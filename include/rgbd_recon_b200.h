/* rgbd_recon_b200.h — C ABI of the B200-native volumetric-fusion path (librr_b200.so).
 *
 * The reference (steppobeck/rgbd-recon) has no plugin/FFI interface: its boundary is the public C++ surface that
 * source/kinect_client.cpp calls plus implicit OpenGL state (SURVEY.md §8b). Each entry point below names the
 * reference interface it stands in for (paths relative to the reference root). The kept C++ classes
 * (rgbd-recon_b200/host/: kinect::CalibVolumes, NetKinectArray, ReconIntegration, CalibrationInverter) are thin
 * shims over these calls. No OpenGL context, no torch types; plain pointers and sizes only.
 *
 * Conventions: every call returns 0 on success or a negative rr_status; rr_last_error(ctx) gives the text.
 * A context is single-caller (the reference issues everything from its one GL thread) and owns one CUDA stream
 * on one device. The one exception mirrors the reference's reader thread (NetKinectArray::readLoop): rr_stage_frames and
 * rr_stage_sync may be called from a second thread while the first one runs the per-frame calls, provided the two threads
 * order rr_stage_frames against rr_swap_frames themselves (the reference's m_mutex_pbo); rr_last_error returns a per-thread
 * copy of the text. Host pointers passed in stay owned by the caller. Arrays are C-contiguous:
 *   depth  float32 [N][H][W]        metres, 0 = no return       (NetKinectArray.cpp:135-142)
 *   colour uint8   [N][CH][CW][3]   RGB8                        (NetKinectArray.cpp:120-131)
 *   cv_xyz float32 [Z][Y][X][3], cv_uv float32 [Z][Y][X][2], cv_xyz_inv float32 [Z][Y][X][4]
 *                                   index z*X*Y + y*X + x       (framework/calibration/calibration_volume.hpp:18-27)
 *   tsdf   float32 [Z][Y][X]        x fastest                   (glsl/tsdf_integration.vs:57-58)
 */
#ifndef RGBD_RECON_B200_H
#define RGBD_RECON_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rr_ctx rr_ctx;

typedef enum rr_status {
  RR_OK = 0,
  RR_ERR_INVALID = -1,     /* bad argument / call order */
  RR_ERR_CUDA = -2,        /* CUDA runtime failure (text in rr_last_error) */
  RR_ERR_NO_DEVICE = -3,   /* no usable GPU: there is no CPU fallback */
  RR_ERR_UNSUPPORTED = -4
} rr_status;

/* How a voxel is stored (rr_config.store_weight). */
enum rr_voxel_format { RR_VOXELS_F32 = 0, RR_VOXELS_F32_WEIGHT = 1, RR_VOXELS_HALF2 = 2 };

/* Runtime knobs of ReconIntegration (framework/reconstruction/recon_integration.cpp:30-60, kinect_client.cpp:87-93). */
typedef struct rr_config {
  float limit;                    /* TSDF truncation in normalised sensor-depth units (setTsdfLimit)            */
  float voxel_size;               /* metres (setVoxelSize, :341-354)                                            */
  float brick_size;               /* metres, rounded to a voxel multiple (setBrickSize, :474-484)               */
  uint32_t min_voxels_per_brick;  /* setMinVoxelsPerBrick, default 10                                           */
  int32_t use_bricks;             /* setUseBricks: integrate occupied bricks only                               */
  int32_t skip_space;             /* setSpaceSkip: raymarch starts/ends at the occupied-brick hull              */
  int32_t store_weight;           /* voxel format, an rr_voxel_format: 0 = R32F tsdf like the reference's image3D
                                     (recon_integration.cpp:86-95); 1 = also keep the shader-local total_weight
                                     in a second R32F volume; 2 = half2 voxels (tsdf, weight), both rounded to
                                     nearest-even binary16 at the store (BASELINE config 5)                        */
} rr_config;

/* Inputs of ReconIntegration::draw (recon_integration.cpp:177-241): the fixed-function matrices it reads back,
 * column-major float[16] like gloost::Matrix / glGetFloatv. */
typedef struct rr_view {
  float modelview[16];
  float projection[16];
  int32_t viewport[4];            /* x, y, width, height (glGetIntegerv(GL_VIEWPORT))                           */
  int32_t shade_mode;             /* Settings.g_shade_mode, glsl/shading.glsl:14-21: 0 colour 1 shaded 2 normal 3 camera */
} rr_view;

/* Intermediate images a test or GUI texture viewer can read back (kinect_client.cpp:486-518). */
typedef enum rr_stage {
  RR_STAGE_MORPH = 0,       /* float32 [N][H][W]     m_textures_depth2.front  */
  RR_STAGE_DEPTH = 1,       /* float32 [N][H][W][2]  m_textures_depth         */
  RR_STAGE_LAB = 2,         /* float32 [N][H][W][3]  m_textures_color         */
  RR_STAGE_DEPTH_B = 3,     /* float32 [N][H][W][2]  m_textures_depth_b       */
  RR_STAGE_SILHOUETTE = 4,  /* float32 [N][H][W]     m_textures_silhouette    */
  RR_STAGE_NORMAL = 5,      /* float32 [N][H][W][3]  m_textures_normal        */
  RR_STAGE_QUALITY = 6      /* float32 [N][H][W]     m_textures_quality       */
} rr_stage;

/* ---- lifetime ------------------------------------------------------------------------------------------- */
/* Replaces the GL object ownership spread over NetKinectArray::init (NetKinectArray.cpp:114-219),
 * CalibVolumes::createVolumeTextures (CalibVolumes.cpp:132-144) and the ReconIntegration ctor. */
int rr_create(rr_ctx** out, int device, int num_sensors, int depth_w, int depth_h, int color_w, int color_h);
void rr_destroy(rr_ctx* ctx);
const char* rr_last_error(const rr_ctx* ctx);
int rr_synchronize(rr_ctx* ctx);
/* The CUDA stream (cudaStream_t) all work of this context is enqueued on; for event timing by the caller. */
void* rr_stream(rr_ctx* ctx);

/* ---- calibration (CalibVolumes) -------------------------------------------------------------------------- */
/* CalibVolumes ctor: bbox UBO binding 2 (CalibVolumes.cpp:45-49). */
int rr_set_bbox(rr_ctx* ctx, const float bbox_min[3], const float bbox_max[3]);
/* CalibVolumes::addVolume + createVolumeTextures (CalibVolumes.cpp:115-144). Also derives the sensor frustum and
 * camera position (Frustum::getCameraPos, frustum.cpp:21-33) used by the quality pass. */
int rr_calib_upload(rr_ctx* ctx, int sensor, const float* cv_xyz, const float* cv_uv, const uint32_t res[3],
                    const float depth_limits[2]);
/* CalibVolumes::loadInverseCalibs (CalibVolumes.cpp:64-80). All sensors must share one resolution (getVolumeRes). */
int rr_calib_upload_inv(rr_ctx* ctx, int sensor, const float* cv_xyz_inv, const uint32_t res[3]);
/* CalibVolumes::getCameraPositions (CalibVolumes.cpp:224-230): out float[N][3]. */
int rr_get_camera_positions(const rr_ctx* ctx, float* out);
/* CalibVolumes::getFrustum(i): the six planes (float[6][4]) of frustum.cpp:166-176. */
int rr_get_frustum_planes(const rr_ctx* ctx, int sensor, float* out);
/* CalibrationInverter::calculateInverseVolumes for one sensor (calibration_inverter.cpp:99-155): exact 8-NN +
 * inverse-distance weighting + frustum cull on the GPU. host_out: float32 [res.z][res.y][res.x][4]. Synchronous.
 * If keep_on_device != 0 the result also becomes the sensor's inverse volume (as rr_calib_upload_inv would). */
int rr_calib_invert(rr_ctx* ctx, int sensor, const uint32_t out_res[3], float* host_out, int keep_on_device);

/* ---- settings (ReconIntegration setters) ------------------------------------------------------------------ */
/* setVoxelSize / setBrickSize / setTsdfLimit / setMinVoxelsPerBrick / setUseBricks / setSpaceSkip in one call;
 * (re)allocates the volume and rebuilds the brick table (divideBox, recon_integration.cpp:361-407). */
int rr_configure(rr_ctx* ctx, const rr_config* cfg);
int rr_get_volume_res(const rr_ctx* ctx, uint32_t res[3]);
/* numBricks / getBrickSize / m_res_bricks. Any out pointer may be NULL. */
int rr_get_brick_info(const rr_ctx* ctx, uint32_t res_bricks[3], float* brick_size, uint32_t* num_bricks);
/* Per-brick voxel ranges int32 [num_bricks][6] = x0,x1,y0,y1,z0,z1 (VolumeSampler::containedVoxels). */
int rr_get_brick_ranges(const rr_ctx* ctx, int32_t* out);
/* Multi-GPU: this context owns voxel slices z in [z0, z1) (SURVEY.md §8e): it raymarches only samples whose nearest z
 * texel it owns and integrates its slab plus a read-only halo of ceil(limit * Z) + 2 slices. Default: the whole volume. */
int rr_set_slab(rr_ctx* ctx, uint32_t z0, uint32_t z1);

/* ---- per frame (NetKinectArray + ReconIntegration) -------------------------------------------------------- */
/* The reference double-buffers ingest (double_pixel_buffer.cpp:18-33,57-82): the reader thread fills the back PBO while
 * the main thread draws from the front one, and NetKinectArray::update (NetKinectArray.cpp:226-238) swaps them. Here:
 *   rr_stage_frames  = the reader's write: one frame set, host buffers (pinned for overlap) -> the BACK device slot,
 *                      asynchronously on a copy stream, overlapping kernels that still read the current slot.
 *                      color may be NULL if no colour is needed (the slot keeps its previous colour).
 *   rr_swap_frames   = update(): the staged slot becomes current; the compute stream waits for the staged copies.
 *   rr_stage_sync    = host wait until the staged copies have completed (the host buffers may be reused).
 *   rr_upload_frames = rr_stage_frames + rr_swap_frames (no overlap; the simple path). */
int rr_stage_frames(rr_ctx* ctx, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes);
/* Stream formats of the reference (KinectCalibrationFile compress_rgb / compress_depth; NetKinectArray.cpp:120-142,
 * 149-159,170-175): colour RGB8 [N][CH][CW][3], DXT1 blocks (compress_rgb == 1: CW*CH/2 bytes per sensor) or DXT5 blocks
 * (compress_rgb == 5, :125-128,153-156: CW*CH bytes per sensor - the reference hard-codes 307200 = 640*480; the alpha half of a
 * block is not sampled downstream and is skipped); CW and CH multiples of 4 for both block formats;
 * depth float32 metres [N][H][W] or 8-bit sqrt-compressed [N][H][W] with per-sensor (near, far) of the calibration file
 * (near_far float [N][2]; pre_depth.fs uncompress(), :51-61, with scale = far - near). Sets the sizes the upload calls
 * expect; packed frame sets are expanded on the device. Default: RGB8 + float32. */
#define RR_COLOR_RGB8 0
#define RR_COLOR_DXT1 1
#define RR_COLOR_DXT5 5
#define RR_DEPTH_F32 0
#define RR_DEPTH_U8 1
int rr_set_frame_format(rr_ctx* ctx, int color_format, int depth_format, const float* near_far);
int rr_swap_frames(rr_ctx* ctx);
int rr_stage_sync(rr_ctx* ctx);
int rr_upload_frames(rr_ctx* ctx, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes);
/* Same, but the frame set is already in device memory of this context's GPU (e.g. after an NCCL broadcast). */
int rr_upload_frames_device(rr_ctx* ctx, const void* d_color, size_t color_bytes, const void* d_depth, size_t depth_bytes);
/* ReconIntegration::clearOccupiedBricks (recon_integration.cpp:272-278). */
int rr_bricks_clear(rr_ctx* ctx);
/* NetKinectArray::processTextures (NetKinectArray.cpp:311-428): morph -> bilateral -> boundary -> normal(+bricks)
 * -> quality, with the flags of filterTextures / useProcessedDepths / refineBoundary. */
int rr_preprocess(rr_ctx* ctx, int filter_textures, int use_processed_depth, int refine_boundary);
/* ReconIntegration::updateOccupiedBricks (recon_integration.cpp:431-446), on the device (ordered compaction).
 * If either out pointer is non-NULL the call synchronises to return the count / occupied ratio. */
int rr_bricks_update(rr_ctx* ctx, uint32_t* out_num_occupied, float* out_ratio);
/* ReconIntegration::integrate (recon_integration.cpp:243-270) + glsl/tsdf_integration.vs. Uses
 *  - the configuration in effect at the call (limit, bricks or dense, voxel format; a setter between the stages of a frame
 *    takes effect here),
 *  - the stage images of the last rr_preprocess,
 *  - the occupied list of the last rr_bricks_update, or an empty list if rr_configure rebuilt the brick grid since (a new
 *    voxel or brick size). rr_bricks_clear does not empty it.
 * Tunables (rr_set_tunable) select kernels and launch shapes, never results. */
int rr_integrate(rr_ctx* ctx);
/* The whole per-frame-set sequence of kinect_client.cpp:572-600 after NetKinectArray::update() in ONE call:
 * clearOccupiedBricks -> processTextures -> updateOccupiedBricks -> integrate (= rr_bricks_clear, rr_preprocess,
 * rr_bricks_update(NULL, NULL), rr_integrate). With stage timing off the launch sequence is captured once per
 * (frame slot, flags) as a CUDA graph and replayed, so a frame costs one launch on the host; any rr_configure /
 * rr_set_slab / rr_set_frame_format / calibration upload / rr_set_tunable drops the captured graphs. Same results. */
int rr_fuse_frame(rr_ctx* ctx, int filter_textures, int use_processed_depth, int refine_boundary);
/* ReconIntegration::numBricks / occupiedRatio (recon_integration.hpp:58-60) for the last rr_bricks_update / rr_fuse_frame:
 * waits for the context's stream, then returns the occupied-brick count and count / number of bricks. No launch. */
int rr_bricks_count(rr_ctx* ctx, uint32_t* out_num_occupied, float* out_ratio);
/* ReconIntegration::drawF/draw (recon_integration.cpp:151-241) + glsl/tsdf_raymarch.fs, bricks.{vs,gs,fs}.
 * out_rgba float32 [h][w][4], out_depth float32 [h][w] (gl_FragDepth, 1.0 where no surface), both host, may be NULL. */
int rr_raymarch(rr_ctx* ctx, const rr_view* view, float* out_rgba, float* out_depth);

/* The point-drawing consumers of the pre-processed maps (SURVEY.md §8f-4), without a rasteriser: one thread per vertex splats
 * a depth-tested square (64-bit atomicMin of depth | vertex id: the first drawn fragment wins depth ties, as GL_LESS), one
 * thread per pixel shades the winner. Both write the context's view images like rr_raymarch (rgba float32 [h][w][4] with
 * alpha 1 on covered pixels and all zeros elsewhere; depth float32 [h][w], 1.0 where nothing was drawn).
 *   rr_draw_points  ReconPoints::draw (recon_points.cpp:71-111; glsl/points.vs, points.gs, points.fs): every depth pixel of
 *                   every sensor (the maps of the last rr_preprocess) as a square of (shade mode 3: 4, else 10) / |pos_eye|
 *                   pixels, shaded from the sensor's colour and normal maps (rr_view.shade_mode as in rr_raymarch).
 *   rr_draw_calibs  ReconCalibs::draw (recon_calibs.cpp:56-66; glsl/calib_vis.vs, calib_vis.fs; VolumeSampler::sample): every
 *                   voxel centre of the inverse-volume grid as a one-pixel point coloured by the TSDF there (red outside,
 *                   green inside, blue at >= limit, nothing at <= -limit). active_kinect only selects lookups whose results
 *                   the shader never uses; tsdf_limit is ReconCalibs' own limit (setTsdfLimit, default 0.01). */
int rr_draw_points(rr_ctx* ctx, const rr_view* view, float* out_rgba, float* out_depth);
int rr_draw_calibs(rr_ctx* ctx, const rr_view* view, int active_kinect, float tsdf_limit, float* out_rgba, float* out_depth);

/* ReconTrigrid::draw (recon_trigrid.cpp:82-149; glsl/trigrid_accum.vs, trigrid_accum.gs, trigrid_accum.fs,
 * trigrid_normalize.fs), the triangle-mesh consumer of the pre-processed maps (SURVEY.md §8f-4): every depth pixel of every
 * sensor spans two triangles (the grid of :48-61, as written there: cells x < height, y < width); pass 1 keeps the nearest
 * window depth of the triangles that survive validSurface (no invalid depth, every edge shorter than
 * min_length * average depth * 4), the bounding box, the colour view's border and back-face culling; pass 2 adds
 * shade() * quality, quality of every fragment within epsilon = 0.075 (:35) of that surface; pass 3 divides by the summed
 * quality. A software rasteriser (OpenGL 4.4 clipping, coverage and perspective-correct interpolation in fp64) that walks the
 * triangles once for both passes and performs the additive blend in draw order (per-pixel fragment lists, epsilon-tested against
 * the final depth and summed by ascending triangle id), so the result is deterministic.
 * min_length: CalibrationFiles::minLength() (the sensor .yml's "min_length:", default 0.0125, KinectCalibrationFile.cpp:96,341).
 * Writes the context's view images like rr_raymarch: rgba float32 [h][w][4] (alpha 1 where something was drawn, zeros
 * elsewhere), depth float32 [h][w] (pass 1's depth, 1.0 elsewhere). Synchronises the context's stream once per call. */
int rr_draw_trigrid(rr_ctx* ctx, const rr_view* view, float min_length, float* out_rgba, float* out_depth);

/* ReconIntegration::fillColors (recon_integration.cpp:280-339; on by default, m_fill_holes, :54) + ViewLod
 * (view_lod.cpp:24-61) + glsl/framebuffer_transfer.fs, tsdf_inpaint.fs, tsdf_colorfill.fs: push-pull colour hole filling
 * of the LAST view (rr_raymarch, rr_composite or rr_upload_view): pixels the raymarch hit but could only colour with the
 * fallback blend (alpha -1) take colour from the coarser lods of the mip atlas. out_rgba float32 [h][w][4], host, may be
 * NULL; pixels without a surface keep the raymarch value. setColorFilling(false) = do not call it. */
int rr_fill_colors(rr_ctx* ctx, float* out_rgba);
/* Test hook: make host images the "last view" (rgba float32 [h][w][4], depth float32 [h][w]) so that rr_fill_colors can
 * be checked on arbitrary inputs. */
int rr_upload_view(rr_ctx* ctx, int width, int height, const float* rgba, const float* depth);

/* Multi-GPU view (z-slab sharding, SURVEY.md §8e): every slab context marches its own samples and writes one 32-byte
 * record per pixel {float rgba[4]; float depth; uint32 first_hit_step (0xFFFFFFFF none); float sample_count; float 0}
 * into d_records (DEVICE memory, viewport w*h records). The records of all slabs are gathered (one NCCL gather) into
 * n_parts consecutive images on the display GPU, where rr_composite keeps, per pixel, the record with the smallest
 * step index — the hit ReconIntegration::draw would have found first — and optionally downloads colour and depth. */
#define RR_PARTIAL_RECORD_BYTES 32
int rr_raymarch_partial(rr_ctx* ctx, const rr_view* view, void* d_records);
int rr_composite(rr_ctx* ctx, const void* d_records, int n_parts, int width, int height, float* out_rgba, float* out_depth);
/* The same compositing by two reductions instead of a gather, so that the display GPU does not receive one record image
 * per slab (tsdf_raymarch.fs:92-142 finds ONE first hit per ray; so does this):
 *   rr_partial_keys         d_keys[i] (int64, DEVICE, w*h) = first_hit_step << 8 | rank for the records of the last
 *                           rr_raymarch_partial; an all-reduce MIN over the ranks names every pixel's winner (smallest
 *                           step, lowest rank on ties - exactly rr_composite's choice);
 *   rr_partial_keep_winners zeroes this rank's record wherever it is not the winner; an integer SUM reduce of the records
 *                           (8 x uint32 per pixel) onto the display GPU then yields the winner's record bit for bit, and
 *                           rr_composite(..., n_parts = 1) turns it into the view. */
int rr_partial_keys(rr_ctx* ctx, const void* d_records, int rank, void* d_keys);
int rr_partial_keep_winners(rr_ctx* ctx, void* d_records, const void* d_keys_min, int rank);

/* ---- one process, several GPUs (SURVEY.md §8e; no reference counterpart - the reference owns one GL context) ---------- */
/* A group = one rr_ctx per device; the TSDF volume is split into contiguous z-slabs, one per member. Every call below is the
 * group form of the per-context call of the same name and has the same meaning and error behaviour; setup is replicated,
 * a frame set goes host -> member 0 (the ingest and display device) -> the other members by peer copies over NVLink on
 * their copy streams (double-buffered like rr_stage_frames), pre-processing and brick tables are replicated, each member
 * integrates its slab, and a view is marched per slab and composited by ONE kernel on member 0 that reads the other
 * members' first-hit keys and the winners' pixels through peer memory. Results equal the single-context ones bit for bit
 * (tests/test_group_gpu.py). A group of one device is a plain pass-through. Single caller, like a context.
 * rr_group_last_error gives the text of the last failing group call (naming the member). */
typedef struct rr_group rr_group;
int rr_group_create(rr_group** out, const int* devices, int n_devices, int num_sensors, int depth_w, int depth_h, int color_w, int color_h);
void rr_group_destroy(rr_group* g);
int rr_group_size(const rr_group* g);
rr_ctx* rr_group_member(rr_group* g, int i);      /* for per-context queries and read-backs (member 0: brick tables, timers, view) */
const char* rr_group_last_error(const rr_group* g);
int rr_group_synchronize(rr_group* g);
int rr_group_set_bbox(rr_group* g, const float bbox_min[3], const float bbox_max[3]);
int rr_group_calib_upload(rr_group* g, int sensor, const float* cv_xyz, const float* cv_uv, const uint32_t res[3], const float depth_limits[2]);
int rr_group_calib_upload_inv(rr_group* g, int sensor, const float* cv_xyz_inv, const uint32_t res[3]);
int rr_group_set_frame_format(rr_group* g, int color_format, int depth_format, const float* near_far);
int rr_group_set_timing(rr_group* g, int level);
/* rr_configure on every member, then equal-thickness slabs (rr_set_slab). */
int rr_group_configure(rr_group* g, const rr_config* cfg);
/* Explicit slab boundaries z_bounds[n + 1] (ascending, tiling [0, Z)); rr_group_get_slabs reads them back. */
int rr_group_set_slabs(rr_group* g, const uint32_t* z_bounds);
int rr_group_get_slabs(const rr_group* g, uint32_t* z_bounds);
/* Slabs of equal integrate cost (clear stream + compute_to_fill x voxels of occupied bricks per slice; <= 0: the measured 45)
 * from the occupied bricks of the last fused frame set. Synchronises; for occasional use. */
int rr_group_balance_slabs(rr_group* g, float compute_to_fill);
int rr_group_stage_frames(rr_group* g, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes);
int rr_group_swap_frames(rr_group* g);
int rr_group_stage_sync(rr_group* g);
int rr_group_upload_frames(rr_group* g, const void* color, size_t color_bytes, const void* depth, size_t depth_bytes);
int rr_group_bricks_clear(rr_group* g);
int rr_group_preprocess(rr_group* g, int filter_textures, int use_processed_depth, int refine_boundary);
int rr_group_bricks_update(rr_group* g, uint32_t* out_num_occupied, float* out_ratio);
int rr_group_integrate(rr_group* g);
int rr_group_fuse_frame(rr_group* g, int filter_textures, int use_processed_depth, int refine_boundary);
int rr_group_bricks_count(rr_group* g, uint32_t* out_num_occupied, float* out_ratio);
int rr_group_raymarch(rr_group* g, const rr_view* view, float* out_rgba, float* out_depth);
int rr_group_fill_colors(rr_group* g, float* out_rgba);
/* The whole volume assembled from the slices each member owns: float32 [Z][Y][X] (4-byte voxels of any format). */
int rr_group_download_tsdf(rr_group* g, float* out);

/* The group's compositing with one process per GPU (torchrun / MPI): every rank marches its slab with rr_raymarch (no
 * download), exports its view images once per viewport size (rr_view_export: RR_VIEW_HANDLE_BYTES of CUDA IPC handles, to be
 * sent to the display rank by any means), and the display rank composites its own view with the peers' directly out of their
 * memory (rr_composite_peers, the kernel of rr_group_raymarch). The caller orders the ranks: the peers' marches must have
 * completed before the call (e.g. a stream-ordered NCCL barrier) and the peers must not march again before it has finished. */
#define RR_VIEW_HANDLE_BYTES 256
int rr_view_export(rr_ctx* ctx, int width, int height, void* out_handle);
int rr_composite_peers(rr_ctx* ctx, const void* peer_handles, int n_peers, int width, int height, float* out_rgba, float* out_depth);

/* ---- surface extraction (no reference counterpart: the reference only raymarches the volume) ---------------------------
 * The fused surface as an indexed triangle mesh with per-vertex normals and colours, by marching cubes on the device.
 *   Grid      corner (x, y, z) = the voxel centre; its value v is the density rr_raymarch reads (R32F, or the low half of a
 *             half2 voxel widened; F32_WEIGHT: the tsdf volume only). Cell = the cube of corners x..x+1, y..y+1, z..z+1 for
 *             x < X-1, y < Y-1, z < Z-1. Inside: v > 0 (the raymarch's hit test); outside: v <= 0. A cell with a
 *             non-finite corner emits nothing.
 *   Cases     generated from a rule, not transcribed: on each cube face two crossed edges give one segment, four crossed
 *             edges the two segments that cut off the inside corners (so neighbouring cells agree along every face and the
 *             mesh is crack-free); the segments are chained into loops oriented counter-clockwise seen from the outside,
 *             so geometric normals point to free space; each loop is a fan from its lowest edge, loops by lowest edge.
 *   Vertices  one per crossed edge (one end > 0, the other <= 0, both finite, on at least one emitting cell), ordered by
 *             edge key (linear index of the lower corner a, then axis x < y < z). Along axis k from a to b:
 *             t = va / (va - vb); texture coordinate q_k = ((float)i_k + 0.5f + t) / (float)R_k, the other two the voxel
 *             centre ((float)i + 0.5f) * (1.0f / (float)R); position (metres) = bbox_min + q * (bbox_max - bbox_min),
 *             binary32 without fused multiply-adds.
 *             normal = normalize(g / (bbox_max - bbox_min)) with g the raymarch's gradient at q (step limit / 2, normalised,
 *             negated; NaN where it vanishes); rgba = blendColors at q (shade mode 0's diffuse colour; alpha 1 when
 *             quality-weighted, -1 for the fallback blend) from the limit, stage images and colour rr_raymarch would use now.
 *   Triangles three uint32 vertex indices, ordered by cell linear index (z, y, x), then by table order within the cell.
 * The order is canonical: it depends neither on scheduling, on the occupied-brick shortcut (in bricks mode only cells
 * near occupied bricks are visited while the brick tables are the ones the volume was integrated with; otherwise every
 * cell is) nor on the number of devices. The result always equals marching cubes over the volume rr_download_tsdf returns.
 *
 * rr_extract_mesh   extracts on the context's stream and synchronises once; returns the counts. RR_ERR_INVALID before any
 *                   integrate into the current volume (an rr_configure that changes the resolution or the voxel format
 *                   starts a new one; a new limit does not) and on a context restricted by rr_set_slab (use
 *                   rr_group_extract_mesh); RR_ERR_UNSUPPORTED for 2^31 or more vertices or triangles. Changes nothing
 *                   else: volume, view images, brick tables and captured frame graphs stay as they are.
 * rr_download_mesh  the last extraction: positions float32 [V][3], normals float32 [V][3], rgba float32 [V][4], triangles
 *                   uint32 [T][3], host, each may be NULL. RR_ERR_INVALID if nothing was extracted from the current volume.
 * rr_group_extract_mesh  the same for a group, bit for bit: member 0 receives the other members' slabs by peer copies (one
 *                   volume per call; its own unowned slices are overwritten, which nothing else reads) and extracts; read
 *                   the mesh with rr_download_mesh(rr_group_member(g, 0), ...). */
int rr_extract_mesh(rr_ctx* ctx, uint32_t* out_num_vertices, uint32_t* out_num_triangles);
int rr_download_mesh(rr_ctx* ctx, float* positions, float* normals, float* rgba, uint32_t* triangles);
int rr_group_extract_mesh(rr_group* g, uint32_t* out_num_vertices, uint32_t* out_num_triangles);

/* ---- mesh simplification (no reference counterpart) --------------------------------------------------------------------
 * A smaller indexed mesh from the last mesh of rr_extract_mesh / rr_group_extract_mesh, by vertex clustering with clusters
 * of c = cluster_voxels voxels per side (c >= 1). Every vertex of the mesh has an edge key (lower corner (x, y, z), axis).
 *   Cluster   of a vertex: (x / c, y / c, z / c) by integer division; id = (z/c * CY + y/c) * CX + x/c with CX = ceil(X / c),
 *             likewise CY and CZ (ids stay below X*Y*Z < 2^31).
 *   Triangles each mesh triangle (i, j, k) becomes (C(i), C(j), C(k)). It is dropped if two of the three are equal; otherwise
 *             it is rotated so that the smallest comes first (cyclic order and orientation kept). Among triangles with the
 *             same rotated triple only the one with the smallest source index is kept (opposite orientations are different
 *             triples: both are kept). Order: ascending source triangle; sources uint32 [T'] = the index of each kept
 *             triangle's source triangle in the last mesh (e.g. for rr_download_mesh_parts' triangle parts).
 *   Vertices  one per cluster a kept triangle references, in ascending cluster id; a vertex's index is its rank in that list.
 *             Position p_k = (float)(S_k / n): n = the number of mesh vertices in the cluster (all of them, also those whose
 *             triangles were all dropped), S_k = the binary64 sum of their coordinate k, each widened from binary32, from +0.0
 *             one vertex at a time in ascending edge key; IEEE binary64 division, rounded to nearest; no fused multiply-adds.
 *             normal and rgba = exactly what rr_sample_points(RR_QUERY_WORLD) returns at p, evaluated over the whole volume
 *             whatever rr_set_slab says (NaN normal and rgba 0 outside the unit cube).
 * The order of every output depends neither on scheduling nor on the number of devices. Cost: one thread per cluster sums its
 * members, and a cluster holds at most 3*c^3 vertices: c <= 8 is the intended range, a larger c is correct but slow.
 *
 * rr_simplify_mesh   simplifies on the context's stream and synchronises once; returns the counts (never more than the
 *                   mesh's). RR_ERR_INVALID for cluster_voxels == 0, a NULL count pointer, no mesh, or a mesh of an older
 *                   volume state (an integrate or a new volume since the extraction). Not a setting: the mesh
 *                   (rr_download_mesh, rr_download_mesh_parts), volume, brick tables, view images (rr_fill_colors still
 *                   fills the last view), cloud, parts, query results, captured frame graphs and rr_integrator_last stay as
 *                   they are.
 * rr_download_simplified_mesh  the last simplification: positions float32 [V'][3], normals float32 [V'][3], rgba float32
 *                   [V'][4], triangles uint32 [T'][3], sources uint32 [T']; each pointer may be NULL, host memory (pageable or
 *                   pinned) or device memory of the context's GPU. Returns after one synchronisation. RR_ERR_INVALID before
 *                   any simplification of the current volume allocation.
 * rr_group_simplify_mesh  the same on member 0 of a group right after rr_group_extract_mesh (member 0 then holds the gathered
 *                   volume and the mesh), with no peer traffic, equal to a single context bit for bit; read it with
 *                   rr_download_simplified_mesh(rr_group_member(g, 0), ...). */
int rr_simplify_mesh(rr_ctx* ctx, uint32_t cluster_voxels, uint32_t* out_num_vertices, uint32_t* out_num_triangles);
int rr_download_simplified_mesh(rr_ctx* ctx, float* positions, float* normals, float* rgba, uint32_t* triangles, uint32_t* sources);
int rr_group_simplify_mesh(rr_group* g, uint32_t cluster_voxels, uint32_t* out_num_vertices, uint32_t* out_num_triangles);

/* ---- connected parts (no reference counterpart) -------------------------------------------------------------------------
 * What is in the volume: its separate objects, where each is, and which mesh triangles belong to which.
 *   Values   the grid of the surface extraction: voxel (x, y, z) has the value v rr_raymarch reads there (R32F; the low
 *            half of a half2 voxel, widened; F32_WEIGHT: the tsdf volume only).
 *   Inside   v > 0 and v finite (the raymarch's hit test, the mesh's inside); NaN and +-inf are never inside.
 *   Part     a maximal set of inside voxels connected through shared faces (6-neighbourhood): voxels that touch only along
 *            an edge or at a corner are in different parts, as the mesh's face rule separates them, so the surfaces of two
 *            parts never share a vertex.
 *   Order    a part's key is the smallest linear index z*X*Y + y*X + x of its voxels; parts are numbered 0..P-1 by
 *            ascending key. The order depends neither on scheduling, on the occupied-brick shortcut nor on the number of
 *            devices. Every voxel of the volume counts, whatever rr_set_slab says.
 *   Per part voxels uint32 [P] (the count); boxes int32 [P][6] = x0, x1, y0, y1, z0, z1, half-open voxel index ranges;
 *            centroids float32 [P][3] in metres: with S_k the exact integer sum of voxel index k over the part and n its
 *            count, c_k = (float)(bmin_k + ((S_k / n) + 0.5) / R_k * (bmax_k - bmin_k)), evaluated in binary64 in that
 *            order without fused multiply-adds, every operand widened from its binary32 or integer value.
 *   Labels   uint32 [Z][Y][X]: the part of every inside voxel, 0xFFFFFFFF everywhere else.
 *   Mesh     vertex_parts uint32 [V]: the part of the inside end of the vertex's edge (exactly one end is > 0 by the mesh's
 *            vertex rule); triangle_parts uint32 [T]: the part its three vertices share (every triangle's edges have their
 *            inside ends in one face-connected group of its cell's inside corners, so there is one).
 *
 * rr_label_parts   labels on the context's stream and synchronises once; returns the part count. RR_ERR_INVALID for a NULL
 *                  count pointer, before any integrate into the current volume (as rr_extract_mesh) and on a context
 *                  restricted by rr_set_slab (use rr_group_label_parts). Not a setting: the volume, brick tables, view
 *                  images (rr_fill_colors still fills the last view), mesh, cloud, query buffers, captured frame graphs and
 *                  rr_integrator_last stay as they are.
 * rr_download_parts  the last labelling. rr_download_mesh_parts  the parts of the last mesh; RR_ERR_INVALID unless the mesh
 *                  and the last labelling were taken from the same volume state (no integrate and no new volume between
 *                  them). rr_download_parts: RR_ERR_INVALID before any labelling of the current volume. For both, each
 *                  pointer may be NULL, host memory (pageable or pinned) or device memory of the context's GPU; they return
 *                  after one synchronisation.
 * rr_group_label_parts  the same for a group, bit for bit: member 0 receives the other members' slabs by peer copies (as
 *                  rr_group_extract_mesh) and labels; read with rr_download_parts(rr_group_member(g, 0), ...) and, after
 *                  rr_group_extract_mesh, rr_download_mesh_parts on member 0. */
int rr_label_parts(rr_ctx* ctx, uint32_t* out_num_parts);
int rr_download_parts(rr_ctx* ctx, uint32_t* voxels, int32_t* boxes, float* centroids, uint32_t* labels);
int rr_download_mesh_parts(rr_ctx* ctx, uint32_t* vertex_parts, uint32_t* triangle_parts);
int rr_group_label_parts(rr_group* g, uint32_t* out_num_parts);

/* ---- removing parts (no reference counterpart) --------------------------------------------------------------------------
 * Takes chosen parts out of the volume itself - the small floating blobs sensor noise leaves in front of the surface, or
 * everything but the objects a client wants to show - so that every output (views, colour fill, meshes, queries, distances,
 * parts and tracks) sees the cleaned volume through its own code path.
 *   Labelling  the context's last labelling (rr_label_parts, or the labelling inside rr_track_parts), which must be of the
 *            current volume state: no integrate, no new volume and no other removal since.
 *   Parts    part p of that labelling (P parts) is removed iff voxels[p] < min_voxels, or keep != NULL and keep[p] == 0.
 *            keep: uint8 [P], host memory (pageable or pinned) or device memory of the context's GPU; it must hold P entries.
 *            min_voxels == 0 with keep == NULL removes nothing.
 *   Voxels   every voxel labelled with a removed part becomes exactly the voxel the bricks-mode clear writes with the limit in
 *            effect now: R32F -limit; F32_WEIGHT tsdf -limit and weight 0; HALF2 half2(-limit, 0). Every other voxel of the
 *            volume and of the weight volume stays bit for bit as it was. The outside band (-limit < v <= 0) around a removed
 *            part stays: it produces no hit, no mesh vertex and no part.
 *
 * rr_remove_parts  rewrites on the context's stream and synchronises once; returns the number of removed parts and the exact
 *                  sum of their voxel counts. RR_ERR_INVALID for a NULL count pointer, no labelling of the current volume
 *                  state, and on a context restricted by rr_set_slab (use rr_group_remove_parts). When a part was removed
 *                  the volume epoch advances (a new volume state): a mesh, labelling or distance field taken before is of
 *                  the previous state under the rules above (rr_download_mesh_parts pairs only a mesh and a labelling of one
 *                  state, rr_sample_distance refuses until the next rr_distance_field, and a second rr_remove_parts needs a
 *                  new labelling); the labelling is not renumbered. Not a setting: brick tables, stage images, view images
 *                  (rr_fill_colors still fills the last view), cloud, query buffers, tracking state, captured frame graphs,
 *                  rr_integrator_last and rr_integrator_cleared stay as they are, and the next integrates clear and write
 *                  exactly what they would have (the incremental clear stays valid: a removed voxel was inside, so it lay in
 *                  a brick the last integrate evaluated).
 * rr_group_remove_parts  the same for a group with member 0's last labelling (rr_group_label_parts / rr_group_track_parts):
 *                  every member rewrites the rows its integrate writes (its slab and halo), so that every member's slab
 *                  and halo, and the group's views, queries and meshes, equal a single context's bit for bit. Member 0
 *                  writes the other members' volumes through peer memory: RR_ERR_UNSUPPORTED when its device cannot address
 *                  a member's memory. */
int rr_remove_parts(rr_ctx* ctx, uint32_t min_voxels, const uint8_t* keep, uint32_t* out_removed_parts,
                    uint32_t* out_removed_voxels);
int rr_group_remove_parts(rr_group* g, uint32_t min_voxels, const uint8_t* keep, uint32_t* out_removed_parts,
                          uint32_t* out_removed_voxels);

/* ---- part tracking (no reference counterpart) ---------------------------------------------------------------------------
 * Persistent identities for the connected parts from one frame set to the next: a part's number depends on what else is in
 * the volume, a track id follows the object by voxel overlap.
 *   State    a context holds optional tracking state: the tracked labelling (the labels and per-part track ids of the last
 *            rr_track_parts) and next_id, which starts at 0. A context that never tracks allocates nothing for it.
 *            rr_reset_part_tracks and a new volume allocation as far as extraction goes (a new resolution or voxel format
 *            in rr_configure) empty it and set next_id to 0; other settings (limit, brick size, rr_set_slab, bbox) leave it.
 *   Labels   the current volume is labelled exactly as rr_label_parts does: rr_download_parts and rr_download_mesh_parts
 *            then return, bit for bit, what they return after rr_label_parts, epoch rule included.
 *   Pairs    a current part p is tracked iff voxels[p] >= min_voxels; a previous part q is a candidate iff it received a
 *            track id in the previous call; O(q, p) counts the voxels labelled q in the tracked labelling and p now. The
 *            candidate pairs are those with q a candidate, p tracked and O(q, p) > 0.
 *   Matching greedy in the strict total order O descending, then q ascending, then p ascending: a pair is accepted iff
 *            neither its q nor its p is accepted already. An accepted p inherits q's track id, prev_parts[p] = q and
 *            overlaps[p] = O(q, p). Tracked parts left unmatched get new ids next_id, next_id + 1, ... in ascending part
 *            index, with prev_parts 0xFFFFFFFF and overlaps 0. Untracked parts get track id 0xFFFFFFFF, prev_parts
 *            0xFFFFFFFF, overlaps 0. Ids are never reused before a reset.
 *   Ended    ended[E]: the track ids of the candidate previous parts that were not accepted, by ascending previous part.
 *            The labelling and its ids then become the tracked labelling; the first call after a reset has no candidates
 *            (every tracked part is new, E = 0).
 *   Overlaps are exact counts and the order is total: no output depends on scheduling, the brick shortcut or the number of
 *   devices. Tracking the same volume twice keeps every id with overlaps == voxels and ends nothing. Matching is by overlap
 *   only: a caller that skips frame sets over which an object moves further than its own extent gets a new id for it.
 *
 * rr_track_parts   labels and tracks on the context's stream, with at most three synchronisations (the part count, the
 *                  pair-record count, the counts returned); returns the part count P and the ended count E.
 *                  RR_ERR_INVALID for min_voxels == 0, a NULL count pointer, before any integrate into the current volume
 *                  and on a context restricted by rr_set_slab (use rr_group_track_parts). RR_ERR_UNSUPPORTED when the call
 *                  would need track id 0xFFFFFFFF; the tracking state then stays as it was. Not a setting: the volume,
 *                  brick tables, view images (rr_fill_colors still fills the last view), mesh, simplified mesh, cloud,
 *                  query buffers, captured frame graphs and rr_integrator_last stay as they are. rr_label_parts keeps its
 *                  results and cost, and a call of it between two rr_track_parts does not change what the second compares
 *                  against.
 * rr_download_part_tracks  the last tracking: track_ids, prev_parts and overlaps uint32 [P], ended uint32 [E]. Each pointer may
 *                  be NULL, host memory (pageable or pinned) or device memory of the context's GPU; returns after one
 *                  synchronisation. Valid until the next rr_track_parts, reset or new volume, whatever rr_label_parts calls
 *                  come in between; RR_ERR_INVALID before any tracking of the current volume allocation (or after a reset).
 * rr_reset_part_tracks  empties the tracking state: the next rr_track_parts starts ids at 0 with no candidates.
 * rr_group_track_parts  the same for a group, bit for bit equal to a single context over the same sequence of frame sets:
 *                  member 0 receives the other members' slabs by peer copies (as rr_group_label_parts) and tracks there;
 *                  read with rr_download_part_tracks(rr_group_member(g, 0), ...), reset with rr_reset_part_tracks on
 *                  member 0. */
int rr_track_parts(rr_ctx* ctx, uint32_t min_voxels, uint32_t* out_num_parts, uint32_t* out_num_ended);
int rr_download_part_tracks(rr_ctx* ctx, uint32_t* track_ids, uint32_t* prev_parts, uint32_t* overlaps, uint32_t* ended);
int rr_reset_part_tracks(rr_ctx* ctx);
int rr_group_track_parts(rr_group* g, uint32_t min_voxels, uint32_t* out_num_parts, uint32_t* out_num_ended);

/* ---- distances (no reference counterpart) -------------------------------------------------------------------------------
 * How far a point is from the captured surface, and the nearest point on it: the volume itself only answers within +-limit
 * of the surface (every voxel farther out holds -limit in bricks mode).
 *   Grid     the grid and inside rule of the connected parts: v is the value rr_raymarch reads (R32F; the low half of a half2
 *            voxel, widened; F32_WEIGHT: the tsdf volume), a voxel is inside iff v > 0 and v is finite, and every voxel of
 *            the volume counts, whatever rr_set_slab says.
 *   Field    nearest uint32 [Z][Y][X]: for every voxel a = (x, y, z), the linear index z*X*Y + y*X + x of an inside voxel s
 *            minimising d^2(a, s) = dx^2 + dy^2 + dz^2 in voxel index units (exact integers); on ties the smallest linear
 *            index. An inside voxel is its own nearest voxel; with no inside voxel every entry is 0xFFFFFFFF. The rule is
 *            total: the field depends neither on scheduling, on the occupied-brick shortcut nor on the number of devices.
 *            Index units: the voxel spacing (bmax_k - bmin_k) / R_k may differ slightly between axes (R_k = ceil(size_k /
 *            voxel_size)), so in an anisotropic box the index-metric nearest voxel can differ from the metric one.
 *   Query    points [n][3] in RR_QUERY_WORLD or RR_QUERY_VOLUME, converted as rr_sample_points does (to_volume). For q in the
 *            closed unit cube the query voxel is a = (floor(q_x X), floor(q_y Y), floor(q_z Z)), each clamped to [0, R_k - 1]
 *            (the nearest-texel rule), and f = nearest[a]:
 *              nearest_voxels uint32 [n]   f;
 *              nearest_points float32 [n][3]  f's voxel centre in the input's space: volume ((float)f_k + 0.5f) / (float)R_k,
 *                                          world c_k = bmin_k + (((float)f_k + 0.5f) / (float)R_k) * (bmax_k - bmin_k);
 *              distances float32 [n]       metres, always: p = the point in world space (a volume-space input q becomes
 *                                          bmin + q * (bmax - bmin)), d = sqrtf((dx*dx + dy*dy) + dz*dz) with dx = p_x - c_x,
 *                                          ... (binary32, no fused multiply-add, sqrtf correctly rounded).
 *            d is the distance from p to the centre of the nearest inside voxel of p's voxel: within one voxel diagonal of
 *            p's distance to the nearest inside-voxel centre. No inside voxel: distance +inf, nearest point NaN, voxel
 *            0xFFFFFFFF. Outside the closed unit cube or non-finite input: distance NaN, nearest point NaN, voxel 0xFFFFFFFF
 *            (as rr_sample_points).
 *   Parts    the part of the nearest voxel is part_labels[nearest_voxels] when a labelling of the same volume state exists.
 *
 * rr_distance_field  computes the field of the current volume on the context's stream and synchronises once; returns the
 *                  number of inside voxels. RR_ERR_INVALID for a NULL count pointer, before any integrate into the current
 *                  volume (as rr_extract_mesh) and on a context restricted by rr_set_slab (use rr_group_distance_field);
 *                  RR_ERR_UNSUPPORTED for a volume with an axis of more than 2048 voxels. The field records the volume
 *                  state (epoch) it was computed from. Not a setting: the volume, brick tables, view images (rr_fill_colors
 *                  still fills the last view), mesh, simplified mesh, cloud, part labels and tracking state, query buffers,
 *                  captured frame graphs and rr_integrator_last stay as they are. A new volume allocation (a new resolution
 *                  or voxel format in rr_configure) releases the field's two volume-sized arrays.
 * rr_download_distance_field  the last field of the current volume allocation (also after later integrates); nearest may be
 *                  NULL, host memory (pageable or pinned) or device memory of the context's GPU; returns after one
 *                  synchronisation. RR_ERR_INVALID before any field of the current volume allocation.
 * rr_sample_distance  the query above against the last field, which must be of the current volume state: a query after an
 *                  integrate is refused until the next rr_distance_field, so it never answers about a previous frame set.
 *                  points and each output may be host (pageable or pinned) or device memory, outputs may be NULL; one
 *                  synchronisation. count 0 does nothing; RR_ERR_INVALID for a bad space, NULL points with count > 0, or no
 *                  field of the current volume state; RR_ERR_UNSUPPORTED for count >= 2^31.
 * rr_group_distance_field  the same for a group, bit for bit: member 0 receives the other members' slabs by peer copies (as
 *                  rr_group_label_parts) and computes the field there; read it with
 *                  rr_download_distance_field(rr_group_member(g, 0), ...).
 * rr_group_sample_distance  rr_sample_distance on member 0 against the group's field, whatever member 0's slab. */
int rr_distance_field(rr_ctx* ctx, uint32_t* out_num_inside);
int rr_download_distance_field(rr_ctx* ctx, uint32_t* nearest);
int rr_sample_distance(rr_ctx* ctx, int space, const float* points, uint32_t count, float* distances, float* nearest_points,
                       uint32_t* nearest_voxels);
int rr_group_distance_field(rr_group* g, uint32_t* out_num_inside);
int rr_group_sample_distance(rr_group* g, int space, const float* points, uint32_t count, float* distances,
                             float* nearest_points, uint32_t* nearest_voxels);

/* ---- point clouds (no reference counterpart: a reference user draws the points and reads pixels back) -------------------
 * The pre-processed, registered sensor points: every kept depth pixel of the sensors in sensor_mask, lifted to the world.
 * For sensor i (bit i of sensor_mask) and pixel (x, y) of its W x H depth image, id = i*W*H + y*W + x:
 *   sx = (float)((x + 0.5) * (double)(1.0f / W)), sy likewise with y and H (the vertex buffer rr_draw_points draws);
 *   d  = depth_b.x of the last rr_preprocess / rr_fuse_frame at the pixel (RR_STAGE_DEPTH_B);
 *   p  = trilinear cv_xyz_i at (sx, sy, d) in metres, t = trilinear cv_uv_i there, with the calibration volumes in effect.
 * The point is kept iff d > 0, bbox_min <= p <= bbox_max componentwise (the bbox in effect) and 0.01 <= t.x, t.y <= 0.99:
 * exactly the vertices rr_draw_points keeps before the view transform. A non-finite p or d is never kept. Per kept point:
 *   positions = p, float32 [n][3];  normals = the normal stage at the pixel (xyz, as RR_STAGE_NORMAL), float32 [n][3];
 *   colors = the bilinear RGB8 fetch of the current colour frame at t (the colour rr_draw_points shades with in shade mode 0),
 *   float32 [n][3] in [0, 1];  quality = the quality stage at the pixel, float32 [n];  pixels = id, uint32 [n].
 * Order: ascending id (sensor, row, column); it depends neither on scheduling nor on the number of devices.
 *
 * rr_extract_points  extracts on the context's stream and synchronises once; returns the count. sensor_mask == 0 gives 0
 *                   points. RR_ERR_INVALID for a mask bit at or above the sensor count, a NULL count pointer, a sensor of the
 *                   mask without rr_calib_upload, and a call before any rr_preprocess / rr_fuse_frame on this context. A
 *                   context restricted by rr_set_slab is fine (its stage images are complete). Not a setting: the volume,
 *                   stage images, brick tables, view images (rr_fill_colors still fills the last view), mesh and captured
 *                   frame graphs stay as they are.
 * rr_download_points  the last extraction; each pointer may be NULL, host memory (pageable or pinned) or device memory of the
 *                   context's GPU. Returns after one synchronisation. RR_ERR_INVALID if nothing was extracted yet.
 * rr_group_extract_points  the same on member 0 of a group (pre-processing is replicated, so no peer traffic), equal to a
 *                   single context bit for bit; read it with rr_download_points(rr_group_member(g, 0), ...). */
int rr_extract_points(rr_ctx* ctx, uint32_t sensor_mask, uint32_t* out_num_points);
int rr_download_points(rr_ctx* ctx, float* positions, float* normals, float* colors, float* quality, uint32_t* pixels);
int rr_group_extract_points(rr_group* g, uint32_t sensor_mask, uint32_t* out_num_points);

/* ---- queries (no reference counterpart: a reference user renders a view and reads pixels back) ------------------------
 * The fused volume evaluated at points and along rays the caller chooses: picking, collision tests, measurements.
 *   space      RR_QUERY_WORLD: coordinates in metres; a point becomes q = (p - bbox_min) / (bbox_max - bbox_min) (one IEEE
 *              division per component, no fused multiply-add), a direction normalize(d / (bbox_max - bbox_min)).
 *              RR_QUERY_VOLUME: volume texture coordinates, [0,1]^3 over the bbox (as rr_download_hit_positions); points
 *              are used as given, directions are normalised. normalize is the raymarch's (v * (1 / sqrt(dot(v, v)))).
 *   rr_sample_points  per point: value = the density rr_raymarch reads at q (trilinear; the low half of a half2 voxel);
 *              normal = normalize(g / (bbox_max - bbox_min)) with g the raymarch's gradient at q (step limit / 2), always
 *              in world space (the mesh vertex normal; NaN where it vanishes); rgba = blendColors at q (alpha 1 when
 *              quality-weighted, -1 for the fallback blend). Outside the closed unit cube, or for a non-finite input, value
 *              and normal are NaN and rgba is 0. Arrays: points float32 [n][3]; values [n], normals [n][3], rgba [n][4].
 *   rr_cast_rays  per ray: rr_raymarch's own march from origin q0 along the normalised direction - live only if the ray
 *              meets the unit cube ahead of q0; it starts at the cube entry (at q0 when q0 is inside), or runs over the
 *              occupied-brick hull when the raymarch would skip space; steps of limit / 2, the raymarch's hit refinement and
 *              empty-space fetch skipping, with the brick tables rr_raymarch would use now. positions = the refined hit in the
 *              input's space (world: bbox_min + q * (bbox_max - bbox_min), no fused multiply-add); normals and rgba as for
 *              points, at the hit; steps = the raymarch's sample count at the hit. Any finite non-zero direction is a ray:
 *              when dot(d, d) (after the division by the bbox size in world space) overflows binary32 or falls below 2^-100,
 *              d is first scaled by an exact power of two (2^-70; or 2^64, at most twice), so it casts as the same direction
 *              of ordinary length. A ray without a hit - also one with a zero or non-finite direction or origin, or an origin
 *              farther than 2^24 bbox sizes (|q0_k| > 2^24), whose march length binary32 cannot resolve - gets NaN positions
 *              and normals, rgba 0 and step 0xFFFFFFFF. Never shaded. Arrays: origins, directions float32 [n][3]; positions [n][3], normals [n][3], rgba [n][4], steps
 *              uint32 [n].
 * Every pointer may be host memory (pageable or pinned) or device memory of the context's GPU (for a group: of member 0's
 * GPU); each output may be NULL. The call runs on the context's stream and returns after one synchronisation. count == 0
 * does nothing and returns RR_OK. RR_ERR_INVALID for a bad space, NULL inputs, a call before anything was integrated into
 * the current volume (as rr_extract_mesh) and a context restricted by rr_set_slab (use the group form);
 * RR_ERR_UNSUPPORTED for count >= 2^31. A query is not a setting: the volume, brick tables, view images (rr_fill_colors
 * still fills the last view), mesh and captured frame graphs stay as they are.
 * rr_group_sample_points / rr_group_cast_rays  the same for a group, equal to a single context bit for bit without moving the
 *              volume: every member marches every ray over the samples it owns and evaluates its own first hit, and one
 *              kernel on member 0 keeps each ray's smallest step (lowest member on ties); a point is evaluated by the member
 *              owning its nearest z slice. Member 0 reads the other members' results through peer memory: RR_ERR_UNSUPPORTED
 *              when it cannot address a member's device. */
#define RR_QUERY_WORLD 0
#define RR_QUERY_VOLUME 1
int rr_sample_points(rr_ctx* ctx, int space, const float* points, uint32_t count, float* values, float* normals, float* rgba);
int rr_cast_rays(rr_ctx* ctx, int space, const float* origins, const float* directions, uint32_t count,
                 float* positions, float* normals, float* rgba, uint32_t* steps);
int rr_group_sample_points(rr_group* g, int space, const float* points, uint32_t count, float* values, float* normals, float* rgba);
int rr_group_cast_rays(rr_group* g, int space, const float* origins, const float* directions, uint32_t count,
                       float* positions, float* normals, float* rgba, uint32_t* steps);

/* ---- read-back (tests, debug views) ------------------------------------------------------------------------ */
int rr_download_tsdf(rr_ctx* ctx, float* out);
int rr_download_weight(rr_ctx* ctx, float* out);
int rr_download_stage(rr_ctx* ctx, int stage, float* out);
/* Brick counters uint32 [num_bricks] and the ordered occupied list; *num_occupied receives its length. */
int rr_download_bricks(rr_ctx* ctx, uint32_t* counters, uint32_t* occupied, uint32_t* num_occupied);
/* Last raymarch: sample-count image float32 [h][w] (tex_num_samples, tsdf_raymarch.fs:403-406). */
int rr_download_num_samples(rr_ctx* ctx, float* out);
/* Last raymarch: surface point per pixel in volume (texture) space, float32 [h][w][4] = x, y, z, hit flag
 * (the refined sample_pos of tsdf_raymarch.fs:100; world = bbox_min + xyz * bbox_size). For tests. */
int rr_download_hit_positions(rr_ctx* ctx, float* out);

/* ---- instrumentation ---------------------------------------------------------------------------------------- */
/* TimerDatabase stage names (framework/rendering/timer_database.cpp:26-41; NetKinectArray.cpp:211-216,
 * recon_integration.cpp:146-148, reconstruction.cpp:25-26): "morph", "bilateral", "boundary", "normal", "quality",
 * "1preprocess", "2integrate", "3recon", "brickdraw", "draw" — CUDA events on the context's stream instead of GL
 * timestamp queries. level 0 = off, 1 = the numbered top-level stages only, 2 = every pass.
 * rr_get_stage_ms: last recorded duration. rr_get_stage_stats: sum and count of all intervals recorded since the
 * previous call (TimerDatabase's running mean), then resets them. Both synchronise on the events they read. */
int rr_set_timing(rr_ctx* ctx, int level);
int rr_get_stage_ms(rr_ctx* ctx, const char* name, float* ms);
int rr_get_stage_stats(rr_ctx* ctx, const char* name, float* total_ms, uint32_t* count);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
uint64_t rr_launch_count(const rr_ctx* ctx);
/* Launch-shape knob of the integrator, process-wide (no reference counterpart; the reference's draw-call structure is
 * fixed). Names: "fused", "zchunk", "fill_rows", "fill_warps", "ctas", "threads", "chunk", "brick_grid",
 * "ldg256", "graph", "staged", "stage_zchunk", "stage_ychunk", "stage_tile", "stage_cwarps", "stage_fill_rows", "stage_bulk_fill", "stage_fill_depth",
 * "stage_tail_cap", "stage_ctas", "stage_fill_lsu", "stage_debug", "fuse_nq" (1: pre_normal and pre_quality as one launch,
 * k_normal_quality; 0: two kernels), "trigrid_pool" (rr_draw_trigrid: initial fragment-pool
 * capacity in fragments per 16 view pixels; the pool grows when a view needs more).
 * Results never depend on these. Returns RR_ERR_INVALID for an unknown name. */
int rr_set_tunable(const char* name, int value);
/* Which integrator the bricks mode of this context runs and with what geometry (no reference counterpart; diagnostics for
 * bench.py and the tests). Waits for the stream. out[16]:
 *  [0] 1 = the TMA-staged kernel is selected (0: the direct kernels), [1] tile edge (pixels), [2..4] staged inverse-volume
 *  box (coarse texels), [5] y-chunk, [6] z-chunk (voxels per work item), [7] y-chunks per brick, [8] z-chunks per brick,
 *  [9] (item, sensor) pairs of the brick grid whose footprint exceeds the tile (read from global memory when occupied and
 *  not settled by a verdict), [10] shared memory per CTA (bytes), [11] consumer warps, [12] clear warps, [13] device-side
 *  consistency flags (0 = healthy: bit 0 box overflow, bit 1 barrier time-out), [14] operand slots in the ring, [15] bytes per slot. */
int rr_integrator_info(rr_ctx* ctx, uint32_t* out);
/* Which integration kernel the last rr_integrate (or the integrate step of rr_fuse_frame) launched. Host-side record, no
 * device access: a replayed frame graph reports what was captured. out[8]:
 *  [0] path: 0 nothing launched (empty slab, no brick extents), 1 TMA-staged kernel, 2 fused clear + integrate kernel,
 *      3 k_fill + k_integrate_bricks, 4 dense kernel; [1] sensors; [2] voxel format (rr_voxel_format);
 *  [3] CTA threads, or consumer warps of the staged kernel;
 *  [4] repairs: bit 0 the staged kernel declined because its item lists were not built for the current tables, limit and
 *      stage images (a direct kernel ran instead), bit 1 the gather texels were packed by this call because the last
 *      rr_preprocess had left them to the staged kernel;
 *  [5] clear: 0 none (dense mode, or nothing launched), 1 the whole slab outside the occupied bricks, 2 incremental: only
 *      the bricks that left the occupied set since the last integrate (the staged kernel, when the volume outside the
 *      bricks that integrate evaluated is known to hold the cleared value); [6..7] 0. */
int rr_integrator_last(const rr_ctx* ctx, uint32_t* out);
/* Bricks the incremental clear of the last integrate reset to the cleared value (evaluated by the integrate before it, not
 * occupied now); 0 when the last integrate did not clear incrementally. The count is kept by the device past later
 * rr_bricks_update calls, until the next integrate. Waits for the stream. out[1]. */
int rr_integrator_cleared(rr_ctx* ctx, uint32_t* out);
/* Cycle counters of the staged integrator's warp roles, accumulated while the tunable "stage_debug" has bit 7 set and reset
 * by this call (diagnostics, no reference counterpart). out[16], SM clock cycles summed over warps / producer threads:
 *  [0] consumer warps waiting for a staged item, [1] evaluating one, [2] items a consumer warp had no columns of,
 *  [4] producers gathering item metadata, [5] waiting for a free stage, [6] issuing + waiting for the copies,
 *  [7] staged items, [8] direct items, [9] clear warps in the clear, [10] other warps helping with the clear,
 *  [11] longest CTA (cycles), [12] sum over warps of their lifetime, [3] sensors evaluated voxel by voxel summed over items,
 *  [13] largest tile edge a staged (item, evaluated sensor) needed, [14] / [15] items needing at most 30 / 36 pixels. */
int rr_integrator_profile(rr_ctx* ctx, uint64_t* out);
/* Library/ABI version. */
int rr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RGBD_RECON_B200_H */
