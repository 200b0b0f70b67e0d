/* ORACLE (test infrastructure, NOT product code): C entry points of the scalar CPU restatement of
 * steppobeck/rgbd-recon's volumetric-fusion path. Loaded with ctypes by tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs ONLY. The reference ships no tests; the
 * restatement is pinned against reference code compiled into oracle/_ref: C++ sources (libref_harness.so, see ro_math.h) and
 * the pre-processing / integration / raymarch / colour-fill SHADERS run on the CPU (libref_glsl.so, oracle/glsl_host/). The
 * space-skipping hull of ro_raymarch.cpp is checked through the shader's skipSpace branch on depth peels produced by the
 * reference's bricks.vs/gs/fs and a rasteriser (glsl_harness.cpp::rg_depth_peels). */
#ifndef RR_ORACLE_H
#define RR_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

void ro_set_threads(int n);
int ro_get_max_threads(void);

/* scalar known-answer hooks for the math pins */
float ro_kat_log2(float x);
float ro_kat_exp2(float x);
float ro_kat_pow(float x, float y);
void ro_kat_tex3d(const float* vol, int C, int X, int Y, int Z, float s, float t, float r, float* out);
float ro_kat_tex2d(const float* img, int W, int H, float s, float t, int nearest);
void ro_kat_rgb_to_lab(const float* rgb, float* lab);

void ro_pre_morph(const float* depth_in, int W, int H, float* depth_out);
void ro_pre_depth(const float* depth_in, int W, int H, const float* cv_xyz, const float* cv_uv, int CX, int CY, int CZ,
                  const uint8_t* color, int CW, int CH, const float* bbox_min, const float* bbox_max,
                  float cv_min_ds, float cv_max_ds, int filter_textures, int compress, float scale, float near_,
                  float scaled_near, float* out_depth, float* out_lab);
void ro_pre_boundary(const float* depth_rg, const float* lab, int W, int H, int refine, float* out_depth_b, float* out_sil);
void ro_pre_normal(const float* depth_b, int W, int H, const float* cv_xyz, int CX, int CY, int CZ,
                   const float* bbox_min, float brick_size, const uint32_t* brick_res, uint32_t num_bricks,
                   uint32_t* bricks, float* out_normal);
void ro_pre_quality(const float* depth_b, const float* normals, int W, int H, const float* cv_xyz, int CX, int CY, int CZ,
                    const float* camera_pos, float* out_quality);

void ro_volume_res(const float* bbox_min, const float* bbox_max, float voxel_size, uint32_t* res_out);
float ro_adjust_brick_size(float voxel_size, float size);
uint32_t ro_divide_box(const float* bbox_min, const float* bbox_max, float brick_size, const uint32_t* res_volume,
                       uint32_t* res_bricks_out, int32_t* ranges);
uint32_t ro_divide_box_args(const float* bbox_min, const float* bbox_max, float brick_size, const uint32_t* res_volume,
                            float* args, int32_t* raw_ranges);
uint32_t ro_occupied_bricks(const uint32_t* counters, uint32_t num_bricks, uint32_t min_voxels, uint32_t* occupied_out);
void ro_integrate(int N, const float* inv, const int32_t* inv_res, const float* sil, const float* depth_b,
                  const float* quality, int W, int H, float limit, const uint32_t* res, int use_bricks,
                  const int32_t* brick_ranges, const uint32_t* occupied, uint32_t num_occupied, float* tsdf, float* weight);

void ro_frustum(const float* cv_xyz, int X, int Y, int Z, float* planes_out, float* campos_out);
int ro_frustum_inside(const float* planes, const float* p);
void ro_calib_invert(const float* cv_xyz, int X, int Y, int Z, const float* bbox_min, const float* bbox_max,
                     const uint32_t* out_res, float* out, uint32_t* neigh_out, int brute);

void ro_raymarch_uniforms(const float* mv, const float* proj, const float* bmin, const float* bmax, int vw, int vh, float* out);
void ro_raymarch_rays(const float* modelview, const float* projection, const float* bbox_min, const float* bbox_max, int vw, int vh,
                      float limit, float* out_points, uint8_t* out_covered);
void ro_raymarch(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                 const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                 const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                 const float* modelview, const float* projection, int vw, int vh, int shade_mode, int skip_space,
                 const uint32_t* occupied, uint32_t n_occ, const uint32_t* brick_res, float brick_size,
                 float* out_rgba, float* out_depth, float* out_samples, float* out_pos);


/* The point-drawing reconstructions (SURVEY.md §8f-4): ReconPoints::draw and ReconCalibs::draw, see ro_points.cpp. */
void ro_draw_points(int N, int W, int H, const float* depth_b, const float* normal, const uint8_t* color, int CW, int CH,
                    const float* cv_xyz, const float* cv_uv, const int32_t* cv_res, const float* bmin, const float* bmax,
                    const float* mv, const float* proj, int vw, int vh, int shade_mode, float* out_rgba, float* out_depth);
void ro_draw_calibs(const float* tsdf, const uint32_t* res, const int32_t* inv_res, float limit, const float* bmin, const float* bmax,
                    const float* mv, const float* proj, int vw, int vh, float* out_rgba, float* out_depth);

/* ReconTrigrid::draw (SURVEY.md §8f-4), see ro_trigrid.cpp. out_accum / out_depth1 may be null. */
void ro_draw_trigrid(int N, int W, int H, const float* depth_b, const float* quality, const uint8_t* color, int CW, int CH,
                     const float* cv_xyz, const float* cv_uv, const int32_t* cv_res, const float* bmin, const float* bmax,
                     const float* mv, const float* proj, int vw, int vh, int shade_mode, float min_length, float epsilon,
                     float* out_rgba, float* out_depth, float* out_accum, float* out_depth1);

/* Compressed ingest (SURVEY.md §8f-2): DXT1 colour blocks -> uint8 [H][W][3]; 8-bit depth -> byte/255. */
void ro_decode_dxt1(const uint8_t* blocks, int W, int H, uint8_t* out_rgb);
void ro_decode_dxt5(const uint8_t* blocks, int W, int H, uint8_t* out_rgb);   /* 16-byte blocks: alpha (skipped) + colour */
void ro_depth8_to_float(const uint8_t* in, size_t n, float* out);

/* Colour hole filling after the raymarch (ReconIntegration::fillColors + ViewLod + framebuffer_transfer / tsdf_inpaint /
 * tsdf_colorfill): rgba [H][W][4] and depth [H][W] in, out_rgba [H][W][4]; atlas_* optional ([H][1.5W][4] / [H][1.5W]). */
int ro_fill_num_lods(int W, int H);
void ro_fill_colors(const float* rgba, const float* depth, int W, int H, float* out_rgba, float* atlas_rgba, float* atlas_depth);

/* Surface extraction (rr_extract_mesh), see ro_mesh.cpp.
 * ro_mesh_case_table: ntri int32[256], tri int32[256][30] (cube edges, -1 past the case's triangles); returns the most
 * triangles any case needs, -1 if the rule is inconsistent.
 * ro_extract_mesh: counts[2] = vertices, triangles; positions [V][3], normals [V][3], rgba [V][4], triangles uint32 [T][3],
 * each may be null (a first call with all null gives the counts). tsdf float32 [Z][Y][X] as rr_download_tsdf returns it;
 * inv, cv_uv, color, depth_b and quality may be null when normals and rgba are. */
int ro_mesh_case_table(int32_t* ntri, int32_t* tri);
void ro_extract_mesh(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                     const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                     const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                     uint64_t* counts, float* positions, float* normals, float* rgba, uint32_t* triangles);

/* Volume queries (rr_sample_points / rr_cast_rays), see ro_query.cpp. tsdf float32 [Z][Y][X] as rr_download_tsdf returns
 * it; N may be 0 (inv, cv_uv, color, depth_b and quality null) when the colours are not wanted. space: 0 world (metres),
 * 1 volume texture coordinates.
 * ro_cast_rays: skip_space selects the march over the occupied-brick hull (occupied: the ordered list of
 * rr_download_bricks, brick_res / brick_size as rr_get_brick_info). Outputs as the library's: values [n] or positions
 * [n][3], normals [n][3], rgba [n][4], steps uint32 [n]. */
void ro_sample_points(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                      const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                      const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                      int space, const float* points, uint32_t count, float* values, float* normals, float* rgba);
void ro_cast_rays(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                  const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                  const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                  int skip_space, const uint32_t* occupied, uint32_t n_occ, const uint32_t* brick_res, float brick_size,
                  int space, const float* origins, const float* directions, uint32_t count,
                  float* positions, float* normals, float* rgba, uint32_t* steps);

/* Point-cloud export (rr_extract_points), see ro_cloud.cpp. depth_b float32 [N][H][W][2], normal float32 [N][H][W][3],
 * quality float32 [N][H][W], colour uint8 [N][CH][CW][3], cv_xyz float32 [N][Z][Y][X][3], cv_uv float32 [N][Z][Y][X][2]
 * (cv_res = X, Y, Z, one resolution for all sensors). Outputs hold up to N*W*H points: positions [n][3], normals [n][3],
 * colours [n][3], quality [n], pixel ids uint32 [n]; *out_n receives n. */
void ro_extract_points(int N, int W, int H, const float* depth_b, const float* normal, const float* quality, const uint8_t* color,
                       int CW, int CH, const float* cv_xyz, const float* cv_uv, const int32_t* cv_res, const float* bmin,
                       const float* bmax, uint32_t sensor_mask, uint32_t* out_n, float* positions, float* normals, float* colors,
                       float* quality_out, uint32_t* pixels);

#ifdef __cplusplus
}
#endif
#endif
