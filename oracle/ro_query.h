/* ORACLE (test infrastructure, NOT product code): C entry points of the scalar restatement of the volume queries
 * (rr_sample_points / rr_cast_rays), see ro_query.cpp. Built as librr_oracle_query.so by query.mk, loaded with ctypes by
 * oracle_query.py. tsdf float32 [Z][Y][X] as rr_download_tsdf returns it; N may be 0 (inv, cv_uv, color, depth_b and
 * quality null) when the colours are not wanted. space: 0 world (metres), 1 volume texture coordinates.
 * ro_cast_rays: skip_space selects the march over the occupied-brick hull (occupied: the ordered list of
 * rr_download_bricks, brick_res / brick_size as rr_get_brick_info). Outputs as the library's: values [n] or positions
 * [n][3], normals [n][3], rgba [n][4], steps uint32 [n]. */
#ifndef RO_QUERY_H
#define RO_QUERY_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

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

#ifdef __cplusplus
}
#endif
#endif
