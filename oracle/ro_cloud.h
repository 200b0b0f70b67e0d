/* ORACLE (test infrastructure, NOT product code): C entry point of the scalar restatement of the point-cloud export
 * (rr_extract_points), see ro_cloud.cpp. Built as librr_oracle_cloud.so by cloud.mk, loaded with ctypes by oracle_cloud.py.
 * depth_b float32 [N][H][W][2], normal float32 [N][H][W][3], quality float32 [N][H][W], colour uint8 [N][CH][CW][3],
 * cv_xyz float32 [N][Z][Y][X][3], cv_uv float32 [N][Z][Y][X][2] (cv_res = X, Y, Z, one resolution for all sensors).
 * Outputs hold up to N*W*H points: positions [n][3], normals [n][3], colours [n][3], quality [n], pixel ids uint32 [n];
 * *out_n receives n. */
#ifndef RO_CLOUD_H
#define RO_CLOUD_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

void ro_extract_points(int N, int W, int H, const float* depth_b, const float* normal, const float* quality, const uint8_t* color,
                       int CW, int CH, const float* cv_xyz, const float* cv_uv, const int32_t* cv_res, const float* bmin,
                       const float* bmax, uint32_t sensor_mask, uint32_t* out_n, float* positions, float* normals, float* colors,
                       float* quality_out, uint32_t* pixels);

#ifdef __cplusplus
}
#endif
#endif
