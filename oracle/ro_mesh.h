/* ORACLE (test infrastructure, NOT product code): C entry points of the scalar restatement of the surface extraction
 * (rr_extract_mesh), see ro_mesh.cpp. Built as librr_oracle_mesh.so by mesh.mk, loaded with ctypes by oracle_mesh.py.
 * ro_mesh_case_table: ntri int32[256], tri int32[256][30] (cube edges, -1 past the case's triangles); returns the most
 * triangles any case needs, -1 if the rule is inconsistent.
 * ro_extract_mesh: counts[2] = vertices, triangles; positions [V][3], normals [V][3], rgba [V][4], triangles uint32 [T][3],
 * each may be null (a first call with all null gives the counts). tsdf float32 [Z][Y][X] as rr_download_tsdf returns it;
 * inv, cv_uv, color, depth_b and quality may be null when normals and rgba are. */
#ifndef RO_MESH_H
#define RO_MESH_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int ro_mesh_case_table(int32_t* ntri, int32_t* tri);
void ro_extract_mesh(const float* tsdf, const uint32_t* res, float limit, int N, const float* inv, const int32_t* inv_res,
                     const float* cv_uv, const int32_t* cv_res, const uint8_t* color, int CW, int CH,
                     const float* depth_b, const float* quality, int W, int H, const float* bbox_min, const float* bbox_max,
                     uint64_t* counts, float* positions, float* normals, float* rgba, uint32_t* triangles);

#ifdef __cplusplus
}
#endif
#endif
