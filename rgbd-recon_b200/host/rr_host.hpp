// GL-free C++ look-alikes of the reference classes on the volumetric-fusion path, implemented over the C ABI of
// librr_b200.so (include/rgbd_recon_b200.h). Same class names, method names, argument meaning and call order as the
// reference, so source/kinect_client.cpp:240-279,572-617 and source/calib_inverter.cpp:12-74 port by deleting their GL /
// GLFW lines (INTEGRATION.md). Differences are confined to what had to change without a GL context:
//   * kinect::gpu::Context replaces the GLFW window + GL context as the process-wide "current device" (GL state was the
//     reference's implicit data bus; here it is one rr_ctx);
//   * ReconIntegration::draw() reads its matrices from setViewMatrices() instead of glGetFloatv, and leaves its image in
//     host buffers (colorImage()/depthImage()) instead of the default framebuffer;
//   * NetKinectArray is fed by pushFrame() / a .stream file reader thread instead of a ZeroMQ socket (SURVEY.md §8f-3).
// Errors: the C ABI's status codes are rethrown as std::runtime_error with rr_last_error() text; file problems throw
// std::runtime_error where the reference asserted or called exit(1).
#ifndef RR_HOST_HPP
#define RR_HOST_HPP

#include <array>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/rgbd_recon_b200.h"
#include "mini_math.hpp"

#define RR_HOST_MAX_SENSORS 8

namespace kinect {

// ---- framework/DataTypes.h:12-34 ---------------------------------------------------------------------------------
struct xyz { float x, y, z; };
struct uv { float u, v; };

// ---- framework/calibration/calibration_volume.hpp:13-84 ------------------------------------------------------------
// File layout: uint32 res.x, res.y, res.z; float depth_min, depth_max; T data[res.x*res.y*res.z], index z*X*Y + y*X + x.
template <typename T>
class CalibrationVolume {
 public:
  explicit CalibrationVolume(std::string const& filename) { read(filename); }
  CalibrationVolume(glm::uvec3 const& res, glm::fvec2 const& depth, std::vector<T> const& vol)
      : m_resolution(res), m_depth_limits(depth), m_volume(vol) {}
  void write(std::string const& filename) const {
    FILE* f = std::fopen(filename.c_str(), "wb");
    if (!f) throw std::runtime_error("cannot write " + filename);
    const unsigned r[3] = {m_resolution.x, m_resolution.y, m_resolution.z};
    const float d[2] = {m_depth_limits.x, m_depth_limits.y};
    bool ok = std::fwrite(r, sizeof(unsigned), 3, f) == 3 && std::fwrite(d, sizeof(float), 2, f) == 2 &&
              std::fwrite(m_volume.data(), sizeof(T), m_volume.size(), f) == m_volume.size();
    std::fclose(f);
    if (!ok) throw std::runtime_error("short write to " + filename);
  }
  glm::uvec3 const& res() const { return m_resolution; }
  glm::fvec2 const& depthLimits() const { return m_depth_limits; }
  std::size_t numVoxels() const { return (std::size_t)m_resolution.x * m_resolution.y * m_resolution.z; }
  std::vector<T> const& volume() const { return m_volume; }
  T const& operator()(unsigned x, unsigned y, unsigned z) const { return m_volume[(std::size_t)z * m_resolution.x * m_resolution.y + (std::size_t)y * m_resolution.x + x]; }
 private:
  void read(std::string const& filename) {
    FILE* f = std::fopen(filename.c_str(), "rb");
    if (!f) throw std::runtime_error("cannot open " + filename);
    unsigned r[3]; float d[2];
    bool ok = std::fread(r, sizeof(unsigned), 3, f) == 3 && std::fread(d, sizeof(float), 2, f) == 2;
    if (ok) {
      m_resolution = glm::uvec3(r[0], r[1], r[2]);
      m_depth_limits = glm::fvec2(d[0], d[1]);
      m_volume.resize(numVoxels());
      ok = std::fread(m_volume.data(), sizeof(T), m_volume.size(), f) == m_volume.size();
    }
    std::fclose(f);
    if (!ok) throw std::runtime_error("short read from " + filename);
  }
  glm::uvec3 m_resolution;
  glm::fvec2 m_depth_limits;
  std::vector<T> m_volume;
};

// ---- framework/calibration/calibration_files.hpp -------------------------------------------------------------------
// ---- framework/calibration/KinectCalibrationFile.{h,cpp}: the stream-format fields of a sensor's .yml -------------------
// Only what the fusion path consumes is kept: rgb_size / depth_size / near_far / compress_rgb / compress_depth / min_length
// (KinectCalibrationFile.cpp:306-352). The tokenizer is the reference's: whitespace tokens, "name:" then everything up
// to "[", then "<a>," "<b>" (kommaStringToFloat drops the last character, getNextFloat is atof; :584-627). Intrinsics and
// extrinsics are not parsed: on this path the sensor geometry comes from the .cv_xyz/.cv_uv volumes.
class KinectCalibrationFile {
 public:
  explicit KinectCalibrationFile(std::string const& filePath) : _filePath(filePath) {}
  bool parse();                                 // false if the file cannot be opened; unknown tokens are skipped (:354-356)
  float getNear() const { return _near; }
  float getFar() const { return _far; }
  unsigned getWidth() const { return _width; }
  unsigned getHeight() const { return _height; }
  unsigned getWidthC() const { return _widthc; }
  unsigned getHeightC() const { return _heightc; }
  unsigned isCompressedRGB() const { return _iscompressedrgb; }
  bool isCompressedDepth() const { return _iscompresseddepth; }
  float min_length = 0.0125f;
 private:
  std::string _filePath;
  float _near = 0.3f, _far = 7.0f;              // defaults of the reference's constructor (:88-95)
  unsigned _width = 0, _height = 0, _widthc = 0, _heightc = 0;
  unsigned _iscompressedrgb = 1;
  bool _iscompresseddepth = false;
};

class CalibrationFiles {
 public:
  // the reference's constructor (calibration_files.cpp:7-34): sizes and stream formats come from the first sensor's .yml
  explicit CalibrationFiles(std::vector<std::string> const& calib_filenames);
  // explicit sizes, for callers without .yml metadata (synthetic scenes)
  CalibrationFiles(std::vector<std::string> const& calib_filenames, unsigned width, unsigned height, unsigned widthc, unsigned heightc,
                   unsigned compressed_rgb = 0, bool compressed_depth = false)
      : m_width(width), m_widthc(widthc), m_height(height), m_heightc(heightc), m_compressed_rgb(compressed_rgb),
        m_compressed_d(compressed_depth), m_filenames(calib_filenames) {}
  unsigned getWidth() const { return m_width; }
  unsigned getWidthC() const { return m_widthc; }
  unsigned getHeight() const { return m_height; }
  unsigned getHeightC() const { return m_heightc; }
  unsigned num() const { return (unsigned)m_filenames.size(); }
  unsigned isCompressedRGB() const { return m_compressed_rgb; }
  bool isCompressedDepth() const { return m_compressed_d; }
  float minLength() const { return m_min_length; }
  // KinectCalibrationFile::getNear / getFar (the range of the 8-bit depth stream), per sensor as in the reference
  // (getCalibs()[i].getNear()); setDepthRange sets one range for every sensor (synthetic scenes)
  void setDepthRange(float near_, float far_) { m_near = near_; m_far = far_; m_near_far.clear(); }
  float getNear() const { return m_near; }
  float getFar() const { return m_far; }
  float getNear(unsigned i) const { return i < m_near_far.size() ? m_near_far[i].first : m_near; }
  float getFar(unsigned i) const { return i < m_near_far.size() ? m_near_far[i].second : m_far; }
  std::vector<std::string> const& getFileNames() const { return m_filenames; }
 private:
  unsigned m_width, m_widthc, m_height, m_heightc, m_compressed_rgb;
  bool m_compressed_d;
  float m_near = 0.5f, m_far = 4.5f, m_min_length = 0.0125f;
  std::vector<std::pair<float, float>> m_near_far;       // (near, far) of every sensor's .yml; empty: m_near / m_far for all
  std::vector<std::string> m_filenames;
};

// ---- the "current device": stands where the GLFW window / GL context stood -----------------------------------------
namespace gpu {
class Context {
 public:
  Context(int device, CalibrationFiles const& cfs);
  // several devices: the TSDF volume is split into z-slabs, one per device (rr_group, include/rgbd_recon_b200.h); frame sets
  // enter on devices[0] and reach the others by peer copies, the view is composited on devices[0]
  Context(std::vector<int> const& devices, CalibrationFiles const& cfs);
  ~Context();
  Context(Context const&) = delete;
  Context& operator=(Context const&) = delete;
  rr_ctx* handle() const { return m_ctx; }   // member 0: queries, read-backs, timers
  rr_group* group() const { return m_group; }
  unsigned numDevices() const { return (unsigned)rr_group_size(m_group); }
  // equal-cost slabs from the occupied bricks of the last fused frame set (rr_group_balance_slabs)
  void balanceSlabs() const { checkGroup(rr_group_balance_slabs(m_group, 0.0f), "rr_group_balance_slabs"); }
  static Context& current();                 // throws if none was created
  void check(int status, char const* what) const;        // rethrow a C-ABI status of member 0
  void checkGroup(int status, char const* what) const;   // ... of a group call
 private:
  rr_group* m_group;
  rr_ctx* m_ctx;
};
}  // namespace gpu

// ---- framework/calibration/frustum.hpp ------------------------------------------------------------------------------
class Frustum {
 public:
  Frustum() {}
  Frustum(std::array<glm::fvec4, 6> const& planes, glm::fvec3 const& cam) : m_planes(planes), m_cam(cam) {}
  glm::fvec3 getCameraPos() const { return m_cam; }
  bool inside(glm::fvec3 const& p) const {
    for (auto const& pl : m_planes)
      if ((pl.x * p.x + pl.y * p.y) + (pl.z * p.z + pl.w * 1.0f) < 0.0f) return false;   // glm::dot(vec4, vec4) order
    return true;
  }
 private:
  std::array<glm::fvec4, 6> m_planes;
  glm::fvec3 m_cam;
};

// ---- framework/calibration/CalibVolumes.hpp:21-81 ---------------------------------------------------------------------
class CalibVolumes {
 public:
  CalibVolumes(std::vector<std::string> const& calib_volume_files, gloost::BoundingBox const& bbox);
  glm::uvec3 getVolumeRes() const;                       // resolution of the inverse volumes
  glm::fvec2 getDepthLimits(unsigned i) const;
  void loadInverseCalibs(std::string const& path);       // <path><basename>.cv_xyz_inv, CalibVolumes.cpp:64-80
  Frustum const& getFrustum(unsigned i) const { return m_frustums.at(i); }
  std::vector<glm::fvec3> getCameraPositions() const;
  gloost::BoundingBox const& getBBox() const { return m_bbox; }
  unsigned num() const { return (unsigned)m_cv_xyz_filenames.size(); }
  std::vector<std::string> const& xyzFileNames() const { return m_cv_xyz_filenames; }
 private:
  void addVolume(unsigned i, std::string const& filename_xyz, std::string const& filename_uv);
  std::vector<std::string> m_cv_xyz_filenames, m_cv_uv_filenames;
  std::vector<glm::uvec3> m_res;
  std::vector<glm::fvec2> m_limits;
  std::vector<Frustum> m_frustums;
  glm::uvec3 m_res_inv;
  gloost::BoundingBox m_bbox;
};

// ---- framework/calibration/calibration_inverter.hpp:20-44 ------------------------------------------------------------
class CalibrationInverter {
 public:
  CalibrationInverter(std::vector<std::string> const& calib_volume_files, gloost::BoundingBox const& bbox);
  void calculateInverseVolumes(glm::uvec3 const& volume_res);
  void writeInverseVolumes(std::string const& path) const;
  std::vector<CalibrationVolume<glm::fvec4>> const& inverseVolumes() const { return m_data_volumes_xyz_inv; }
  double lastGpuMilliseconds() const { return m_ms; }
 private:
  std::vector<std::string> m_cv_xyz_filenames;
  std::vector<CalibrationVolume<glm::fvec4>> m_data_volumes_xyz_inv;
  gloost::BoundingBox m_bbox;
  double m_ms = 0.0;
};

// ---- framework/NetKinectArray.h:35-128 -------------------------------------------------------------------------------
class NetKinectArray {
 public:
  // serverport/slaveport are kept for signature compatibility; with readfromfile the "serverport" is a list of
  // .stream files separated by ';' (frame = colour bytes then depth bytes per sensor, NetKinectArray.cpp:724-764)
  NetKinectArray(std::string const& serverport, std::string const& slaveport, CalibrationFiles const* calibs, CalibVolumes const* vols,
                 bool readfromfile = false);
  ~NetKinectArray();
  bool update();                                  // NetKinectArray.cpp:226-238: upload the newest complete frame set, if any
  void processTextures();                         // :311-428
  void filterTextures(bool filter);               // each of these re-runs processTextures(), :470-482
  void useProcessedDepths(bool filter);
  void refineBoundary(bool filter);
  glm::uvec2 getDepthResolution() const { return m_resolution_depth; }
  glm::uvec2 getColorResolution() const { return m_resolution_color; }
  // producer side (what readLoop did with the mapped PBOs, :484-544): copies one frame set into the back staging buffer
  void pushFrame(void const* color, void const* depth);
  // one message of the server's stream as readLoop receives it from the ZMQ SUB socket (NetKinectArray.cpp:511-538):
  // N x [colour bytes | depth bytes], sensor-major; the first 8 bytes double as the frame time (:525). Throws on a size
  // mismatch. The transport itself (libzmq) stays outside this library: a recv loop calls this with zmq_msg_data().
  void pushMessage(void const* data, std::size_t bytes);
  double getCurrentFrameTime() const { return m_curr_frametime; }
  // the de-interleave of pushMessage, usable without a device: message -> [colour x N] and [depth x N]
  static double splitMessage(void const* data, std::size_t bytes, unsigned num_sensors, std::size_t colorsize, std::size_t depthsize,
                             uint8_t* colors_out, uint8_t* depths_out);
  std::size_t framesRead() const { return m_num_frame; }
 private:
  void readFromFiles();
  glm::uvec2 m_resolution_color, m_resolution_depth;
  unsigned m_numLayers;
  std::size_t m_colorsize, m_depthsize;            // per sensor
  uint8_t* m_staging[2] = {nullptr, nullptr};      // pinned, [colour N | depth N]
  int m_back = 0;
  std::atomic<bool> m_dirty{false};            // written by the reader thread, read by update()
  std::mutex m_mutex_pbo;
  std::unique_ptr<std::thread> m_readThread;
  std::atomic<bool> m_running{false};
  bool m_filter_textures = true, m_refine_bound = true, m_use_processed_depth = true;
  std::string m_serverport, m_slaveport;
  std::size_t m_num_frame = 0;
  double m_curr_frametime = 0.0;
  CalibrationFiles const* m_calib_files;
  CalibVolumes const* m_calib_vols;
};

// ---- framework/reconstruction/reconstruction.hpp:11-36 ----------------------------------------------------------------
class Reconstruction {
 public:
  Reconstruction(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox);
  virtual ~Reconstruction() {}
  virtual void draw() = 0;
  virtual void drawF();
  virtual void reload() {}
  virtual void resize(std::size_t width, std::size_t height);
  void setColorMaskMode(unsigned mode) { m_color_mask_mode = mode; }
  virtual void setViewportOffset(float x, float y);
  // replaces the fixed-function state draw() used to read back with glGetFloatv / glGetIntegerv
  void setViewMatrices(float const* modelview16, float const* projection16);
 protected:
  CalibVolumes const* m_cv;
  CalibrationFiles const* m_cf;
  unsigned m_num_kinects;
  gloost::BoundingBox m_bbox;
  unsigned m_color_mask_mode = 0;
  rr_view m_view;
};

// ---- surface extraction (no reference counterpart): the fused surface as an indexed, coloured triangle mesh ---------------
// The arrays of rr_download_mesh (include/rgbd_recon_b200.h states what they hold).
struct Mesh {
  std::vector<float> positions;      // [V][3] metres
  std::vector<float> normals;        // [V][3] unit length, or NaN where the gradient vanishes
  std::vector<float> rgba;           // [V][4] blendColors; alpha 1 quality-weighted, -1 the fallback blend
  std::vector<uint32_t> triangles;   // [T][3] vertex indices, counter-clockwise seen from free space
};
// Binary little-endian PLY: vertex "float x y z nx ny nz uchar red green blue", face "list uchar uint vertex_indices".
// Colour byte = (uint8)(min(max(c, 0), 1) * 255 + 0.5f), a NaN channel counting as 0. Throws if the file cannot be written.
void writePly(std::string const& path, Mesh const& mesh);

// ---- connected parts (no reference counterpart): the separate objects in the fused volume -------------------------------
// The per-part arrays of rr_download_parts (include/rgbd_recon_b200.h states what they hold), in ascending key order.
struct Parts {
  std::vector<uint32_t> voxels;      // [P] inside voxels of the part
  std::vector<int32_t> boxes;        // [P][6] x0, x1, y0, y1, z0, z1, half-open voxel index ranges
  std::vector<float> centroids;      // [P][3] metres
};

// The tracks of rr_download_part_tracks, per part of the Parts they come with (the header states the matching).
struct PartTracks {
  std::vector<uint32_t> track_ids;   // [P] persistent id; 0xFFFFFFFF for a part below min_voxels
  std::vector<uint32_t> prev_parts;  // [P] the previous part it continues; 0xFFFFFFFF for a new track or an untracked part
  std::vector<uint32_t> overlaps;    // [P] voxels shared with that previous part; 0 for none
  std::vector<uint32_t> ended;       // [E] ids of the tracks that ended, by ascending previous part
};

// ---- point clouds (no reference counterpart): the pre-processed, registered sensor points --------------------------------
// The arrays of rr_download_points (include/rgbd_recon_b200.h states what they hold).
struct PointCloud {
  std::vector<float> positions;      // [n][3] metres
  std::vector<float> normals;        // [n][3] the normal stage at the pixel
  std::vector<float> colors;         // [n][3] in [0, 1], the bilinear colour-frame fetch
  std::vector<float> quality;        // [n]
  std::vector<uint32_t> pixels;      // [n] sensor * W * H + y * W + x, ascending
};
// Binary little-endian PLY: vertex "float x y z nx ny nz uchar red green blue float quality", no faces. Colour bytes as the
// mesh writer's: (uint8)(min(max(c, 0), 1) * 255 + 0.5f), a NaN channel counting as 0. Throws if the file cannot be written.
void writePly(std::string const& path, PointCloud const& cloud);

// ---- framework/reconstruction/recon_integration.hpp:33-107 ------------------------------------------------------------
class ReconIntegration : public Reconstruction {
 public:
  ReconIntegration(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox, float limit, float size);
  void draw() override;
  void drawF() override;
  void integrate();
  void setColorFilling(bool active) { m_fill_holes = active; }
  void setUseBricks(bool active);
  void setSpaceSkip(bool active);
  void setVoxelSize(float size);
  void setTsdfLimit(float limit);
  void setBrickSize(float size);
  void setShadeMode(int mode) { m_view.shade_mode = mode; }     // Settings UBO g_shade_mode (kinect_client.cpp:263-266)
  unsigned numBricks() const;
  float occupiedRatio() const { return m_ratio_occupied; }
  float getBrickSize() const;
  void clearOccupiedBricks() const;
  void updateOccupiedBricks();
  void setMinVoxelsPerBrick(unsigned i);
  void resize(std::size_t width, std::size_t height) override;
  glm::uvec3 volumeResolution() const;
  std::vector<float> const& colorImage() const { return m_rgba; }   // RGBA32F, viewport w*h, row 0 = bottom (GL window coords)
  std::vector<float> const& depthImage() const { return m_depth; }  // gl_FragDepth, 1.0 where no surface
  void downloadTsdf(std::vector<float>& out) const;
  // marching cubes over the fused volume on the device (rr_extract_mesh; with several devices rr_group_extract_mesh)
  void extractMesh(Mesh& out) const;
  // the 6-connected parts of the fused volume (rr_label_parts; with several devices rr_group_label_parts), and the part of
  // every vertex [V] and triangle [T] of the last extractMesh, which must come from the same volume state
  void labelParts(Parts& out) const;
  // takes parts of the last labelParts / trackParts (of the current volume state) out of the fused volume: those of fewer
  // than min_voxels voxels and, with keep (one entry per part), those whose entry is 0 (rr_remove_parts; with several devices
  // rr_group_remove_parts); returns (removed parts, removed voxels)
  std::pair<uint32_t, uint32_t> removeParts(uint32_t min_voxels, const std::vector<uint8_t>* keep = nullptr) const;
  void meshParts(std::vector<uint32_t>& vertex_parts, std::vector<uint32_t>& triangle_parts) const;
  // the parts of the fused volume with track ids persistent across frame sets, matched by voxel overlap against the last
  // trackParts (rr_track_parts; with several devices rr_group_track_parts); resetPartTracks starts ids at 0 again
  void trackParts(uint32_t min_voxels, Parts& parts, PartTracks& tracks) const;
  void resetPartTracks() const;
  // the last extractMesh simplified by vertex clustering with clusters of cluster_voxels voxels per side (rr_simplify_mesh;
  // with several devices rr_group_simplify_mesh); sources: per simplified triangle, its source triangle in that mesh
  void simplifyMesh(uint32_t cluster_voxels, Mesh& out, std::vector<uint32_t>* sources = nullptr) const;
  // Queries of the fused volume in metres (rr_sample_points / rr_cast_rays; with several devices their group forms).
  // points, origins, directions, normals, positions: [n][3]; values [n]; rgba [n][4]; steps [n] (0xFFFFFFFF: no hit, with
  // NaN positions and normals). The outputs are resized to n.
  void samplePoints(std::vector<float> const& points, std::vector<float>& values, std::vector<float>& normals, std::vector<float>& rgba) const;
  // distances to the surface: distanceField computes the nearest inside voxel of every voxel of the fused volume and returns
  // the inside count (rr_distance_field; with several devices rr_group_distance_field); sampleDistance queries that field at
  // world points (rr_sample_distance, which refuses a field older than the last integrate): distances [n] in metres, the
  // nearest inside-voxel centres [n][3] in metres and their linear voxel indices [n]
  uint32_t distanceField() const;
  void sampleDistance(std::vector<float> const& points, std::vector<float>& distances, std::vector<float>& nearest_points,
                      std::vector<uint32_t>& nearest_voxels) const;
  void castRays(std::vector<float> const& origins, std::vector<float> const& directions, std::vector<float>& positions,
                std::vector<float>& normals, std::vector<float>& rgba, std::vector<uint32_t>& steps) const;
 private:
  void configure();
  rr_config m_cfg;
  bool m_fill_holes = true;
  float m_ratio_occupied = 0.0f;
  std::vector<float> m_rgba, m_depth;
  mutable uint32_t m_mesh_nv = 0, m_mesh_nt = 0;   // counts of the last extractMesh (meshParts sizes its outputs by them)
};

// ---- framework/reconstruction/recon_points.hpp: every depth pixel of every sensor as a shaded, depth-tested point sprite -----
// (runs on the first device of the context: the pre-processed maps are replicated on every member)
class ReconPoints : public Reconstruction {
 public:
  ReconPoints(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox) : Reconstruction(cfs, cv, bbox) {}
  void draw() override;
  void setShadeMode(int mode) { m_view.shade_mode = mode; }
  std::vector<float> const& colorImage() const { return m_rgba; }
  std::vector<float> const& depthImage() const { return m_depth; }
  // the points draw() keeps before the view transform, of the sensors in sensor_mask, as a point cloud (rr_extract_points;
  // with several devices rr_group_extract_points)
  void extractPoints(PointCloud& out, uint32_t sensor_mask = 0xFFFFFFFFu) const;
 private:
  std::vector<float> m_rgba, m_depth;
};

// ---- framework/reconstruction/recon_trigrid.hpp: a triangle mesh over every sensor's depth pixels, the sensors blended by ----
// quality within epsilon of the front-most surface (depth pass, additive accumulation pass, normalisation pass). m_min_length
// comes from the calibration files like Reconstruction::m_min_length (reconstruction.cpp:20).
class ReconTrigrid : public Reconstruction {
 public:
  ReconTrigrid(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox)
      : Reconstruction(cfs, cv, bbox), m_min_length(cfs.minLength()) {}
  void draw() override;
  void setShadeMode(int mode) { m_view.shade_mode = mode; }
  void setMinLength(float min_length) { m_min_length = min_length; }     // (the reference takes it from the .yml only)
  std::vector<float> const& colorImage() const { return m_rgba; }
  std::vector<float> const& depthImage() const { return m_depth; }
 private:
  float m_min_length;
  std::vector<float> m_rgba, m_depth;
};

// ---- framework/reconstruction/recon_calibs.hpp: the inverse-volume grid's voxel centres coloured by the TSDF (debug view) ----
// Reads the TSDF volume of the first device; with several devices that member holds its own z-slab only.
class ReconCalibs : public Reconstruction {
 public:
  ReconCalibs(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox) : Reconstruction(cfs, cv, bbox) {}
  void draw() override;
  void setActiveKinect(unsigned num_kinect) { m_active_kinect = num_kinect; }
  void setTsdfLimit(float limit) { m_tsdf_limit = limit; }
  std::vector<float> const& colorImage() const { return m_rgba; }
  std::vector<float> const& depthImage() const { return m_depth; }
 private:
  unsigned m_active_kinect = 0;
  float m_tsdf_limit = 0.01f;
  std::vector<float> m_rgba, m_depth;
};

// ---- framework/rendering/timer_database.hpp: the stage names survive, CUDA events replace GL timestamp queries ------------
class TimerDatabase {
 public:
  static TimerDatabase& instance();
  void enable(int level) const;                       // 0 off, 1 numbered top-level stages, 2 every pass
  double duration(std::string const& name) const;     // last interval in milliseconds
  double mean(std::string const& name);               // mean since the previous call of mean() for this name
};

// ---- .ks scene files (kinect_client.cpp:213-234, calib_inverter.cpp:37-59) -----------------------------------------------
struct SceneFile {
  std::vector<std::string> calib_filenames;   // "kinect <path.yml>", relative to the .ks directory unless absolute
  gloost::BoundingBox bbox;                   // "bbx x0 y0 z0 x1 y1 z1", default (-1,0,-1)-(1,2.2,1)
  std::string resource_path;                  // directory of the .ks file, with trailing '/'
};
SceneFile readSceneFile(std::string const& ks_path);

}  // namespace kinect

// ---- framework/io/FeedbackReceiver.h:16-22: the view/mode message a remote client sends back ---------------------------
// Plain data, same layout (three column-major glm::mat4, two unsigned = 200 bytes). The receiver thread and its socket are
// control plane and stay outside; a transport hands the payload to parseFeedback.
namespace sys {
struct feedback {
  float cyclops_mat[16];
  float screen_mat[16];
  float model_mat[16];
  unsigned recon_mode;
  unsigned stream_slot;
};
static_assert(sizeof(feedback) == 200, "sys::feedback must keep the reference's wire layout");
bool parseFeedback(void const* data, std::size_t bytes, feedback& out);   // false unless bytes == sizeof(feedback)
}  // namespace sys
#endif
