// Implementation of the GL-free host classes declared in rr_host.hpp. Every method forwards to the C ABI of
// librr_b200.so; no computation of the fusion path happens in this file.
#include "rr_host.hpp"

#include <cuda_runtime_api.h>

#include <chrono>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

namespace kinect {

// ---------------------------------------------------------------------------------------------------- gpu::Context
namespace gpu {
static Context* g_current = nullptr;

Context::Context(int device, CalibrationFiles const& cfs) : Context(std::vector<int>(1, device), cfs) {}
Context::Context(std::vector<int> const& devices, CalibrationFiles const& cfs) : m_group(nullptr), m_ctx(nullptr) {
  const int rc = rr_group_create(&m_group, devices.data(), (int)devices.size(), (int)cfs.num(), (int)cfs.getWidth(), (int)cfs.getHeight(),
                                 (int)cfs.getWidthC(), (int)cfs.getHeightC());
  if (rc != RR_OK) throw std::runtime_error("rr_group_create failed with status " + std::to_string(rc) + " (CUDA devices are required; there is no CPU fallback)");
  m_ctx = rr_group_member(m_group, 0);
  g_current = this;
}
Context::~Context() {
  if (g_current == this) g_current = nullptr;
  rr_group_destroy(m_group);
}
Context& Context::current() {
  if (!g_current) throw std::runtime_error("no kinect::gpu::Context: create one before CalibVolumes / NetKinectArray / ReconIntegration");
  return *g_current;
}
void Context::check(int status, char const* what) const {
  if (status != RR_OK) throw std::runtime_error(std::string(what) + ": " + rr_last_error(m_ctx));
}
void Context::checkGroup(int status, char const* what) const {
  if (status != RR_OK) throw std::runtime_error(std::string(what) + ": " + rr_group_last_error(m_group));
}
}  // namespace gpu

// member 0 of the device group: queries, read-backs, timers (brick tables and calibration are identical on every member)
static rr_ctx* ctx() { return gpu::Context::current().handle(); }
static void ck(int status, char const* what) { gpu::Context::current().check(status, what); }
// everything that changes state goes to the whole group (one device: a pass-through)
static rr_group* grp() { return gpu::Context::current().group(); }
static void gk(int status, char const* what) { gpu::Context::current().checkGroup(status, what); }

// basefile = calib_file minus its 3-character extension (CalibVolumes.cpp:34-39, calibration_inverter.cpp:17-21)
static std::string strip_ext3(std::string const& f) {
  if (f.size() < 3) throw std::runtime_error("calibration file name too short: " + f);
  return f.substr(0, f.size() - 3);
}
static std::string basename_of(std::string const& f) { return f.substr(f.find_last_of("/\\") + 1); }

// ---------------------------------------------------------------------------------------------------- CalibVolumes
CalibVolumes::CalibVolumes(std::vector<std::string> const& calib_volume_files, gloost::BoundingBox const& bbox) : m_res_inv(0), m_bbox(bbox) {
  for (auto const& f : calib_volume_files) {
    m_cv_xyz_filenames.push_back(strip_ext3(f) + "cv_xyz");
    m_cv_uv_filenames.push_back(strip_ext3(f) + "cv_uv");
  }
  const float mn[3] = {bbox.getPMin()[0], bbox.getPMin()[1], bbox.getPMin()[2]};
  const float mx[3] = {bbox.getPMax()[0], bbox.getPMax()[1], bbox.getPMax()[2]};
  gk(rr_group_set_bbox(grp(), mn, mx), "rr_set_bbox");
  m_res.resize(num()); m_limits.resize(num()); m_frustums.resize(num());
  for (unsigned i = 0; i < num(); ++i) addVolume(i, m_cv_xyz_filenames[i], m_cv_uv_filenames[i]);
}

void CalibVolumes::addVolume(unsigned i, std::string const& filename_xyz, std::string const& filename_uv) {
  CalibrationVolume<xyz> vx{filename_xyz};
  CalibrationVolume<uv> vu{filename_uv};
  if (vx.res() != vu.res()) throw std::runtime_error("cv_xyz / cv_uv resolutions differ: " + filename_xyz);
  const uint32_t res[3] = {vx.res().x, vx.res().y, vx.res().z};
  const float lim[2] = {vx.depthLimits().x, vx.depthLimits().y};
  gk(rr_group_calib_upload(grp(), (int)i, reinterpret_cast<float const*>(vx.volume().data()), reinterpret_cast<float const*>(vu.volume().data()), res, lim), "rr_calib_upload");
  m_res[i] = vx.res();
  m_limits[i] = vx.depthLimits();
  float planes[24], cams[RR_HOST_MAX_SENSORS * 3];
  ck(rr_get_frustum_planes(ctx(), (int)i, planes), "rr_get_frustum_planes");
  ck(rr_get_camera_positions(ctx(), cams), "rr_get_camera_positions");
  std::array<glm::fvec4, 6> pl;
  for (int k = 0; k < 6; ++k) pl[k] = glm::fvec4(planes[k * 4], planes[k * 4 + 1], planes[k * 4 + 2], planes[k * 4 + 3]);
  m_frustums[i] = Frustum(pl, glm::fvec3(cams[i * 3], cams[i * 3 + 1], cams[i * 3 + 2]));
}

void CalibVolumes::loadInverseCalibs(std::string const& path) {
  for (unsigned i = 0; i < num(); ++i) {
    const std::string name = path + basename_of(m_cv_xyz_filenames[i]) + "_inv";
    CalibrationVolume<glm::fvec4> v{name};
    const uint32_t res[3] = {v.res().x, v.res().y, v.res().z};
    gk(rr_group_calib_upload_inv(grp(), (int)i, reinterpret_cast<float const*>(v.volume().data()), res), "rr_calib_upload_inv");
    m_res_inv = v.res();
  }
}

glm::uvec3 CalibVolumes::getVolumeRes() const { return m_res_inv; }
glm::fvec2 CalibVolumes::getDepthLimits(unsigned i) const { return m_limits.at(i); }
std::vector<glm::fvec3> CalibVolumes::getCameraPositions() const {
  std::vector<glm::fvec3> out;
  for (auto const& f : m_frustums) out.push_back(f.getCameraPos());
  return out;
}

// ---------------------------------------------------------------------------------------------------- CalibrationInverter
CalibrationInverter::CalibrationInverter(std::vector<std::string> const& calib_volume_files, gloost::BoundingBox const& bbox) : m_bbox(bbox) {
  for (auto const& f : calib_volume_files) m_cv_xyz_filenames.push_back(strip_ext3(f) + "cv_xyz");
  const float mn[3] = {bbox.getPMin()[0], bbox.getPMin()[1], bbox.getPMin()[2]};
  const float mx[3] = {bbox.getPMax()[0], bbox.getPMax()[1], bbox.getPMax()[2]};
  gk(rr_group_set_bbox(grp(), mn, mx), "rr_set_bbox");
  for (unsigned i = 0; i < m_cv_xyz_filenames.size(); ++i) {
    std::cerr << "loading " << m_cv_xyz_filenames[i] << std::endl;
    CalibrationVolume<xyz> vx{m_cv_xyz_filenames[i]};
    std::vector<float> no_uv((std::size_t)vx.numVoxels() * 2, 0.0f);     // the inverter needs cv_xyz only
    const uint32_t res[3] = {vx.res().x, vx.res().y, vx.res().z};
    const float lim[2] = {vx.depthLimits().x, vx.depthLimits().y};
    gk(rr_group_calib_upload(grp(), (int)i, reinterpret_cast<float const*>(vx.volume().data()), no_uv.data(), res, lim), "rr_calib_upload");
  }
}

void CalibrationInverter::calculateInverseVolumes(glm::uvec3 const& volume_res) {
  m_data_volumes_xyz_inv.clear();
  const uint32_t res[3] = {volume_res.x, volume_res.y, volume_res.z};
  const auto t0 = std::chrono::steady_clock::now();
  for (unsigned i = 0; i < m_cv_xyz_filenames.size(); ++i) {
    std::vector<glm::fvec4> inv((std::size_t)volume_res.x * volume_res.y * volume_res.z);
    ck(rr_calib_invert(ctx(), (int)i, res, reinterpret_cast<float*>(inv.data()), 0), "rr_calib_invert");
    // the inverse volume's header carries the constants (0.5, 4.5) (calibration_inverter.cpp:153)
    m_data_volumes_xyz_inv.emplace_back(volume_res, glm::fvec2(0.5f, 4.5f), inv);
  }
  m_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

void CalibrationInverter::writeInverseVolumes(std::string const& path) const {
  for (unsigned i = 0; i < m_data_volumes_xyz_inv.size(); ++i) {
    const std::string name_output = path + basename_of(m_cv_xyz_filenames[i]) + "_inv";
    std::cout << "writing to file " << name_output << std::endl;
    m_data_volumes_xyz_inv[i].write(name_output);
  }
}

// ---------------------------------------------------------------------------------------------------- calibration .yml
static float komma_string_to_float(std::string const& token) {                          // KinectCalibrationFile.cpp:601-605
  return token.empty() ? 0.0f : (float)std::atof(token.substr(0, token.length() - 1).c_str());
}
static float next_token_as_float(std::ifstream& in) { std::string t; in >> t; return komma_string_to_float(t); }   // :611-618
static float next_float(std::ifstream& in) { std::string t; in >> t; return (float)std::atof(t.c_str()); }          // :621-627
static void advance_to(std::string const& what, std::ifstream& in) { std::string t; while (in >> t) if (t == what) return; }   // :583-595

bool KinectCalibrationFile::parse() {
  std::ifstream infile(_filePath.c_str());
  if (!infile) return false;
  std::string token;
  while (infile >> token) {
    if (token == "rgb_size:") { advance_to("[", infile); _widthc = (unsigned)next_token_as_float(infile); _heightc = (unsigned)next_float(infile); }
    else if (token == "depth_size:") { advance_to("[", infile); _width = (unsigned)next_token_as_float(infile); _height = (unsigned)next_float(infile); }
    else if (token == "near_far:") { advance_to("[", infile); _near = next_token_as_float(infile); _far = next_float(infile); }
    else if (token == "compress_rgb:") { advance_to("[", infile); _iscompressedrgb = (unsigned)next_token_as_float(infile); next_float(infile); }
    else if (token == "min_length:") { advance_to("[", infile); min_length = next_token_as_float(infile); next_float(infile); }
    else if (token == "compress_depth:") { advance_to("[", infile); _iscompresseddepth = ((unsigned)next_token_as_float(infile)) != 0; next_float(infile); }
  }
  return true;
}

CalibrationFiles::CalibrationFiles(std::vector<std::string> const& calib_filenames)
    : m_width(0), m_widthc(0), m_height(0), m_heightc(0), m_compressed_rgb(0), m_compressed_d(false), m_filenames(calib_filenames) {
  if (calib_filenames.empty()) throw std::invalid_argument("CalibrationFiles: no calibration files");
  KinectCalibrationFile first(calib_filenames[0]);
  if (!first.parse()) throw std::invalid_argument("cannot open calibration file " + calib_filenames[0]);
  m_width = first.getWidth(); m_height = first.getHeight(); m_widthc = first.getWidthC(); m_heightc = first.getHeightC();
  if (!m_width || !m_height || !m_widthc || !m_heightc)
    throw std::invalid_argument("calibration file " + calib_filenames[0] + " lacks rgb_size: / depth_size:");
  m_compressed_rgb = first.isCompressedRGB(); m_compressed_d = first.isCompressedDepth();
  m_near = first.getNear(); m_far = first.getFar(); m_min_length = first.min_length;
  // every sensor's own depth range (the reference keeps a KinectCalibrationFile per sensor, calibration_files.cpp:12-20)
  m_near_far.assign(1, std::make_pair(m_near, m_far));
  for (std::size_t i = 1; i < calib_filenames.size(); ++i) {
    KinectCalibrationFile f(calib_filenames[i]);
    if (!f.parse()) throw std::invalid_argument("cannot open calibration file " + calib_filenames[i]);
    m_near_far.push_back(std::make_pair(f.getNear(), f.getFar()));
  }
}

// ---------------------------------------------------------------------------------------------------- NetKinectArray
double NetKinectArray::splitMessage(void const* data, std::size_t bytes, unsigned num_sensors, std::size_t colorsize, std::size_t depthsize,
                                    uint8_t* colors_out, uint8_t* depths_out) {
  if (!data || bytes != (colorsize + depthsize) * num_sensors)
    throw std::invalid_argument("stream message has " + std::to_string(bytes) + " bytes, expected " +
                                std::to_string((colorsize + depthsize) * num_sensors));
  double t = 0.0;
  if (bytes >= sizeof(double)) std::memcpy(&t, data, sizeof(double));                  // NetKinectArray.cpp:525
  const uint8_t* src = static_cast<const uint8_t*>(data);
  std::size_t offset = 0;
  for (unsigned i = 0; i < num_sensors; ++i) {                                            // :531-538
    std::memcpy(colors_out + i * colorsize, src + offset, colorsize); offset += colorsize;
    std::memcpy(depths_out + i * depthsize, src + offset, depthsize); offset += depthsize;
  }
  return t;
}

void NetKinectArray::pushMessage(void const* data, std::size_t bytes) {
  std::vector<uint8_t> color(m_colorsize * m_numLayers), depth(m_depthsize * m_numLayers);
  const double t = splitMessage(data, bytes, m_numLayers, m_colorsize, m_depthsize, color.data(), depth.data());
  pushFrame(color.data(), depth.data());
  m_curr_frametime = t;
}

NetKinectArray::NetKinectArray(std::string const& serverport, std::string const& slaveport, CalibrationFiles const* calibs, CalibVolumes const* vols, bool readfromfile)
    : m_resolution_color(calibs->getWidthC(), calibs->getHeightC()), m_resolution_depth(calibs->getWidth(), calibs->getHeight()),
      m_numLayers(calibs->num()), m_serverport(serverport), m_slaveport(slaveport), m_calib_files(calibs), m_calib_vols(vols) {
  // NetKinectArray.cpp:120-142: DXT1 = w*h/2 bytes, DXT5 = w*h (the reference's 307200 at 640x480), RGB8 = w*h*3;
  // depth 1 byte (sqrt-compressed) or a float per texel
  const unsigned crgb = calibs->isCompressedRGB();
  if (crgb != 0 && crgb != 1 && crgb != 5) throw std::runtime_error("compress_rgb must be 0 (RGB8), 1 (DXT1) or 5 (DXT5)");
  const std::size_t cpx = (std::size_t)m_resolution_color.x * m_resolution_color.y;
  m_colorsize = crgb == 1 ? cpx / 2 : (crgb == 5 ? cpx : cpx * 3);
  m_depthsize = (std::size_t)m_resolution_depth.x * m_resolution_depth.y * (calibs->isCompressedDepth() ? 1 : sizeof(float));
  std::vector<float> near_far;
  // per sensor, as the reference reads them (getCalibs()[i].getNear() / getFar(), NetKinectArray.cpp:345-351)
  for (unsigned i = 0; i < m_numLayers; ++i) { near_far.push_back(calibs->getNear(i)); near_far.push_back(calibs->getFar(i)); }
  gk(rr_group_set_frame_format(grp(), crgb == 1 ? RR_COLOR_DXT1 : (crgb == 5 ? RR_COLOR_DXT5 : RR_COLOR_RGB8),
                         calibs->isCompressedDepth() ? RR_DEPTH_U8 : RR_DEPTH_F32, near_far.data()), "rr_set_frame_format");
  for (int b = 0; b < 2; ++b)
    if (cudaMallocHost((void**)&m_staging[b], (m_colorsize + m_depthsize) * m_numLayers) != cudaSuccess) throw std::runtime_error("pinned staging allocation failed");
  if (readfromfile) {
    m_running = true;
    m_readThread.reset(new std::thread(&NetKinectArray::readFromFiles, this));
  }
}

NetKinectArray::~NetKinectArray() {
  m_running = false;
  if (m_readThread) m_readThread->join();
  rr_group_synchronize(grp());
  for (int b = 0; b < 2; ++b) cudaFreeHost(m_staging[b]);
}

void NetKinectArray::pushFrame(void const* color, void const* depth) {
  std::lock_guard<std::mutex> lock(m_mutex_pbo);
  // the reader's side of the double buffer: fill the back pinned buffer and start its copy into the back device slot;
  // the copy overlaps whatever the main thread is still computing on the current slot
  gk(rr_group_stage_sync(grp()), "rr_stage_sync");          // the copy that last read this pinned buffer pair has finished
  uint8_t* dst = m_staging[m_back];
  std::memcpy(dst, color, m_colorsize * m_numLayers);
  std::memcpy(dst + m_colorsize * m_numLayers, depth, m_depthsize * m_numLayers);
  gk(rr_group_stage_frames(grp(), dst, m_colorsize * m_numLayers, dst + m_colorsize * m_numLayers, m_depthsize * m_numLayers), "rr_stage_frames");
  m_back ^= 1;
  m_dirty = true;
  ++m_num_frame;
}

// .stream playback: one file per sensor, each frame = colour bytes then depth bytes (NetKinectArray.cpp:724-764); loops at EOF
void NetKinectArray::readFromFiles() {
  std::vector<std::string> names;
  std::stringstream ss(m_serverport);
  for (std::string tok; std::getline(ss, tok, ';');) if (!tok.empty()) names.push_back(tok);
  if (names.size() != m_numLayers) { std::cerr << "expected " << m_numLayers << " stream files" << std::endl; m_running = false; return; }
  std::vector<std::ifstream> files;
  for (auto const& n : names) {
    files.emplace_back(n, std::ios::binary);
    if (!files.back()) { std::cerr << "cannot open stream " << n << std::endl; m_running = false; return; }
  }
  std::vector<uint8_t> color(m_colorsize * m_numLayers), depth(m_depthsize * m_numLayers);
  while (m_running) {
    bool ok = true;
    for (unsigned i = 0; i < m_numLayers && ok; ++i) {
      files[i].read(reinterpret_cast<char*>(color.data() + m_colorsize * i), (std::streamsize)m_colorsize);
      files[i].read(reinterpret_cast<char*>(depth.data() + m_depthsize * i), (std::streamsize)m_depthsize);
      ok = (bool)files[i];
    }
    if (!ok) {
      for (auto& f : files) { f.clear(); f.seekg(0); }
      continue;
    }
    pushFrame(color.data(), depth.data());
    while (m_running) {                      // HWM 1: wait until the consumer took the frame (NetKinectArray.cpp:491-492)
      { std::lock_guard<std::mutex> lock(m_mutex_pbo); if (!m_dirty) break; }
      std::this_thread::sleep_for(std::chrono::microseconds(200));
    }
  }
}

bool NetKinectArray::update() {
  std::lock_guard<std::mutex> lock(m_mutex_pbo);
  if (!m_dirty) return false;
  // swapBuffers (NetKinectArray.cpp:229-236): the staged device slot becomes the one the kernels read
  gk(rr_group_swap_frames(grp()), "rr_swap_frames");
  m_dirty = false;
  return true;
}

void NetKinectArray::processTextures() {
  gk(rr_group_preprocess(grp(), m_filter_textures ? 1 : 0, m_use_processed_depth ? 1 : 0, m_refine_bound ? 1 : 0), "rr_preprocess");
}
void NetKinectArray::filterTextures(bool filter) { m_filter_textures = filter; processTextures(); }
void NetKinectArray::useProcessedDepths(bool filter) { m_use_processed_depth = filter; processTextures(); }
void NetKinectArray::refineBoundary(bool filter) { m_refine_bound = filter; processTextures(); }

// ---------------------------------------------------------------------------------------------------- Reconstruction
Reconstruction::Reconstruction(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox)
    : m_cv(cv), m_cf(&cfs), m_num_kinects(cfs.num()), m_bbox(bbox) {
  std::memset(&m_view, 0, sizeof(m_view));
  for (int i = 0; i < 4; ++i) m_view.modelview[i * 5] = m_view.projection[i * 5] = 1.0f;
  m_view.viewport[2] = 1280; m_view.viewport[3] = 720;     // View(1280, 720), recon_integration.cpp:32-34
}
void Reconstruction::drawF() {
  TimerDatabase::instance();      // "draw" is timed inside the library (reconstruction.cpp:35-39)
  draw();
}
void Reconstruction::resize(std::size_t width, std::size_t height) { m_view.viewport[2] = (int)width; m_view.viewport[3] = (int)height; }
void Reconstruction::setViewportOffset(float x, float y) { m_view.viewport[0] = (int)x; m_view.viewport[1] = (int)y; }
void Reconstruction::setViewMatrices(float const* modelview16, float const* projection16) {
  std::memcpy(m_view.modelview, modelview16, sizeof(float) * 16);
  std::memcpy(m_view.projection, projection16, sizeof(float) * 16);
}

// ---------------------------------------------------------------------------------------------------- ReconIntegration
ReconIntegration::ReconIntegration(CalibrationFiles const& cfs, CalibVolumes const* cv, gloost::BoundingBox const& bbox, float limit, float size)
    : Reconstruction(cfs, cv, bbox) {
  m_cfg.limit = limit; m_cfg.voxel_size = size; m_cfg.brick_size = 0.1f; m_cfg.min_voxels_per_brick = 10;   // recon_integration.cpp:51-59
  m_cfg.use_bricks = 1; m_cfg.skip_space = 1; m_cfg.store_weight = 0;
  setVoxelSize(size);
}
void ReconIntegration::configure() { gk(rr_group_configure(grp(), &m_cfg), "rr_configure"); }
void ReconIntegration::setVoxelSize(float size) {
  m_cfg.voxel_size = size;
  configure();
  uint32_t r[3];
  ck(rr_get_volume_res(ctx(), r), "rr_get_volume_res");
  std::cout << "resolution " << r[0] << ", " << r[1] << ", " << r[2] << " - " << ((std::size_t)r[0] * r[1] * r[2]) / 1000 << "k voxels" << std::endl;
}
void ReconIntegration::setBrickSize(float size) { m_cfg.brick_size = size; configure(); }
void ReconIntegration::setTsdfLimit(float limit) { m_cfg.limit = limit; configure(); }
void ReconIntegration::setUseBricks(bool active) { m_cfg.use_bricks = active ? 1 : 0; configure(); }
void ReconIntegration::setSpaceSkip(bool active) { m_cfg.skip_space = active ? 1 : 0; configure(); }
void ReconIntegration::setMinVoxelsPerBrick(unsigned i) {
  // kinect_client.cpp:391-395: the GUI callback re-runs updateOccupiedBricks() and integrate() itself
  m_cfg.min_voxels_per_brick = i;
  configure();
}
unsigned ReconIntegration::numBricks() const { uint32_t n = 0; ck(rr_get_brick_info(ctx(), nullptr, nullptr, &n), "rr_get_brick_info"); return n; }
float ReconIntegration::getBrickSize() const { float s = 0; ck(rr_get_brick_info(ctx(), nullptr, &s, nullptr), "rr_get_brick_info"); return s; }
glm::uvec3 ReconIntegration::volumeResolution() const { uint32_t r[3]; ck(rr_get_volume_res(ctx(), r), "rr_get_volume_res"); return glm::uvec3(r[0], r[1], r[2]); }
void ReconIntegration::clearOccupiedBricks() const { gk(rr_group_bricks_clear(grp()), "rr_bricks_clear"); }
void ReconIntegration::updateOccupiedBricks() {
  uint32_t n = 0;
  gk(rr_group_bricks_update(grp(), &n, &m_ratio_occupied), "rr_bricks_update");
}
void ReconIntegration::integrate() { gk(rr_group_integrate(grp()), "rr_integrate"); }
void ReconIntegration::resize(std::size_t width, std::size_t height) { Reconstruction::resize(width, height); }
void ReconIntegration::draw() {
  const std::size_t n = (std::size_t)m_view.viewport[2] * m_view.viewport[3];
  m_rgba.resize(n * 4); m_depth.resize(n);
  gk(rr_group_raymarch(grp(), &m_view, m_rgba.data(), m_depth.data()), "rr_raymarch");
}
void ReconIntegration::drawF() {
  // drawDepthLimits + draw + fillColors (recon_integration.cpp:151-175): brick space skipping happens inside
  // rr_raymarch; with m_fill_holes (the default) the colour image is the hole-filled one
  Reconstruction::drawF();
  if (m_fill_holes) gk(rr_group_fill_colors(grp(), m_rgba.data()), "rr_fill_colors");
}
void ReconPoints::draw() {                                   // recon_points.cpp:71-111
  const std::size_t n = (std::size_t)m_view.viewport[2] * m_view.viewport[3];
  m_rgba.resize(n * 4); m_depth.resize(n);
  ck(rr_draw_points(ctx(), &m_view, m_rgba.data(), m_depth.data()), "rr_draw_points");
}
void ReconPoints::extractPoints(PointCloud& out, uint32_t sensor_mask) const {
  if (sensor_mask == 0xFFFFFFFFu && m_num_kinects < 32) sensor_mask = (1u << m_num_kinects) - 1u;   // the default: every sensor
  uint32_t n = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_extract_points(grp(), sensor_mask, &n), "rr_group_extract_points");
  else ck(rr_extract_points(ctx(), sensor_mask, &n), "rr_extract_points");
  out.positions.resize((std::size_t)n * 3); out.normals.resize((std::size_t)n * 3); out.colors.resize((std::size_t)n * 3);
  out.quality.resize(n); out.pixels.resize(n);
  ck(rr_download_points(ctx(), out.positions.data(), out.normals.data(), out.colors.data(), out.quality.data(), out.pixels.data()),
     "rr_download_points");
}
void ReconTrigrid::draw() {                                  // recon_trigrid.cpp:82-149
  const std::size_t n = (std::size_t)m_view.viewport[2] * m_view.viewport[3];
  m_rgba.resize(n * 4); m_depth.resize(n);
  ck(rr_draw_trigrid(ctx(), &m_view, m_min_length, m_rgba.data(), m_depth.data()), "rr_draw_trigrid");
}
void ReconCalibs::draw() {                                   // recon_calibs.cpp:56-66
  const std::size_t n = (std::size_t)m_view.viewport[2] * m_view.viewport[3];
  m_rgba.resize(n * 4); m_depth.resize(n);
  ck(rr_draw_calibs(ctx(), &m_view, (int)m_active_kinect, m_tsdf_limit, m_rgba.data(), m_depth.data()), "rr_draw_calibs");
}
void ReconIntegration::downloadTsdf(std::vector<float>& out) const {
  const glm::uvec3 r = volumeResolution();
  out.resize((std::size_t)r.x * r.y * r.z);
  gk(rr_group_download_tsdf(grp(), out.data()), "rr_download_tsdf");
}

void ReconIntegration::extractMesh(Mesh& out) const {
  uint32_t nv = 0, nt = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_extract_mesh(grp(), &nv, &nt), "rr_group_extract_mesh");
  else ck(rr_extract_mesh(ctx(), &nv, &nt), "rr_extract_mesh");
  out.positions.resize((std::size_t)nv * 3); out.normals.resize((std::size_t)nv * 3); out.rgba.resize((std::size_t)nv * 4);
  out.triangles.resize((std::size_t)nt * 3);
  ck(rr_download_mesh(ctx(), out.positions.data(), out.normals.data(), out.rgba.data(), out.triangles.data()), "rr_download_mesh");
  m_mesh_nv = nv; m_mesh_nt = nt;
}

void ReconIntegration::labelParts(Parts& out) const {
  uint32_t n = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_label_parts(grp(), &n), "rr_group_label_parts");
  else ck(rr_label_parts(ctx(), &n), "rr_label_parts");
  out.voxels.resize(n); out.boxes.resize((std::size_t)n * 6); out.centroids.resize((std::size_t)n * 3);
  ck(rr_download_parts(ctx(), out.voxels.data(), out.boxes.data(), out.centroids.data(), nullptr), "rr_download_parts");
}

std::pair<uint32_t, uint32_t> ReconIntegration::removeParts(uint32_t min_voxels, const std::vector<uint8_t>* keep) const {
  uint32_t parts = 0, voxels = 0;
  const uint8_t* k = keep ? keep->data() : nullptr;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_remove_parts(grp(), min_voxels, k, &parts, &voxels), "rr_group_remove_parts");
  else ck(rr_remove_parts(ctx(), min_voxels, k, &parts, &voxels), "rr_remove_parts");
  return {parts, voxels};
}

void ReconIntegration::trackParts(uint32_t min_voxels, Parts& parts, PartTracks& tracks) const {
  uint32_t n = 0, e = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_track_parts(grp(), min_voxels, &n, &e), "rr_group_track_parts");
  else ck(rr_track_parts(ctx(), min_voxels, &n, &e), "rr_track_parts");
  parts.voxels.resize(n); parts.boxes.resize((std::size_t)n * 6); parts.centroids.resize((std::size_t)n * 3);
  ck(rr_download_parts(ctx(), parts.voxels.data(), parts.boxes.data(), parts.centroids.data(), nullptr), "rr_download_parts");
  tracks.track_ids.resize(n); tracks.prev_parts.resize(n); tracks.overlaps.resize(n); tracks.ended.resize(e);
  ck(rr_download_part_tracks(ctx(), tracks.track_ids.data(), tracks.prev_parts.data(), tracks.overlaps.data(), tracks.ended.data()),
     "rr_download_part_tracks");
}

void ReconIntegration::resetPartTracks() const { ck(rr_reset_part_tracks(ctx()), "rr_reset_part_tracks"); }

void ReconIntegration::simplifyMesh(uint32_t cluster_voxels, Mesh& out, std::vector<uint32_t>* sources) const {
  uint32_t nv = 0, nt = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_simplify_mesh(grp(), cluster_voxels, &nv, &nt), "rr_group_simplify_mesh");
  else ck(rr_simplify_mesh(ctx(), cluster_voxels, &nv, &nt), "rr_simplify_mesh");
  out.positions.resize((std::size_t)nv * 3); out.normals.resize((std::size_t)nv * 3); out.rgba.resize((std::size_t)nv * 4);
  out.triangles.resize((std::size_t)nt * 3);
  if (sources) sources->resize(nt);
  ck(rr_download_simplified_mesh(ctx(), out.positions.data(), out.normals.data(), out.rgba.data(), out.triangles.data(),
                                 sources ? sources->data() : nullptr), "rr_download_simplified_mesh");
}

void ReconIntegration::meshParts(std::vector<uint32_t>& vertex_parts, std::vector<uint32_t>& triangle_parts) const {
  vertex_parts.resize(m_mesh_nv); triangle_parts.resize(m_mesh_nt);
  ck(rr_download_mesh_parts(ctx(), vertex_parts.data(), triangle_parts.data()), "rr_download_mesh_parts");
}

void ReconIntegration::samplePoints(std::vector<float> const& points, std::vector<float>& values, std::vector<float>& normals,
                                    std::vector<float>& rgba) const {
  if (points.size() % 3) throw std::runtime_error("samplePoints: points must hold whole [x, y, z] triples");
  const std::size_t n = points.size() / 3;
  if (n >= (std::size_t(1) << 31)) throw std::runtime_error("samplePoints: 2^31 or more points");
  values.resize(n); normals.resize(n * 3); rgba.resize(n * 4);
  if (gpu::Context::current().numDevices() > 1)
    gk(rr_group_sample_points(grp(), RR_QUERY_WORLD, points.data(), (uint32_t)n, values.data(), normals.data(), rgba.data()), "rr_group_sample_points");
  else
    ck(rr_sample_points(ctx(), RR_QUERY_WORLD, points.data(), (uint32_t)n, values.data(), normals.data(), rgba.data()), "rr_sample_points");
}

uint32_t ReconIntegration::distanceField() const {
  uint32_t n = 0;
  if (gpu::Context::current().numDevices() > 1) gk(rr_group_distance_field(grp(), &n), "rr_group_distance_field");
  else ck(rr_distance_field(ctx(), &n), "rr_distance_field");
  return n;
}

void ReconIntegration::sampleDistance(std::vector<float> const& points, std::vector<float>& distances, std::vector<float>& nearest_points,
                                      std::vector<uint32_t>& nearest_voxels) const {
  if (points.size() % 3) throw std::runtime_error("sampleDistance: points must hold whole [x, y, z] triples");
  const std::size_t n = points.size() / 3;
  if (n >= (std::size_t(1) << 31)) throw std::runtime_error("sampleDistance: 2^31 or more points");
  distances.resize(n); nearest_points.resize(n * 3); nearest_voxels.resize(n);
  if (gpu::Context::current().numDevices() > 1)
    gk(rr_group_sample_distance(grp(), RR_QUERY_WORLD, points.data(), (uint32_t)n, distances.data(), nearest_points.data(),
                                nearest_voxels.data()), "rr_group_sample_distance");
  else
    ck(rr_sample_distance(ctx(), RR_QUERY_WORLD, points.data(), (uint32_t)n, distances.data(), nearest_points.data(),
                          nearest_voxels.data()), "rr_sample_distance");
}

void ReconIntegration::castRays(std::vector<float> const& origins, std::vector<float> const& directions, std::vector<float>& positions,
                                std::vector<float>& normals, std::vector<float>& rgba, std::vector<uint32_t>& steps) const {
  if (origins.size() % 3 || origins.size() != directions.size()) throw std::runtime_error("castRays: origins and directions must be equal-length [n][3]");
  const std::size_t n = origins.size() / 3;
  if (n >= (std::size_t(1) << 31)) throw std::runtime_error("castRays: 2^31 or more rays");
  positions.resize(n * 3); normals.resize(n * 3); rgba.resize(n * 4); steps.resize(n);
  if (gpu::Context::current().numDevices() > 1)
    gk(rr_group_cast_rays(grp(), RR_QUERY_WORLD, origins.data(), directions.data(), (uint32_t)n, positions.data(), normals.data(), rgba.data(),
                          steps.data()), "rr_group_cast_rays");
  else
    ck(rr_cast_rays(ctx(), RR_QUERY_WORLD, origins.data(), directions.data(), (uint32_t)n, positions.data(), normals.data(), rgba.data(),
                    steps.data()), "rr_cast_rays");
}

static uint8_t ply_byte(float v) {
  v = v > 0.0f ? v : 0.0f;                     // NaN -> 0
  v = v < 1.0f ? v : 1.0f;
  return (uint8_t)(v * 255.0f + 0.5f);
}

void writePly(std::string const& path, Mesh const& mesh) {
  const std::size_t nv = mesh.positions.size() / 3, nt = mesh.triangles.size() / 3;
  std::ofstream o(path, std::ios::binary);
  if (!o) throw std::runtime_error("cannot write " + path);
  o << "ply\nformat binary_little_endian 1.0\ncomment fused surface (rr_extract_mesh)\n"
    << "element vertex " << nv << "\nproperty float x\nproperty float y\nproperty float z\n"
    << "property float nx\nproperty float ny\nproperty float nz\n"
    << "property uchar red\nproperty uchar green\nproperty uchar blue\n"
    << "element face " << nt << "\nproperty list uchar uint vertex_indices\nend_header\n";
  static_assert(sizeof(float) == 4 && sizeof(uint32_t) == 4, "PLY float / uint are 4 bytes");
  std::vector<char> buf;
  buf.reserve(nv * 27 + nt * 13);
  auto put = [&](void const* p, std::size_t n) { buf.insert(buf.end(), static_cast<char const*>(p), static_cast<char const*>(p) + n); };
  for (std::size_t i = 0; i < nv; ++i) {
    put(&mesh.positions[i * 3], 12);
    put(&mesh.normals[i * 3], 12);
    for (int c = 0; c < 3; ++c) { const uint8_t b = ply_byte(mesh.rgba[i * 4 + c]); put(&b, 1); }
  }
  const uint8_t three = 3;
  for (std::size_t t = 0; t < nt; ++t) { put(&three, 1); put(&mesh.triangles[t * 3], 12); }
  o.write(buf.data(), (std::streamsize)buf.size());
  if (!o) throw std::runtime_error("cannot write " + path);
}

void writePly(std::string const& path, PointCloud const& cloud) {
  const std::size_t n = cloud.positions.size() / 3;
  std::ofstream o(path, std::ios::binary);
  if (!o) throw std::runtime_error("cannot write " + path);
  o << "ply\nformat binary_little_endian 1.0\ncomment pre-processed sensor points (rr_extract_points)\n"
    << "element vertex " << n << "\nproperty float x\nproperty float y\nproperty float z\n"
    << "property float nx\nproperty float ny\nproperty float nz\n"
    << "property uchar red\nproperty uchar green\nproperty uchar blue\nproperty float quality\nend_header\n";
  std::vector<char> buf;
  buf.reserve(n * 31);
  auto put = [&](void const* p, std::size_t k) { buf.insert(buf.end(), static_cast<char const*>(p), static_cast<char const*>(p) + k); };
  for (std::size_t i = 0; i < n; ++i) {
    put(&cloud.positions[i * 3], 12);
    put(&cloud.normals[i * 3], 12);
    for (int c = 0; c < 3; ++c) { const uint8_t b = ply_byte(cloud.colors[i * 3 + c]); put(&b, 1); }
    put(&cloud.quality[i], 4);
  }
  o.write(buf.data(), (std::streamsize)buf.size());
  if (!o) throw std::runtime_error("cannot write " + path);
}

// ---------------------------------------------------------------------------------------------------- TimerDatabase
TimerDatabase& TimerDatabase::instance() { static TimerDatabase t; return t; }
void TimerDatabase::enable(int level) const { gk(rr_group_set_timing(grp(), level), "rr_set_timing"); }
double TimerDatabase::duration(std::string const& name) const {
  float ms = 0.0f;
  ck(rr_get_stage_ms(ctx(), name.c_str(), &ms), "rr_get_stage_ms");
  return ms;
}
double TimerDatabase::mean(std::string const& name) {
  float total = 0.0f; uint32_t n = 0;
  ck(rr_get_stage_stats(ctx(), name.c_str(), &total, &n), "rr_get_stage_stats");
  return n ? total / n : 0.0;
}

// ---------------------------------------------------------------------------------------------------- .ks files
SceneFile readSceneFile(std::string const& ks_path) {
  SceneFile sc;
  sc.bbox = gloost::BoundingBox(gloost::Point3(-1.0f, 0.0f, -1.0f), gloost::Point3(1.0f, 2.2f, 1.0f));   // kinect_client.cpp:208-209
  const std::size_t slash = ks_path.find_last_of("/\\");
  sc.resource_path = slash == std::string::npos ? std::string("./") : ks_path.substr(0, slash + 1);
  std::ifstream in(ks_path);
  if (!in) throw std::invalid_argument("cannot open scene file " + ks_path);
  std::string token;
  while (in >> token) {
    if (token == "kinect") {
      std::string f;
      in >> f;
      if (f.empty()) break;
      sc.calib_filenames.push_back(f[0] == '/' ? f : sc.resource_path + f);
    } else if (token == "bbx") {
      float v[6];
      for (float& x : v) in >> x;
      sc.bbox = gloost::BoundingBox(gloost::Point3(v[0], v[1], v[2]), gloost::Point3(v[3], v[4], v[5]));
    }
  }
  if (sc.calib_filenames.empty()) throw std::invalid_argument("scene file names no 'kinect <file.yml>' entries: " + ks_path);
  return sc;
}

}  // namespace kinect

namespace sys {
bool parseFeedback(void const* data, std::size_t bytes, feedback& out) {
  if (!data || bytes != sizeof(feedback)) return false;
  std::memcpy(&out, data, sizeof(feedback));
  return true;
}
}  // namespace sys
