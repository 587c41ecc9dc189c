#include "Triangulator.h"

#include <cmath>
#include <cstdint>
#include <mutex>
#include <stdexcept>

namespace {
std::mutex g_reg_mutex;
std::vector<Triangulator*> g_registry;  // live triangulators: getDistFromRay is static in the reference

[[noreturn]] void raise(int status, int mode) {
  if (status == TRI_ERR_DIM) throw std::runtime_error("Every camera should have the same number of points");
  if (status == TRI_ERR_TOO_FEW) throw std::runtime_error(mode == TRI_MATRIX ? "Too few rays are found" : "Too few detections are found");
  throw std::runtime_error(std::string("tri_b200: ") + tri_last_error());
}
}  // namespace

Triangulator::Triangulator(std::vector<const tdr::Camera*> cams, int mode, const char* type, int device)
    : type_(type), cameras(std::move(cams)), mode_(mode) {
  std::vector<tri_camera> desc;
  for (const tdr::Camera* c : cameras) desc.push_back(c->describe());
  int st = tri_create((int)desc.size(), desc.data(), device, &engine_);
  if (st != TRI_OK) throw std::runtime_error(std::string("tri_b200: ") + tri_last_error());
  std::lock_guard<std::mutex> lock(g_reg_mutex);
  g_registry.push_back(this);
}

Triangulator::~Triangulator() {
  {
    std::lock_guard<std::mutex> lock(g_reg_mutex);
    for (size_t i = 0; i < g_registry.size(); i++)
      if (g_registry[i] == this) { g_registry.erase(g_registry.begin() + i); break; }
  }
  tri_destroy(engine_);
}

int Triangulator::cameraIndex(const tdr::Camera* cam) const {
  for (size_t i = 0; i < cameras.size(); i++)
    if (cameras[i] == cam) return (int)i;
  return -1;
}

std::vector<std::pair<cv::Point3d, double>> Triangulator::triangulatePointsOfSubsets(
    const std::vector<std::vector<CamPointPair>>& items) {
  std::vector<int32_t> offs(items.size() + 1, 0), cam;
  std::vector<double> xy;
  for (size_t i = 0; i < items.size(); i++) {
    for (const CamPointPair& p : items[i]) {
      const int idx = cameraIndex(p.camera);
      if (idx < 0) throw std::runtime_error("tri_b200: camera does not belong to this triangulator");
      cam.push_back(idx);
      xy.push_back(p.point.x);
      xy.push_back(p.point.y);
    }
    offs[i + 1] = (int32_t)cam.size();
  }
  std::vector<double> xyz(3 * items.size()), err(items.size());
  int st = tri_triangulate_subsets(engine_, mode_, flags_, (int64_t)items.size(), offs.data(), cam.data(), xy.data(), xyz.data(),
                                   err.data(), nullptr);
  if (st != TRI_OK) raise(st, mode_);
  std::vector<std::pair<cv::Point3d, double>> out(items.size());
  for (size_t i = 0; i < items.size(); i++) out[i] = {cv::Point3d(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]), err[i]};
  return out;
}

std::pair<cv::Point3d, double> Triangulator::triangulatePoint(std::vector<CamPointPair> images) {
  return triangulatePointsOfSubsets({images})[0];
}

unsigned Triangulator::pixelFormatFor(const std::vector<std::vector<cv::Point2d>>& points) {
  // pack [cam][frame] pixel pairs in the narrowest format that holds every value exactly: ushort2 (integer pixels
  // below 65535 -- what DetectionsContainer::readFiles produces, DetectionsContainer.cpp:36 -- with 0xFFFF,0xFFFF
  // for a pair the reference would skip, MatrixTriangulator.cpp:86), float2, else double2
  bool exact16 = true, exact32 = true;
  for (const auto& row : points) {
    for (const cv::Point2d& p : row) {
      if ((double)(float)p.x != p.x || (double)(float)p.y != p.y) { exact32 = false; break; }
      if (exact16 && !(p.x == -1 || p.y == -1) &&
          !(p.x >= 0 && p.x < 65535 && p.y >= 0 && p.y < 65535 && p.x == (double)(uint16_t)p.x && p.y == (double)(uint16_t)p.y))
        exact16 = false;
    }
    if (!exact32) break;
  }
  exact16 = exact16 && exact32;
  return exact16 ? (unsigned)TRI_PIX_U16 : exact32 ? 0u : (unsigned)TRI_PIX_F64;
}

namespace {
// points[cam][frame] packed in the narrowest exact pixel format, then handed to `call(flags, xy)`
template <class Call>
int withPackedPixels(const std::vector<std::vector<cv::Point2d>>& points, int64_t n_frames, Call call) {
  const int n_rows = (int)points.size();
  const unsigned fmt = Triangulator::pixelFormatFor(points);
  if (fmt == TRI_PIX_U16) {
    std::vector<uint16_t> xy(2 * (size_t)n_rows * n_frames);
    for (int c = 0; c < n_rows; c++)
      for (int64_t f = 0; f < n_frames; f++) {
        const cv::Point2d& p = points[c][f];
        const bool missing = p.x == -1 || p.y == -1;
        xy[2 * ((size_t)c * n_frames + f)] = missing ? (uint16_t)0xFFFF : (uint16_t)p.x;
        xy[2 * ((size_t)c * n_frames + f) + 1] = missing ? (uint16_t)0xFFFF : (uint16_t)p.y;
      }
    return call(fmt, (const void*)xy.data());
  }
  if (fmt == 0) {
    std::vector<float> xy(2 * (size_t)n_rows * n_frames);
    for (int c = 0; c < n_rows; c++)
      for (int64_t f = 0; f < n_frames; f++) {
        xy[2 * ((size_t)c * n_frames + f)] = (float)points[c][f].x;
        xy[2 * ((size_t)c * n_frames + f) + 1] = (float)points[c][f].y;
      }
    return call(fmt, (const void*)xy.data());
  }
  std::vector<double> xy(2 * (size_t)n_rows * n_frames);
  for (int c = 0; c < n_rows; c++)
    for (int64_t f = 0; f < n_frames; f++) {
      xy[2 * ((size_t)c * n_frames + f)] = points[c][f].x;
      xy[2 * ((size_t)c * n_frames + f) + 1] = points[c][f].y;
    }
  return call(fmt, (const void*)xy.data());
}
}  // namespace

std::vector<cv::Point3d> MatrixTriangulator::triangulatePointsRobust(const std::vector<std::vector<cv::Point2d>>& points,
                                                                     double maxReprojPx, std::vector<uint32_t>* inliers,
                                                                     std::vector<double>* reprojRms) {
  for (size_t i = 1; i < points.size(); i++)
    if (points[i - 1].size() != points[i].size()) throw std::runtime_error("Every camera should have the same number of points");
  const int64_t n_frames = points.empty() ? 0 : (int64_t)points[0].size();
  std::vector<double> xyz(3 * (size_t)n_frames);
  tri_batch_out out{};
  out.xyz_f64 = xyz.data();
  if (inliers) { inliers->assign((size_t)n_frames, 0); out.mask = inliers->data(); }
  if (reprojRms) { reprojRms->assign((size_t)n_frames, 0.0); out.err = reprojRms->data(); }
  int64_t bad = -1;
  const int st = withPackedPixels(points, n_frames, [&](unsigned fmt, const void* xy) {
    return tri_triangulate_points_robust(engine_, (flags_ & TRI_F32) | fmt, maxReprojPx, xy, (int)points.size(), n_frames, n_frames,
                                         &out, &bad);
  });
  if (st != TRI_OK) raise(st, TRI_MATRIX);
  std::vector<cv::Point3d> result((size_t)n_frames);
  for (int64_t f = 0; f < n_frames; f++) result[f] = cv::Point3d(xyz[3 * f], xyz[3 * f + 1], xyz[3 * f + 2]);
  return result;
}

std::vector<cv::Point3d> Triangulator::triangulatePoints(std::vector<std::vector<cv::Point2d>> points) {
  // MatrixTriangulator.cpp:72-76 / RayTriangulator.cpp:54-58
  for (size_t i = 1; i < points.size(); i++)
    if (points[i - 1].size() != points[i].size()) throw std::runtime_error("Every camera should have the same number of points");
  const int64_t n_frames = points.empty() ? 0 : (int64_t)points[0].size();
  const int n_rows = (int)points.size();
  const unsigned fmt = pixelFormatFor(points);
  const bool exact16 = fmt == TRI_PIX_U16, exact32 = fmt != TRI_PIX_F64;
  std::vector<double> xyz(3 * (size_t)n_frames);
  tri_batch_out out{};
  out.xyz_f64 = xyz.data();
  int64_t bad = -1;
  int st;
  if (exact16) {
    std::vector<uint16_t> xy(2 * (size_t)n_rows * n_frames);
    for (int c = 0; c < n_rows; c++)
      for (int64_t f = 0; f < n_frames; f++) {
        const cv::Point2d& p = points[c][f];
        const bool missing = p.x == -1 || p.y == -1;
        xy[2 * ((size_t)c * n_frames + f)] = missing ? (uint16_t)0xFFFF : (uint16_t)p.x;
        xy[2 * ((size_t)c * n_frames + f) + 1] = missing ? (uint16_t)0xFFFF : (uint16_t)p.y;
      }
    st = tri_triangulate_points(engine_, mode_, flags_ | TRI_PIX_U16, xy.data(), n_rows, n_frames, n_frames, &out, &bad);
  } else if (exact32) {
    std::vector<float> xy(2 * (size_t)n_rows * n_frames);
    for (int c = 0; c < n_rows; c++)
      for (int64_t f = 0; f < n_frames; f++) {
        xy[2 * ((size_t)c * n_frames + f)] = (float)points[c][f].x;
        xy[2 * ((size_t)c * n_frames + f) + 1] = (float)points[c][f].y;
      }
    st = tri_triangulate_points(engine_, mode_, flags_, xy.data(), n_rows, n_frames, n_frames, &out, &bad);
  } else {
    std::vector<double> xy(2 * (size_t)n_rows * n_frames);
    for (int c = 0; c < n_rows; c++)
      for (int64_t f = 0; f < n_frames; f++) {
        xy[2 * ((size_t)c * n_frames + f)] = points[c][f].x;
        xy[2 * ((size_t)c * n_frames + f) + 1] = points[c][f].y;
      }
    st = tri_triangulate_points(engine_, mode_, flags_ | TRI_PIX_F64, xy.data(), n_rows, n_frames, n_frames, &out, &bad);
  }
  if (st != TRI_OK) raise(st, mode_);
  std::vector<cv::Point3d> result((size_t)n_frames);
  for (int64_t f = 0; f < n_frames; f++) result[f] = cv::Point3d(xyz[3 * f], xyz[3 * f + 1], xyz[3 * f + 2]);
  return result;
}

double Triangulator::getDistFromRay(CamPointPair pair, cv::Point3d point) {
  Triangulator* owner = nullptr;
  int idx = -1;
  {
    std::lock_guard<std::mutex> lock(g_reg_mutex);
    for (Triangulator* t : g_registry)
      if ((idx = t->cameraIndex(pair.camera)) >= 0) { owner = t; break; }
  }
  if (!owner) throw std::runtime_error("tri_b200: getDistFromRay needs a live triangulator that owns the camera");
  const int32_t cam = idx;
  const double xy[2] = {pair.point.x, pair.point.y}, p[3] = {point.x, point.y, point.z};
  double d = 0;
  if (tri_dist_from_ray(owner->engine_, 1, &cam, xy, p, &d) != TRI_OK) throw std::runtime_error(std::string("tri_b200: ") + tri_last_error());
  return d;
}

MatrixTriangulator::MatrixTriangulator(std::vector<const tdr::Camera*> cams, int device)
    : Triangulator(std::move(cams), TRI_MATRIX, "matrix", device) {}

RayTriangulator::RayTriangulator(std::vector<const tdr::Camera*> cams, int device, bool exact)
    : Triangulator(std::move(cams), TRI_RAY, "ray", device) {
  flags_ = exact ? (unsigned)TRI_RAY_REFERENCE_LM : (unsigned)TRI_RAY_CLOSED_FORM;
}
