// project_selftest.cpp -- round-trips points through Triangulator::projectPoints and MatrixTriangulator::triangulatePoints
// on the GPU and prints the results as text for tests/test_gpu_project.py.  usage: host_project_selftest <n_cams> <n_points>
// The rig is synthetic.ring_rig(n_cams): cameras on a ring of radius 6 m at z = 3 m looking at (0, 0, 1 m), 1920 x 1080.
// The points fill the synthetic volume, plus two that some cameras cannot see (outside the ring, far above it).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>

#include "Triangulator.h"
#include "utils.h"

namespace {
// synthetic.look_at_quat: (w,x,y,z) of the camera-to-world rotation whose +z axis points from pos to target
void look_at_quat(const double p[3], const double t[3], double q[4]) {
  double z[3] = {t[0] - p[0], t[1] - p[1], t[2] - p[2]};
  const double zn = std::sqrt(z[0] * z[0] + z[1] * z[1] + z[2] * z[2]);
  for (double& v : z) v /= zn;
  double x[3] = {z[1], -z[0], 0.0};  // z x (0,0,1)
  const double xn = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
  for (double& v : x) v /= xn;
  const double y[3] = {z[1] * x[2] - z[2] * x[1], z[2] * x[0] - z[0] * x[2], z[0] * x[1] - z[1] * x[0]};
  const double R[3][3] = {{x[0], y[0], z[0]}, {x[1], y[1], z[1]}, {x[2], y[2], z[2]}};
  const double tr = R[0][0] + R[1][1] + R[2][2];
  if (tr > 0) {
    const double s = std::sqrt(tr + 1.0) * 2;
    q[0] = 0.25 * s; q[1] = (R[2][1] - R[1][2]) / s; q[2] = (R[0][2] - R[2][0]) / s; q[3] = (R[1][0] - R[0][1]) / s;
  } else if (R[0][0] > R[1][1] && R[0][0] > R[2][2]) {
    const double s = std::sqrt(1.0 + R[0][0] - R[1][1] - R[2][2]) * 2;
    q[0] = (R[2][1] - R[1][2]) / s; q[1] = 0.25 * s; q[2] = (R[0][1] + R[1][0]) / s; q[3] = (R[0][2] + R[2][0]) / s;
  } else if (R[1][1] > R[2][2]) {
    const double s = std::sqrt(1.0 + R[1][1] - R[0][0] - R[2][2]) * 2;
    q[0] = (R[0][2] - R[2][0]) / s; q[1] = (R[0][1] + R[1][0]) / s; q[2] = 0.25 * s; q[3] = (R[1][2] + R[2][1]) / s;
  } else {
    const double s = std::sqrt(1.0 + R[2][2] - R[0][0] - R[1][1]) * 2;
    q[0] = (R[1][0] - R[0][1]) / s; q[1] = (R[0][2] + R[2][0]) / s; q[2] = (R[1][2] + R[2][1]) / s; q[3] = 0.25 * s;
  }
}
}  // namespace

int main(int argc, const char** argv) {
  if (argc < 3) return 2;
  const int nc = std::atoi(argv[1]), n = std::atoi(argv[2]);
  if (nc < 2 || nc > TRI_MAX_CAMS || n < 1) return 2;
  std::vector<const tdr::Camera*> cams;
  const double target[3] = {0.0, 0.0, 1000.0};
  for (int k = 0; k < nc; k++) {
    const double a = 2 * M_PI * k / nc;
    const double pos[3] = {6000.0 * std::cos(a), 6000.0 * std::sin(a), 3000.0};
    double q[4];
    look_at_quat(pos, target, q);
    cams.push_back(createCamera(k + 1, 1920, 1080, 1081.0810546875, pos, q));
  }
  std::vector<cv::Point3d> pts;
  for (int i = 0; i < n; i++) {  // a low-discrepancy fill of the synthetic volume
    const double fx = std::fmod(0.5 + i * 0.6180339887498949, 1.0), fy = std::fmod(0.5 + i * 0.7548776662466927, 1.0),
                 fz = std::fmod(0.5 + i * 0.5698402909980532, 1.0);
    pts.push_back(cv::Point3d(-2000.0 + 4000.0 * fx, -2000.0 + 4000.0 * fy, 200.0 + 2300.0 * fz));
  }
  pts.push_back(cv::Point3d(9000.0, 0.0, 3000.0));  // outside the ring: behind the cameras on its side
  pts.push_back(cv::Point3d(0.0, 0.0, 60000.0));    // far above the frustums
  MatrixTriangulator matrix(cams);
  std::vector<uint32_t> vis;
  const std::vector<std::vector<cv::Point2d>> px = matrix.projectPoints(pts, &vis);
  for (size_t i = 0; i < pts.size(); i++) {
    std::printf("point %zu %.17g %.17g %.17g %u\n", i, pts[i].x, pts[i].y, pts[i].z, vis[i]);
    for (int c = 0; c < nc; c++) std::printf("pix %zu %d %.17g %.17g\n", i, c, px[c][i].x, px[c][i].y);
  }
  // the round trip over the points at least two cameras see: triangulatePoints(projectPoints(X)) == X
  std::vector<size_t> keep;
  for (size_t i = 0; i < pts.size(); i++)
    if (__builtin_popcount(vis[i]) >= 2) keep.push_back(i);
  std::vector<std::vector<cv::Point2d>> in(nc, std::vector<cv::Point2d>(keep.size()));
  for (int c = 0; c < nc; c++)
    for (size_t k = 0; k < keep.size(); k++) in[c][k] = px[c][keep[k]];
  const std::vector<cv::Point3d> back = matrix.triangulatePoints(in);
  double worst = 0;
  for (size_t k = 0; k < keep.size(); k++) {
    const cv::Point3d& X = pts[keep[k]];
    const double scale = std::fmax(std::fmax(std::fabs(X.x), std::fabs(X.y)), std::fmax(std::fabs(X.z), 1.0));
    worst = std::fmax(worst, cv::norm(back[k] - X) / scale);
  }
  std::printf("roundtrip %zu %.17g\n", keep.size(), worst);
  // an empty batch projects to empty rows
  const std::vector<std::vector<cv::Point2d>> none = matrix.projectPoints({});
  std::printf("empty %zu %zu\n", none.size(), none.empty() ? (size_t)0 : none[0].size());
  for (const auto& cam : cams) delete cam;
  return 0;
}
