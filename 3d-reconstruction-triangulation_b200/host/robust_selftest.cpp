// robust_selftest.cpp -- drives MatrixTriangulator::triangulatePointsRobust on the GPU and prints its results as text
// for tests/test_gpu_robust.py.  usage: host_robust_selftest <cameras.xml> <points.txt> <max_reproj_px>
// points.txt: "n_cams n_frames", then one line per camera of n_frames "x y" pairs ((-1,-1) = no detection).
#include <cstdio>
#include <cstdlib>
#include <stdexcept>

#include "Triangulator.h"
#include "utils.h"

int main(int argc, const char** argv) {
  if (argc < 4) return 2;
  std::vector<const tdr::Camera*> cams = loadCamerasXML(argv[1]);
  FILE* fh = std::fopen(argv[2], "r");
  if (!fh) return 2;
  int nc = 0, nf = 0;
  if (std::fscanf(fh, "%d %d", &nc, &nf) != 2) return 2;
  std::vector<std::vector<cv::Point2d>> pts(nc, std::vector<cv::Point2d>(nf));
  for (int c = 0; c < nc; c++)
    for (int f = 0; f < nf; f++)
      if (std::fscanf(fh, "%lf %lf", &pts[c][f].x, &pts[c][f].y) != 2) return 2;
  std::fclose(fh);
  const double tau = std::atof(argv[3]);
  MatrixTriangulator matrix(cams);

  std::vector<uint32_t> inliers;
  std::vector<double> rms;
  const std::vector<cv::Point3d> xyz = matrix.triangulatePointsRobust(pts, tau, &inliers, &rms);
  for (int f = 0; f < nf; f++)
    std::printf("robust %d %.17g %.17g %.17g %u %.17g\n", f, xyz[f].x, xyz[f].y, xyz[f].z, inliers[f], rms[f]);

  // the reference's exceptions
  try {
    std::vector<std::vector<cv::Point2d>> ragged = pts;
    ragged[1].pop_back();
    matrix.triangulatePointsRobust(ragged, tau);
    std::printf("throw_dim none\n");
  } catch (const std::runtime_error& e) { std::printf("throw_dim %s\n", e.what()); }
  try {
    std::vector<std::vector<cv::Point2d>> few = pts;
    for (size_t c = 1; c < few.size(); c++) few[c][0] = cv::Point2d(-1, -1);
    matrix.triangulatePointsRobust(few, tau);
    std::printf("throw_few none\n");
  } catch (const std::runtime_error& e) { std::printf("throw_few %s\n", e.what()); }
  for (const auto& cam : cams) delete cam;
  return 0;
}
