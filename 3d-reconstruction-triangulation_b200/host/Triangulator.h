// Triangulator.h -- the reference's Triangulator interface (src/Triangulator.h:9-59) backed by the
// B200 engine.  Same class names, member names, argument meaning and runtime_error texts as the
// reference, so src/main.cpp:54-65 and src/DroneClassifier.cpp compile against it unchanged apart from
// the include; all arithmetic happens on the GPU through include/tri_b200.h (no CPU path).
#pragma once
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include "Camera.h"
#include "cv_compat.h"

class Triangulator {
 public:
  struct CamPointPair {  // src/Triangulator.h:11-15
    const tdr::Camera* camera;
    cv::Point2d point;
  };
  struct Ray {  // src/Triangulator.h:17-20
    cv::Point3d origin;
    cv::Point3d dir;
  };

  virtual ~Triangulator();

  std::vector<const tdr::Camera*> getCameras() { return cameras; }  // :44
  const tdr::Camera* getCamera(int camera) { return cameras[camera]; }  // :54
  std::string getType() { return type_; }  // :56

  // :46-47 -- one (camera subset, pixels) solve; returns (point, error)
  virtual std::pair<cv::Point3d, double> triangulatePoint(std::vector<CamPointPair> images);
  // :51-52 -- points[cam][frame], (-1,-1) = no detection; throws like the reference
  virtual std::vector<cv::Point3d> triangulatePoints(std::vector<std::vector<cv::Point2d>> points);
  // many subsets in one launch (what a batched caller of triangulatePoint should use)
  std::vector<std::pair<cv::Point3d, double>> triangulatePointsOfSubsets(const std::vector<std::vector<CamPointPair>>& items);

  // narrowest pixel format of the C ABI that holds every value of `points` exactly: TRI_PIX_U16 (integer pixels
  // below 65535; a pair with x == -1 or y == -1 becomes the missing marker), 0 (float2) or TRI_PIX_F64
  static unsigned pixelFormatFor(const std::vector<std::vector<cv::Point2d>>& points);

  // Extension (the reference has no such method): the forward model of the rig, points -> pixels
  // (tri_project_points).  Returns points[cam][frame] for every camera of the triangulator, (-1,-1) where the camera
  // does not see the point (behind it or outside the image) -- exactly triangulatePoints' input.  visible[f]: bit c =
  // camera c sees point f.  FP64 (FP32 if flags() has TRI_F32).
  std::vector<std::vector<cv::Point2d>> projectPoints(const std::vector<cv::Point3d>& points, std::vector<uint32_t>* visible = nullptr);

  // :58 -- distance of `point` to the pixel ray of `pair`
  static double getDistFromRay(CamPointPair pair, cv::Point3d point);

  // engine access for the batched classifier and for callers that own device / pinned buffers
  tri_engine* engine() const { return engine_; }
  unsigned flags() const { return flags_; }
  void setFlags(unsigned f) { flags_ = f; }
  int mode() const { return mode_; }

 protected:
  Triangulator(std::vector<const tdr::Camera*> cameras, int mode, const char* type, int device);
  int cameraIndex(const tdr::Camera* cam) const;

  std::string type_;
  std::vector<const tdr::Camera*> cameras;
  tri_engine* engine_ = nullptr;
  int mode_ = 0;
  unsigned flags_ = 0;
};

class MatrixTriangulator : public Triangulator {  // src/MatrixTriangulator.h:19, type "matrix"
 public:
  explicit MatrixTriangulator(std::vector<const tdr::Camera*> cameras, int device = 0);

  // Extension (the reference has no such method): triangulatePoints that ignores wrong detections.  Same input, packing
  // and runtime_error texts as triangulatePoints; per frame, the two-view hypothesis with the most views within
  // maxReprojPx pixels wins and the point is the DLT over those inlier views (tri_triangulate_points_robust).  A frame
  // where no two views agree gives (0,0,0).  inliers[f]: bit c = camera c used; reprojRms[f]: RMS reprojection error in
  // pixels over the inliers (NaN without consensus).
  std::vector<cv::Point3d> triangulatePointsRobust(const std::vector<std::vector<cv::Point2d>>& points, double maxReprojPx,
                                                   std::vector<uint32_t>* inliers = nullptr, std::vector<double>* reprojRms = nullptr);
};

class RayTriangulator : public Triangulator {  // src/RayTriangulator.h:34, type "ray"
 public:
  // exact = true follows cv::LMSolver's trajectory (TRI_RAY_REFERENCE_LM): bit-comparable with the
  // reference, needed for identical classifier decisions; false = analytic-Jacobian LM (fast path)
  explicit RayTriangulator(std::vector<const tdr::Camera*> cameras, int device = 0, bool exact = true);
};
