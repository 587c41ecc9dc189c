// tri_engine.cuh -- the engine object behind the C ABI (one GPU + one camera rig).
#pragma once
#include <string>

#include "tri_common.cuh"

namespace tri {

constexpr int N_SLOTS = 3;  // host-buffer path: H2D of chunk k+1 | kernel of chunk k | D2H of chunk k-1

struct Slot {
  cudaStream_t stream = nullptr;
  void* cls_work = nullptr;             // classifier work buffers (tri_classify.cu), grow-only
  void (*cls_work_free)(void*) = nullptr;
  char* d_in = nullptr;
  size_t in_cap = 0;
  char* d_out = nullptr;
  size_t out_cap = 0;
};

void set_error(const std::string& s);
int fail(int status, const std::string& s);
int cuda_fail(cudaError_t err, const char* what);

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace tri

struct tri_engine {
  int device = 0;
  int n_cams = 0;
  int sm_count = 0;
  tri_camera cams[TRI_MAX_CAMS];
  tri::DltRig<double> rig64;
  tri::DltRig<float> rig32;
  tri::RayRig ray;
  tri::RayFold<double> fold64;
  tri::RayFold<float> fold32;
  unsigned long long* d_first_bad = nullptr;  // [0]: latch of the device entry point (collected by tri_device_status), [1]: of the host-buffer path
  tri::Slot slots[tri::N_SLOTS];
  int64_t launches = 0;
  // scratch for the small host-buffer entry points (subsets, dist_from_ray, classify)
  char* d_scratch = nullptr;
  size_t scratch_cap = 0;
  cudaStream_t stream = nullptr;
  void* cls_work = nullptr;             // classifier work buffers (tri_classify.cu), grow-only
  void (*cls_work_free)(void*) = nullptr;

  tri::LaunchCtx ctx(cudaStream_t s, int64_t frame_base = 0, bool host_path = false) {
    return tri::LaunchCtx{s, sm_count, d_first_bad + (host_path ? 1 : 0), frame_base, &launches};
  }
};
