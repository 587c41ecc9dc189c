// tri_engine.cuh -- the engine object behind the C ABI (one GPU + one camera rig).
#pragma once
#include <string>
#include <thread>
#include <vector>

#include "tri_common.cuh"

namespace tri {

constexpr int N_SLOTS = 3;  // host-buffer path: H2D of chunk k+1 | kernel of chunk k | D2H of chunk k-1

// Grow-only device buffer: work space that lives on the engine across calls (cudaMalloc / cudaFree of a few hundred MB
// per call cost up to a second, far more than the kernels).  Growing frees the old buffer first and never copies it.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t bytes) {
    if (bytes <= cap && p) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
    if (e == cudaSuccess) cap = bytes ? bytes : 1;
    return e;
  }
  template <typename T> T* as() { return static_cast<T*>(p); }
};

inline size_t up256(size_t v) { return (v + 255) / 256 * 256; }

struct Slot {
  cudaStream_t stream = nullptr;
  DevBuf in, out;
};

int fail(int status, const std::string& s);
int cuda_fail(cudaError_t err, const char* what);

#define TRI_CUDA(call)                                         \
  do {                                                         \
    cudaError_t err__ = (call);                                \
    if (err__ != cudaSuccess) return cuda_fail(err__, #call);  \
  } while (0)

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

// The *_multi calls: fn(g) for every engine g, each on a host thread of its own.  Returns TRI_OK, or the status and
// message of the lowest-indexed engine that failed.
template <class Fn>
int fan_out(int n_engines, Fn fn) {
  std::vector<int> status(n_engines, TRI_OK);
  std::vector<std::string> msg(n_engines);
  std::vector<std::thread> workers;
  for (int g = 0; g < n_engines; g++)
    workers.emplace_back([&, g]() {
      status[g] = fn(g);
      if (status[g] != TRI_OK) msg[g] = tri_last_error();  // the message is thread-local
    });
  for (std::thread& t : workers) t.join();
  for (int g = 0; g < n_engines; g++)
    if (status[g] != TRI_OK) return fail(status[g], msg[g]);
  return TRI_OK;
}

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
  tri::DevBuf scratch;  // for the small host-buffer entry points (subsets, dist_from_ray)
  cudaStream_t stream = nullptr;
  void* cls_work = nullptr;             // classifier work buffers (tri_classify.cu), grow-only
  void (*cls_work_free)(void*) = nullptr;

  tri::LaunchCtx ctx(cudaStream_t s, int64_t frame_base = 0, bool host_path = false) {
    return tri::LaunchCtx{s, sm_count, d_first_bad + (host_path ? 1 : 0), frame_base, &launches};
  }
};
