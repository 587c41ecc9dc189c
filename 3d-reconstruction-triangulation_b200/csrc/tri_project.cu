// tri_project.cu -- forward projection (tri_project_points*) for sm_100a: world points to per-camera pixels, written in
// the batch input layout ([n_cams][cam_stride] pixel pairs, the missing marker where a camera does not see the point).
//
// Point i, camera c: (x, y, w) = P_c (X_i, 1), (u, v) = (x / w, y / w); visible iff w > 0 and u, v lie in the pixel
// areas of the image, -0.5 <= u < width - 0.5, -0.5 <= v < height - 0.5.  FP64 runs on the cameraPerspectiveMatrix as
// is; FP32 on the rig's centred form (DltRig<float>: the point minus the rig centre `origin`, pix0 added back to (u, v)),
// so the FP32 sums do not cancel at the 10 m scale of a rig.
//
// The shape is the reverse of the streaming skeleton: 12 or 24 B in, n_cams x {8, 16, 4} B out per point.  A
// persistent grid-stride kernel, one point per thread in FP32 and two in FP64 (below): the camera loop is warp-uniform
// and every camera's row is stored coalesced along the warp (256 B
// per warp for float2, 128 B for ushort2, streaming stores).  Nothing is staged: a view's pixel leaves as soon as it is
// computed.  The same device function computes every view in every instantiation (camera-count class, paired or scalar
// stores), so a point's pixels and mask do not depend on which kernel ran it or where it sat in the batch.
#include <math.h>

#include <algorithm>

#include "tri_common.cuh"

namespace tri {

template <typename T>
struct __align__(16) ProjRig {
  DltRig<T> d;
  float lim[TRI_MAX_CAMS][2];  // width - 0.5, height - 0.5 (exact in float for any int32 size below 2^23)
};

constexpr int PROJ_THREADS = 256;
constexpr int PROJ_MIN_CTAS = 4;  // <= 64 registers

// the point in the rig's frame: FP64 rig origin = 0; FP32 subtracts the rig centre in the input's precision
template <typename T, typename In>
__device__ __forceinline__ bool proj_load(const In* __restrict__ xyz, int64_t i, const DltRig<T>& d, T (&X)[3]) {
  const In a = __ldg(xyz + 3 * i), b = __ldg(xyz + 3 * i + 1), c = __ldg(xyz + 3 * i + 2);
  X[0] = (T)(a - (In)d.origin[0]);
  X[1] = (T)(b - (In)d.origin[1]);
  X[2] = (T)(c - (In)d.origin[2]);
  return isfinite(a) && isfinite(b) && isfinite(c);
}

// one view: pixel (u, v) and the visibility rule
template <typename T>
__device__ __forceinline__ bool proj_view(const ProjRig<T>& r, int c, const T (&X)[3], T& u, T& v) {
  const T* P = r.d.P[c];
  const T w = fma_(P[8], X[0], fma_(P[9], X[1], fma_(P[10], X[2], P[11])));
  const T iw = rcp_(w);
  u = fma_(fma_(P[0], X[0], fma_(P[1], X[1], fma_(P[2], X[2], P[3]))), iw, r.d.pix0[c][0]);
  v = fma_(fma_(P[4], X[0], fma_(P[5], X[1], fma_(P[6], X[2], P[7]))), iw, r.d.pix0[c][1]);
  return w > (T)0 && u >= (T)-0.5 && u < (T)r.lim[c][0] && v >= (T)-0.5 && v < (T)r.lim[c][1];
}

__device__ __forceinline__ unsigned short pix_u16(double x) { return (unsigned short)__double2int_rn(x); }  // half to even
__device__ __forceinline__ unsigned short pix_u16(float x) { return (unsigned short)__float2int_rn(x); }

// store one view's pixel pair at row[i]: PAIR = one vector store (the base is aligned to the pair), otherwise two
// scalar stores (a base aligned only to the component type)
template <int PIX, bool PAIR, typename T>
__device__ __forceinline__ void proj_store(char* row, int64_t i, bool vis, T u, T v) {
  if constexpr (PIX == PIX_F32) {
    const float x = vis ? (float)u : -1.0f, y = vis ? (float)v : -1.0f;
    if constexpr (PAIR) __stcs(reinterpret_cast<float2*>(row) + i, make_float2(x, y));
    else { float* p = reinterpret_cast<float*>(row) + 2 * i; __stcs(p, x); __stcs(p + 1, y); }
  } else if constexpr (PIX == PIX_F64) {
    const double x = vis ? (double)u : -1.0, y = vis ? (double)v : -1.0;
    if constexpr (PAIR) __stcs(reinterpret_cast<double2*>(row) + i, make_double2(x, y));
    else { double* p = reinterpret_cast<double*>(row) + 2 * i; __stcs(p, x); __stcs(p + 1, y); }
  } else {
    const unsigned short x = vis ? pix_u16(u) : (unsigned short)0xFFFF, y = vis ? pix_u16(v) : (unsigned short)0xFFFF;
    if constexpr (PAIR) __stcs(reinterpret_cast<unsigned*>(row) + i, (unsigned)x | (unsigned)y << 16);
    else { unsigned short* p = reinterpret_cast<unsigned short*>(row) + 2 * i; __stcs(p, x); __stcs(p + 1, y); }
  }
}

// PPT points per thread, PROJ_THREADS apart (each camera's stores stay coalesced along the warp): the camera loop loads a
// view's constants once for all of them.
template <typename T, typename In, int PIX, int NC, bool PAIR, int PPT>
__global__ void __launch_bounds__(PROJ_THREADS, PROJ_MIN_CTAS)
project_kernel(const __grid_constant__ ProjRig<T> rig, const In* __restrict__ xyz, int64_t n_points, char* __restrict__ xy,
               int64_t row_bytes, uint32_t* __restrict__ mask, int n_cams) {
  const int64_t step = (int64_t)gridDim.x * PROJ_THREADS * PPT;
  for (int64_t i0 = (int64_t)blockIdx.x * PROJ_THREADS * PPT + threadIdx.x; i0 < n_points; i0 += step) {
    T X[PPT][3];
    bool fin[PPT], live[PPT];
    uint32_t m[PPT];
#pragma unroll
    for (int k = 0; k < PPT; k++) {
      live[k] = i0 + k * PROJ_THREADS < n_points;
      X[k][0] = X[k][1] = X[k][2] = (T)0;
      fin[k] = live[k] && proj_load<T, In>(xyz, i0 + k * PROJ_THREADS, rig.d, X[k]);
      m[k] = 0;
    }
    for_cams<NC>(n_cams, [&](int c) {
#pragma unroll
      for (int k = 0; k < PPT; k++) {
        T u, v;
        const bool vis = proj_view<T>(rig, c, X[k], u, v) && fin[k];
        m[k] |= (uint32_t)vis << c;
        if (xy && live[k]) proj_store<PIX, PAIR, T>(xy + c * row_bytes, i0 + k * PROJ_THREADS, vis, u, v);
      }
    });
#pragma unroll
    for (int k = 0; k < PPT; k++)
      if (mask && live[k]) __stcs(mask + i0 + k * PROJ_THREADS, m[k]);
  }
}

template <typename T, typename In, int PIX, int NC, bool PAIR, int PPT = 1>
static cudaError_t project_run(const LaunchCtx& ctx, const ProjRig<T>& rig, const In* xyz, int64_t n_points, char* xy,
                               int64_t row_bytes, uint32_t* mask, int n_cams) {
  auto kern = project_kernel<T, In, PIX, NC, PAIR, PPT>;
  int per_sm = 0;
  cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, PROJ_THREADS, 0);
  if (err != cudaSuccess) return err;
  const int64_t blocks = (n_points + PROJ_THREADS * PPT - 1) / (PROJ_THREADS * PPT);
  const int64_t grid = std::min<int64_t>(blocks, (int64_t)ctx.sm_count * std::max(per_sm, 1));
  kern<<<(unsigned)grid, PROJ_THREADS, 0, ctx.stream>>>(rig, xyz, n_points, xy, row_bytes, mask, n_cams);
  ++*ctx.launches;
  return cudaGetLastError();
}

// camera-count class and store width
template <typename T, typename In, int PIX>
static cudaError_t project_dispatch(const LaunchCtx& ctx, const ProjRig<T>& rig, const In* xyz, int64_t n_points, void* d_xy,
                                    int64_t cam_stride, uint32_t* mask, int n_cams) {
  char* xy = static_cast<char*>(d_xy);
  const int64_t row_bytes = cam_stride * pix_bytes(PIX);
  if ((uintptr_t)xy % pix_bytes(PIX) != 0)  // rows aligned only to the component: scalar stores, the rolled loop
    return project_run<T, In, PIX, 0, false>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
  // FP64 stays rolled at every camera count: its DFMAs take the rig constants through registers (LDC.64), and unrolled,
  // ptxas hoists the loads of every camera's twelve constants ahead of the arithmetic -- 8 cameras: 127 registers and
  // spills without a register cap, 64 and 430+ bytes of spills with one.  Rolled, the constants are LDCs with a
  // run-time index, so each thread takes two points and loads a view's constants once for both (measured on a B200,
  // 8 cameras x 100 M points: 3.11 -> 2.18 ms)
  if constexpr (sizeof(T) == 8) {
    return project_run<T, In, PIX, 0, true, 2>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
  } else {
    if (n_cams <= 4) return project_run<T, In, PIX, 4, true>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
    if (n_cams <= 8) return project_run<T, In, PIX, 8, true>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
    if (n_cams <= 16) return project_run<T, In, PIX, 16, true>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
    return project_run<T, In, PIX, 0, true>(ctx, rig, xyz, n_points, xy, row_bytes, mask, n_cams);
  }
}

template <typename T, typename In>
static cudaError_t project_fmt(const LaunchCtx& ctx, int pixfmt, const ProjRig<T>& rig, const In* xyz, int64_t n_points, void* d_xy,
                               int64_t cam_stride, uint32_t* mask, int n_cams) {
  if (pixfmt == PIX_F32) return project_dispatch<T, In, PIX_F32>(ctx, rig, xyz, n_points, d_xy, cam_stride, mask, n_cams);
  if (pixfmt == PIX_F64) return project_dispatch<T, In, PIX_F64>(ctx, rig, xyz, n_points, d_xy, cam_stride, mask, n_cams);
  return project_dispatch<T, In, PIX_U16>(ctx, rig, xyz, n_points, d_xy, cam_stride, mask, n_cams);
}

template <typename T>
static cudaError_t project_rig(const LaunchCtx& ctx, int pixfmt, const DltRig<T>& d, const tri_camera* cams, int n_cams,
                               const float* xyz_f32, const double* xyz_f64, int64_t n_points, void* d_xy, int64_t cam_stride,
                               uint32_t* mask) {
  ProjRig<T> r;
  r.d = d;
  r.d.n_use = n_cams;
  for (int c = 0; c < TRI_MAX_CAMS; c++) {
    r.lim[c][0] = c < n_cams ? (float)((double)cams[c].width - 0.5) : 0.0f;
    r.lim[c][1] = c < n_cams ? (float)((double)cams[c].height - 0.5) : 0.0f;
  }
  if (xyz_f32) return project_fmt<T, float>(ctx, pixfmt, r, xyz_f32, n_points, d_xy, cam_stride, mask, n_cams);
  return project_fmt<T, double>(ctx, pixfmt, r, xyz_f64, n_points, d_xy, cam_stride, mask, n_cams);
}

cudaError_t launch_project(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64, const DltRig<float>& rig32,
                           const tri_camera* cams, int n_cams, const float* d_xyz_f32, const double* d_xyz_f64, int64_t n_points,
                           void* d_xy, int64_t cam_stride, uint32_t* d_mask) {
  if (n_points <= 0) return cudaSuccess;
  if (f32) return project_rig<float>(ctx, pixfmt, rig32, cams, n_cams, d_xyz_f32, d_xyz_f64, n_points, d_xy, cam_stride, d_mask);
  return project_rig<double>(ctx, pixfmt, rig64, cams, n_cams, d_xyz_f32, d_xyz_f64, n_points, d_xy, cam_stride, d_mask);
}

}  // namespace tri
