// tri_common.cuh -- shared declarations of the sm_100a triangulation kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tri_b200.h"

namespace tri {

// ---- per-rig constants, passed BY VALUE as __grid_constant__ kernel parameters so that every FP
// instruction can take its camera operand straight from the constant bank (no loads, no registers).

// MatrixTriangulator rows (MatrixTriangulator.cpp:16-49): a = P[r,0:3] - u*P[2,0:3], b = u*P[2,3] - P[r,3]
constexpr int DLT_TABLE_ROW = 12;  // M00 M01 M02 M11 M12 M22 v0 v1 v2 + padding (16-byte vector loads)
template <typename T>
struct __align__(16) DltRig {
  T P[TRI_MAX_CAMS][12];  // FP64: cameraPerspectiveMatrix as is.  FP32: world origin moved to the
                          // rig centre and pixel origin to (cx,cy) (algebraically the same rows)
  T pix0[TRI_MAX_CAMS][2];  // pixel origin subtracted before use (0 for FP64)
  T origin[3];              // world origin added back to the solution (0 for FP64)
  // device, [TRI_MAX_CAMS / 8][256][DLT_TABLE_ROW]: row (g, m) = what the cameras 8g + {bits of m} add to the normal
  // equations at the canonical pixel (the rig's pixel origin) -- absent views are accumulated there and this row is
  // subtracted afterwards (tri_matrix.cu); built by the host with the kernels' own dlt_view.  FP32 rig only (null in
  // the FP64 rig, whose kernels clear an absent view's coefficients instead)
  const T* absent;
  int n_use;  // pixel rows of this launch (set per launch)
};

// Ray constants (Triangulator.cpp:15-55).  depth = 1/tan(fovy*0.0174533/2) is evaluated on the
// host with the same libm call as the reference so the kernels never call tan().
struct RayRig {  // literal form: what the reference-LM emulation reads (same operation order)
  double aspect[TRI_MAX_CAMS];  // (double)width / (double)height
  double width[TRI_MAX_CAMS], height[TRI_MAX_CAMS];
  double depth[TRI_MAX_CAMS];
  double quat[TRI_MAX_CAMS][4];
  double pos[TRI_MAX_CAMS][3];
};

// Folded form for the fused ray kernel.  With v = (ax*px+bx, ay*py+by, depth) the pixel ray of
// Triangulator.cpp:27-44 before normalisation and R the (unnormalised) quaternion sandwich matrix of
// Triangulator.cpp:15-25, the rotated direction is dir = u / |v| with u = R v = U0*px + U1*py + U2.
// |dir|^2 = n4 = |q|^4.  Positions are relative to the rig centre `origin`.
template <typename T>
struct __align__(16) RayFold {
  T U0[TRI_MAX_CAMS][3], U1[TRI_MAX_CAMS][3], U2[TRI_MAX_CAMS][3];
  T ax[TRI_MAX_CAMS], bx[TRI_MAX_CAMS], ay[TRI_MAX_CAMS], by[TRI_MAX_CAMS], dd[TRI_MAX_CAMS];  // dd = depth^2
  T n4[TRI_MAX_CAMS];
  T ob[TRI_MAX_CAMS][3];    // camera position - origin
  T n4ob[TRI_MAX_CAMS][3];  // n4 * ob
  T n4ob2[TRI_MAX_CAMS];    // n4 * |ob|^2
  T origin[3];
  // device, [256][8]: the sums that depend on the validity mask alone -- n4ob (3), n4, ob (3), n4ob2 -- over the
  // cameras of an 8-bit mask, added in camera order (bit-identical to adding them view by view)
  const T* mask_table;
};
constexpr int TRI_RAY_TABLE_CAMS = 8;

struct BatchOut {
  float* xyz_f32;
  double* xyz_f64;
  uint32_t* mask;
  double* err;
  int32_t* iters;
};

enum PixFmt { PIX_F32 = 0, PIX_F64 = 1, PIX_U16 = 2 };

__host__ __device__ inline int pix_bytes(int fmt) { return fmt == PIX_F32 ? 8 : fmt == PIX_F64 ? 16 : 4; }

// The sentinel test of MatrixTriangulator.cpp:86 / RayTriangulator.cpp:66 on the stored type.
__device__ __forceinline__ bool pix_valid(float x, float y) { return x != -1.0f && y != -1.0f; }
__device__ __forceinline__ bool pix_valid(double x, double y) { return x != -1.0 && y != -1.0; }
// ushort2 pixels, one 32-bit word each (x in the low half): (0xFFFF, 0xFFFF) marks "no detection"
__device__ __forceinline__ bool pix_valid(unsigned q) { return q != 0xffffffffu; }
__device__ __forceinline__ unsigned u16_x(unsigned q) { return q & 0xffffu; }
__device__ __forceinline__ unsigned u16_y(unsigned q) { return q >> 16; }

template <typename T> __device__ __forceinline__ T to_real(float v);
template <> __device__ __forceinline__ float to_real<float>(float v) { return v; }
template <> __device__ __forceinline__ double to_real<double>(float v) { return (double)v; }

// streaming (read-once) vector loads
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float2 ld_stream(const float2* p) { return __ldcs(p); }
__device__ __forceinline__ double2 ld_stream(const double2* p) { return __ldcs(p); }
__device__ __forceinline__ uint2 ld_stream(const uint2* p) { return __ldcs(p); }
__device__ __forceinline__ unsigned ld_stream(const unsigned* p) { return __ldcs(p); }

// Solve the 3x3 symmetric positive definite system M X = v by the adjugate (one reciprocal).
// M = (m00 m01 m02 m11 m12 m22).  cond(A^T A) <= ~25 on real rigs (SURVEY.md F1), so this matches
// cv::invert(DECOMP_SVD) X = pinv(A) b (MatrixTriangulator.cpp:53-54) to ~1e-15 relative in FP64.
// Explicit fused multiply-adds everywhere below (and in the policies): the rounding sequence is then
// fixed by the source, so every kernel variant (vector / scalar path, any camera-count template)
// returns bit-identical points for the same frame.  fma_ is also the host's correctly rounded fma, so the
// host builds its tables with the kernels' own functions.
__host__ __device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }
__host__ __device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }

// Reciprocal for the solves.  FP64: MUFU.RCP64H seed + two Newton steps (5 FP64 instructions, <= 1 ulp)
// instead of the ~35-instruction IEEE division -- the FP64 pipe is the bound of every FP64 kernel here
// (the ray solve has one reciprocal per view).  Deterministic, so all kernel variants stay bit-identical.
// FP32 keeps the correctly rounded division.  The oracle-order code (tri_ref.cuh) does not use this.
__device__ __forceinline__ double rcp_(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(fma(-x, r, 1.0), r, r);
  r = fma(fma(-x, r, 1.0), r, r);
  return r;
}
__device__ __forceinline__ float rcp_(float x) { return 1.0f / x; }
// 1 / |v|^2 of a pixel ray (|v|^2 >= depth^2 > 0, finite): FP64 as above; FP32 one MUFU.RCP (<= 1 ulp) instead of
// the ~9-instruction IEEE division with its slow-path branch -- the FP32 ray kernel is issue-bound.
__device__ __forceinline__ double rcp_ray(double x) { return rcp_(x); }
__device__ __forceinline__ float rcp_ray(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

template <typename T>
__device__ __forceinline__ void solve_sym3(const T M[6], const T v[3], T X[3]) {
  const T c00 = fma_(M[3], M[5], -mul_(M[4], M[4]));
  const T c01 = fma_(M[2], M[4], -mul_(M[1], M[5]));
  const T c02 = fma_(M[1], M[4], -mul_(M[2], M[3]));
  const T c11 = fma_(M[0], M[5], -mul_(M[2], M[2]));
  const T c12 = fma_(M[1], M[2], -mul_(M[0], M[4]));
  const T c22 = fma_(M[0], M[3], -mul_(M[1], M[1]));
  const T det = fma_(M[0], c00, fma_(M[1], c01, mul_(M[2], c02)));
  const T inv = rcp_(det);
  X[0] = mul_(fma_(c00, v[0], fma_(c01, v[1], mul_(c02, v[2]))), inv);
  X[1] = mul_(fma_(c01, v[0], fma_(c11, v[1], mul_(c12, v[2]))), inv);
  X[2] = mul_(fma_(c02, v[0], fma_(c12, v[1], mul_(c22, v[2]))), inv);
}

// ---- the DLT rows of one view (MatrixTriangulator.cpp:16-49), shared by every DLT kernel and the host's tables ----
// One row (a, b) into the normal equations.
template <typename T>
__host__ __device__ __forceinline__ void acc_row(T a0, T a1, T a2, T b, T (&M)[6], T (&v)[3]) {
  M[0] = fma_(a0, a0, M[0]); M[1] = fma_(a0, a1, M[1]); M[2] = fma_(a0, a2, M[2]); v[0] = fma_(a0, b, v[0]);
  M[3] = fma_(a1, a1, M[3]); M[4] = fma_(a1, a2, M[4]); v[1] = fma_(a1, b, v[1]);
  M[5] = fma_(a2, a2, M[5]); v[2] = fma_(a2, b, v[2]);
}

// How an absent view is kept out of the sums.
//   MASK_TABLE      FP32: accumulate it at the canonical pixel (0, 0), subtract its constant contribution from a table afterwards
//                   (DltRig::absent); a caller that passes valid views only (the robust solve) needs nothing else
//   MASK_SELECT_HI  FP64: clear only the HIGH word of the three coefficients -- what is left is a denormal below 2^-1042
//                   whose products with the other coefficients (< 2^40) vanish against the sums; half the selects
// Measured on the FP64 kernel (100 M frames, profiles/r2_dlt_variants.log): table 1.96 ms, select of both words 1.90 ms,
// high-word select 1.86 ms -- the kernel is bound by the FP64 pipe (time follows the count of FP64 instructions, 2.9 cycles
// each), so the table's 18 extra DADD per frame pair cost more than the selects it removes from the other pipes.
enum { MASK_TABLE = 0, MASK_SELECT_HI = 1 };
__device__ __forceinline__ double mask_coeff(double a, bool ok) { return __hiloint2double(ok ? __double2hiint(a) : 0, __double2loint(a)); }

// One view's two rows a = P[r,0:3] - u P[2,0:3], b = u P[2,3] - P[r,3] (u = x, then y; pixel relative to the rig's
// pixel origin) into the normal equations.
template <int MASKING, typename T>
__host__ __device__ __forceinline__ void dlt_view(const T (&P)[12], T x, T y, bool valid, T (&M)[6], T (&v)[3]) {
  if constexpr (MASKING == MASK_TABLE) { x = valid ? x : T(0); y = valid ? y : T(0); }  // the canonical pixel
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int r = 0; r < 2; r++) {
    const T u = r == 0 ? x : y;
    T a0 = fma_(-u, P[8], P[4 * r]), a1 = fma_(-u, P[9], P[4 * r + 1]), a2 = fma_(-u, P[10], P[4 * r + 2]);
    const T b = fma_(u, P[11], -P[4 * r + 3]);
    if constexpr (MASKING == MASK_SELECT_HI) { a0 = mask_coeff(a0, valid); a1 = mask_coeff(a1, valid); a2 = mask_coeff(a2, valid); }
    acc_row<T>(a0, a1, a2, b, M, v);
  }
}

// Camera loop over a compile-time class: NC > 0 unrolls NC cameras (static camera indices: the constants are constant-bank
// operands) and predicates off those >= n; NC = 0 is a rolled loop.  n is the same for the whole grid and every thread walks
// the same cameras in the same order -- a frame's absent views are predicated off by f, not skipped -- so the rig index is
// warp-uniform (a divergent index would serialise the constant-bank reads).
template <int NC, class F>
__device__ __forceinline__ void for_cams(int n, F&& f) {
  if constexpr (NC > 0) {
#pragma unroll
    for (int c = 0; c < NC; c++)
      if (c < n) f(c);
  } else {
#pragma unroll 1
    for (int c = 0; c < n; c++) f(c);
  }
}

}  // namespace tri

// ---- launchers (defined in the .cu files, called from tri_api.cu) ----
namespace tri {

struct LaunchCtx {
  cudaStream_t stream;
  int sm_count;
  unsigned long long* d_first_bad;  // latched index of the first frame with < 2 views
  int64_t frame_base;               // global index of frame 0 of this launch (chunked host path)
  int64_t* launches;
};

cudaError_t launch_ray_fold(const LaunchCtx& ctx, bool lm, bool f32, int pixfmt, const RayFold<double>& r64,
                            const RayFold<float>& r32, const void* d_xy, int n_use, int64_t n_frames,
                            int64_t cam_stride, const BatchOut& out);
cudaError_t launch_ray_reference(const LaunchCtx& ctx, int pixfmt, const RayRig& rig, const void* d_xy, int n_use,
                                 int64_t n_frames, int64_t cam_stride, const BatchOut& out);

cudaError_t launch_dlt(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64,
                       const DltRig<float>& rig32, const void* d_xy, int n_use, int64_t n_frames,
                       int64_t cam_stride, const BatchOut& out);

// two-view consensus + inlier refit (tri_robust.cu); out.mask = the inlier set, out.err = RMS reprojection error in pixels
cudaError_t launch_robust(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64, const DltRig<float>& rig32,
                          double max_reproj_px, const void* d_xy, int n_use, int64_t n_frames, int64_t cam_stride,
                          const BatchOut& out);

// forward projection (tri_project.cu): points [n][3] (exactly one of d_xyz_f32 / d_xyz_f64) to the pixel rows of all
// n_cams cameras in format `pixfmt` (d_xy may be null) and the visibility masks (d_mask may be null)
cudaError_t launch_project(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64, const DltRig<float>& rig32,
                           const tri_camera* cams, int n_cams, const float* d_xyz_f32, const double* d_xyz_f64, int64_t n_points,
                           void* d_xy, int64_t cam_stride, uint32_t* d_mask);

}  // namespace tri
