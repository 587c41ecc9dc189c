// tri_robust.cu -- outlier-robust batched triangulation (tri_triangulate_points_robust*) for sm_100a.
//
// Per frame, over the valid views V (same sentinel test and camera rows as the plain DLT):
//   1. every pair i < j of V gives a hypothesis X_ij, the DLT of the two views (4 rows rebuilt from the pixels and the
//      constant P, the plain path's normal equations and adjugate solve); usable only if its projective depth
//      w_c(X) = P_c[8..10].X + P_c[11] is > 0 on both cameras;
//   2. its inliers are the views c of V with w_c(X_ij) > 0 and pixel reprojection error r_c <= tau;
//   3. the best hypothesis has the most inliers (at least 2), then the smallest sum of r_c^2 over them, then comes first
//      in (i, j) order;
//   4. the output is the DLT over the winning inlier set I (only those views accumulated -- no absent-view table, whose
//      subtraction loses accuracy when most views are excluded), mask = I, err = sqrt(mean r_c^2) over I in pixels.
// No qualifying hypothesis: (0,0,0), mask 0, err NaN.  Fewer than 2 valid views: exactly the plain call's too-few frame.
//
// Two kernels:
//   * RobustTile, a tile of the streaming skeleton (tri_pipe.cuh) for 2..8 cameras with float2 / ushort2 pixels: the
//     per-thread cp.async ring holds the frame's pixels in shared memory and the solve reads them from there camera by
//     camera (LAZY feeder), one frame per thread;
//   * robust_kernel for everything else (9..32 cameras, double2 pixels, tails, unaligned rows): one frame per thread,
//     pixels read through the read-only cache as the solve needs them (a hypothesis pairs views of any two cameras, so
//     the camera-chunked ring cannot serve it).
// FP64 runs on the cameraPerspectiveMatrix as is; FP32 on the rig's centred form (DltRig<float>: pixel origin at the
// image centre, world origin at the rig centre) -- the same projective depth and the same pixel residuals.
#include <math.h>

#include "tri_pipe.cuh"

namespace tri {

template <typename T>
struct __align__(16) RobustRig {
  DltRig<T> d;
  T tau2;  // max_reproj_px^2: r <= tau  <=>  r^2 <= tau^2
};

// one view's two DLT rows into the normal equations (the plain path's fma sequence, DltPolicy::add)
template <typename T>
__device__ __forceinline__ void robust_add(const T (&P)[12], T x, T y, T (&M)[6], T (&v)[3]) {
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const T u = r == 0 ? x : y;
    const T a0 = fma_(-u, P[8], P[4 * r]), a1 = fma_(-u, P[9], P[4 * r + 1]), a2 = fma_(-u, P[10], P[4 * r + 2]);
    const T b = fma_(u, P[11], -P[4 * r + 3]);
    M[0] = fma_(a0, a0, M[0]); M[1] = fma_(a0, a1, M[1]); M[2] = fma_(a0, a2, M[2]); v[0] = fma_(a0, b, v[0]);
    M[3] = fma_(a1, a1, M[3]); M[4] = fma_(a1, a2, M[4]); v[1] = fma_(a1, b, v[1]);
    M[5] = fma_(a2, a2, M[5]); v[2] = fma_(a2, b, v[2]);
  }
}

// projective depth w and squared pixel reprojection error r2 of X on a camera, pixel (x, y)
template <typename T>
__device__ __forceinline__ void robust_project(const T (&P)[12], const T (&X)[3], T x, T y, T& w, T& r2) {
  w = fma_(P[8], X[0], fma_(P[9], X[1], fma_(P[10], X[2], P[11])));
  const T iw = rcp_(w);
  const T du = fma_(fma_(P[0], X[0], fma_(P[1], X[1], fma_(P[2], X[2], P[3]))), iw, -x);
  const T dv = fma_(fma_(P[4], X[0], fma_(P[5], X[1], fma_(P[6], X[2], P[7]))), iw, -y);
  r2 = fma_(du, du, mul_(dv, dv));
}

// Camera loop of the consensus solve: unrolled over a compile-time count (static camera indices: the constants are
// constant-bank operands), a plain loop otherwise.  Every thread of a warp walks the same cameras in the same order --
// a frame's absent views are predicated off, not skipped -- so the rig index is warp-uniform (a divergent index would
// serialise the constant-bank reads), and a warp costs what its busiest frame costs either way.
template <int NC, class F>
__device__ __forceinline__ void for_cams(int c0, int n, F&& f) {
  if constexpr (NC > 0) {
#pragma unroll
    for (int c = 0; c < NC; c++)
      if (c >= c0) f(c);
  } else {
#pragma unroll 1
    for (int c = c0; c < n; c++) f(c);
  }
}

// The consensus solve of one frame.  NC > 0: compile-time camera count; NC = 0: n cameras at run time.
// pix(c, x, y) -> validity of camera c, (x, y) relative to the rig's pixel origin.  views = the number of valid views
// (the too-few test of the plain path).
template <typename T, int NC, class Pix>
__device__ __forceinline__ void robust_frame(const RobustRig<T>& rig, int n, const Pix& pix, T (&X)[3], uint32_t& mask,
                                             double& err, int& views) {
  const DltRig<T>& d = rig.d;
  if constexpr (NC > 0) n = NC;
  uint32_t V = 0;
  for_cams<NC>(0, n, [&](int c) {
    T x, y;
    V |= (pix(c, x, y) ? 1u : 0u) << c;
  });
  views = __popc(V);
  X[0] = X[1] = X[2] = 0;
  err = 0;
  mask = V;
  if (views < 2) return;  // the plain path's too-few frame

  int best_n = 1;
  T best_s = 0;
  uint32_t best_I = 0;
#pragma unroll 1
  for (int i = 0; i < n - 1; i++) {
    T xi, yi;
    if (!pix(i, xi, yi)) continue;
#pragma unroll 1
    for (int j = i + 1; j < n; j++) {
      T xj, yj;
      if (!pix(j, xj, yj)) continue;
      T M[6] = {0, 0, 0, 0, 0, 0}, v[3] = {0, 0, 0}, H[3];
      robust_add<T>(d.P[i], xi, yi, M, v);
      robust_add<T>(d.P[j], xj, yj, M, v);
      solve_sym3<T>(M, v, H);
      uint32_t I = 0;
      T s = 0;
      bool front = true;
      for_cams<NC>(0, n, [&](int c) {
        T x, y, w, r2;
        if (!pix(c, x, y)) return;
        robust_project<T>(d.P[c], H, x, y, w, r2);
        if (c == i || c == j) front = front && w > 0;
        if (w > 0 && r2 <= rig.tau2) { I |= 1u << c; s += r2; }
      });
      const int k = __popc(I);
      if (front && k >= 2 && (k > best_n || (k == best_n && s < best_s))) { best_n = k; best_s = s; best_I = I; }
    }
  }
  mask = best_I;
  if (!best_I) { err = __longlong_as_double(0x7ff8000000000000ll); return; }  // no consensus: NaN

  // the refit: the DLT over the inliers only, in camera order
  T M[6] = {0, 0, 0, 0, 0, 0}, v[3] = {0, 0, 0};
  for_cams<NC>(0, n, [&](int c) {
    T x, y;
    pix(c, x, y);
    if (best_I >> c & 1) robust_add<T>(d.P[c], x, y, M, v);
  });
  solve_sym3<T>(M, v, X);
  T s = 0;
  for_cams<NC>(0, n, [&](int c) {
    T x, y, w, r2;
    pix(c, x, y);
    robust_project<T>(d.P[c], X, x, y, w, r2);
    if (best_I >> c & 1) s += r2;
  });
  err = sqrt((double)s / (double)best_n);
  X[0] += d.origin[0]; X[1] += d.origin[1]; X[2] += d.origin[2];
}

// ---- 2..8 cameras, float2 / ushort2 pixels: a tile of the streaming skeleton ----
template <typename T>
struct RobustTile {
  static constexpr int FPT = 1;
  using Rig = RobustRig<T>;
  using Real = T;
  static constexpr bool MASK_IS_VALIDITY = false;  // mask = the inlier set; `iters` carries the valid-view count
  template <int NC, int PIX, bool WIDE, class RS>
  static __device__ __forceinline__ void run(const Rig& rig, const RS& raw, int, T (&X)[1][3],
                                             uint32_t (&mask)[1], double (&err)[1], int (&iters)[1]) {
    auto pix = [&](int c, T& x, T& y) -> bool {
      const Views<T, PIX, 1> q = decode<T, PIX, 1>(raw[c]);
      x = q.x[0] - rig.d.pix0[c][0];
      y = q.y[0] - rig.d.pix0[c][1];
      return q.v[0];
    };
    // the camera loops stay rolled: unrolled over NC the compiler keeps every camera's constants and pixels live across
    // the pair loop (FP64 at 8 cameras: 255 registers and spills, against 64 registers rolled)
    robust_frame<T, 0>(rig, NC, pix, X[0], mask[0], err[0], iters[0]);
  }
};

// ---- everything else: one frame per thread, pixels through the read-only cache ----
template <typename T, int PIX>
__device__ __forceinline__ bool robust_load(const char* xy, int64_t row_bytes, int c, int64_t f, T& x, T& y) {
  const char* row = xy + c * row_bytes;
  if constexpr (PIX == PIX_F32) {
    const float2 q = __ldg(reinterpret_cast<const float2*>(row) + f);
    x = (T)q.x; y = (T)q.y;
    return pix_valid(q.x, q.y);
  } else if constexpr (PIX == PIX_F64) {
    const double2 q = __ldg(reinterpret_cast<const double2*>(row) + f);
    x = (T)q.x; y = (T)q.y;
    return pix_valid(q.x, q.y);
  } else {
    const unsigned q = __ldg(reinterpret_cast<const unsigned*>(row) + f);
    x = (T)(q & 0xffffu); y = (T)(q >> 16);
    return q != 0xffffffffu;
  }
}

template <typename T, int PIX>
__global__ void __launch_bounds__(BATCH_THREADS)
robust_kernel(const __grid_constant__ RobustRig<T> rig, const char* __restrict__ xy, int64_t row_bytes, int64_t n_frames, int n_use,
              BatchOut out, unsigned long long* first_bad, int64_t frame_base) {
  const int64_t f = (int64_t)blockIdx.x * BATCH_THREADS + threadIdx.x;
  if (f >= n_frames) return;
  auto pix = [&](int c, T& x, T& y) -> bool {
    const bool ok = robust_load<T, PIX>(xy, row_bytes, c, f, x, y);
    x -= rig.d.pix0[c][0];
    y -= rig.d.pix0[c][1];
    return ok;
  };
  T X[3];
  uint32_t mask;
  double err;
  int views;
  robust_frame<T, 0>(rig, n_use, pix, X, mask, err, views);
  if (views < 2) atomicMin(first_bad, (unsigned long long)(frame_base + f));
  if (out.xyz_f32) { float* o = out.xyz_f32 + 3 * f; o[0] = (float)X[0]; o[1] = (float)X[1]; o[2] = (float)X[2]; }
  if (out.xyz_f64) { double* o = out.xyz_f64 + 3 * f; o[0] = X[0]; o[1] = X[1]; o[2] = X[2]; }
  if (out.mask) out.mask[f] = mask;
  if (out.err) out.err[f] = err;
}

template <typename T, int PIX>
static cudaError_t robust_streamed(const LaunchCtx& ctx, const RobustRig<T>& rig, const void* d_xy, int n_use, int64_t n_frames,
                                   int64_t cam_stride, const BatchOut& out) {
  int64_t covered = 0;
  if constexpr (PIX != PIX_F64) {
    const cudaError_t err = launch_stream<RobustTile<T>, PIX, 2, 2, true>(ctx, rig, d_xy, n_use, n_frames, cam_stride, out, 0, &covered);
    if (err != cudaSuccess || covered == n_frames) return err;
  }
  const int64_t rest = n_frames - covered;
  const unsigned grid = (unsigned)((rest + BATCH_THREADS - 1) / BATCH_THREADS);
  robust_kernel<T, PIX><<<grid, BATCH_THREADS, 0, ctx.stream>>>(rig, static_cast<const char*>(d_xy) + covered * pix_bytes(PIX),
                                                                 cam_stride * pix_bytes(PIX), rest, n_use, advance(out, covered),
                                                                 ctx.d_first_bad, ctx.frame_base + covered);
  ++*ctx.launches;
  return cudaGetLastError();
}

cudaError_t launch_robust(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64, const DltRig<float>& rig32,
                          double max_reproj_px, const void* d_xy, int n_use, int64_t n_frames, int64_t cam_stride,
                          const BatchOut& out) {
  if (n_frames <= 0) return cudaSuccess;
  if (f32) {
    RobustRig<float> r;
    r.d = rig32;
    r.d.n_use = n_use;
    r.tau2 = (float)(max_reproj_px * max_reproj_px);
    if (pixfmt == PIX_F32) return robust_streamed<float, PIX_F32>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
    if (pixfmt == PIX_F64) return robust_streamed<float, PIX_F64>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
    return robust_streamed<float, PIX_U16>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
  }
  RobustRig<double> r;
  r.d = rig64;
  r.d.n_use = n_use;
  r.tau2 = max_reproj_px * max_reproj_px;
  if (pixfmt == PIX_F32) return robust_streamed<double, PIX_F32>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
  if (pixfmt == PIX_F64) return robust_streamed<double, PIX_F64>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
  return robust_streamed<double, PIX_U16>(ctx, r, d_xy, n_use, n_frames, cam_stride, out);
}

}  // namespace tri
