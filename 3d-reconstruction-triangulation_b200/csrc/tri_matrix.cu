// tri_matrix.cu -- kernel 1: batched MatrixTriangulator::triangulatePoints for sm_100a.
//
// Reference semantics (src/MatrixTriangulator.cpp): per frame, every camera whose pixel is not the
// (-1,-1) sentinel (:86-87) contributes the two rows
//     P[0,0:3] - x P[2,0:3] | x P[2,3] - P[0,3]        (:16-27, :42-45)
//     P[1,0:3] - y P[2,0:3] | y P[2,3] - P[1,3]        (:29-40, :46-49)
// of a 2n x 3 system A X = b solved by X = pinv_SVD(A) b (:53-54); the reported error is
// sqrt(|A X - b|^2 / 2n) (:55-59).  One thread owns two frames (tri_batch.cuh), accumulates the
// 3x3 normal matrix A^T A and A^T b in registers -- 26 FMA per view with the camera constants read
// from the constant bank -- and solves by the adjugate.  The full-rank pseudo-inverse solution IS
// the normal-equation solution; cond(A) <= ~5 on real rigs so nothing is lost (SURVEY.md F1).
// HBM traffic per frame: 8 B x n_cams in, 12 B out.
//
// Absent views (round 2, FP32; FP64: MASK_SELECT_HI, tri_common.cuh): no select, predicate or branch sits in the FMA
// chain any more.  An absent view's pixel is replaced by a canonical one (the pixel origin of the rig) BEFORE
// the conversion, every camera is accumulated unconditionally, and what the absent cameras added -- a constant
// per camera at the canonical pixel -- is taken back after the camera loop from a 256-row table indexed by the
// complement of the frame's validity mask (one row per group of 8 cameras; built on the host with the same fma
// sequence, tri_api.cu).
// Round 1 zeroed the three row coefficients with selects: 192 FSEL per pair of frames in the FP64 kernel, in the
// dependency chain between the row FMAs and the accumulation FMAs (profiles/ncu_r1g.md: issue 66 %, FP64 pipe
// 67 %, both short of their limits because each starved the other).
#include "tri_pipe.cuh"

namespace tri {

// one camera's 3x4 matrix as 16-byte vector loads
__device__ __forceinline__ void load12(const double (&src)[12], double (&P)[12]) {
  const double2* v = reinterpret_cast<const double2*>(src);
#pragma unroll
  for (int k = 0; k < 6; k++) { const double2 q = v[k]; P[2 * k] = q.x; P[2 * k + 1] = q.y; }
}
__device__ __forceinline__ void load12(const float (&src)[12], float (&P)[12]) {
  const float4* v = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int k = 0; k < 3; k++) { const float4 q = v[k]; P[4 * k] = q.x; P[4 * k + 1] = q.y; P[4 * k + 2] = q.z; P[4 * k + 3] = q.w; }
}

// the absent-view table row of `mask` (validity bits of the cameras [8g, 8g+8) at bits 8g..): 10 T per row
template <typename T>
__device__ __forceinline__ const T* absent_row(const DltRig<T>& rig, uint32_t mask, int group, int n_in_group) {
  const uint32_t absent = ~(mask >> (8 * group)) & ((1u << n_in_group) - 1u);
  return rig.absent + ((size_t)group * 256 + absent) * DLT_TABLE_ROW;
}
__device__ __forceinline__ void sub_row(const float* row, float (&M)[6], float (&v)[3]) {
  const float4* r = reinterpret_cast<const float4*>(row);
  const float4 t0 = __ldg(r), t1 = __ldg(r + 1), t2 = __ldg(r + 2);
  M[0] -= t0.x; M[1] -= t0.y; M[2] -= t0.z; M[3] -= t0.w; M[4] -= t1.x; M[5] -= t1.y; v[0] -= t1.z; v[1] -= t1.w; v[2] -= t2.x;
}

// |A X - b|^2 of one view's two rows (MatrixTriangulator.cpp:55-58), pixel relative to the rig's pixel origin
template <typename T>
__device__ __forceinline__ T dlt_residual(const T (&P)[12], T x, T y, const T (&X)[3]) {
  const T e0 = fma_(fma_(-x, P[8], P[0]), X[0], fma_(fma_(-x, P[9], P[1]), X[1], fma_(fma_(-x, P[10], P[2]), X[2], -fma_(x, P[11], -P[3]))));
  const T e1 = fma_(fma_(-y, P[8], P[4]), X[0], fma_(fma_(-y, P[9], P[5]), X[1], fma_(fma_(-y, P[10], P[6]), X[2], -fma_(y, P[11], -P[7]))));
  return fma_(e0, e0, mul_(e1, e1));
}

template <typename T_, bool CENTRED, int MASKING>
struct DltPolicy {
  using T = T_;
  using Rig = DltRig<T>;
  // more than 8 cameras stay on the generic batch_kernel: the chunked pipeline measured slower for the DLT
  // (32 cameras x 20 M frames: FP64 2.40 ms at one frame per thread, 2.03 ms at two, vs 1.84 ms; FP32 1.29 vs 0.99 ms)
  static constexpr bool CHUNKED = false;
  static constexpr int CHUNK_FPT = 2;
  struct Acc {
    T M[6] = {0, 0, 0, 0, 0, 0};
    T v[3] = {0, 0, 0};
  };
  // (x, y) relative to the rig's pixel origin
  static __device__ __forceinline__ void add(const Rig& rig, int c, T x, T y, bool valid, Acc& a) {
    T P[12];
    load12(rig.P[c], P);
    if constexpr (CENTRED) { x -= rig.pix0[c][0]; y -= rig.pix0[c][1]; }
    dlt_view<MASKING>(P, x, y, valid, a.M, a.v);
  }
  static __device__ __forceinline__ void add_chunk(const Rig& rig, int c, T x, T y, bool valid, Acc& a) { add(rig, c, x, y, valid, a); }
  // take back what the absent cameras added (group g = cameras 8g .. 8g+7, in order), then the adjugate solve
  static __device__ __forceinline__ void solve(const Rig& rig, const Acc& a, uint32_t mask, int, T (&X)[3], int, int&) {
    Acc r = a;
    if constexpr (MASKING == MASK_TABLE)
      for (int g = 0; 8 * g < rig.n_use; g++) sub_row(absent_row<T>(rig, mask, g, min(8, rig.n_use - 8 * g)), r.M, r.v);
    solve_sym3<T>(r.M, r.v, X);
  }
  // |A X - b|^2 contribution of one camera (MatrixTriangulator.cpp:55-58)
  static __device__ __forceinline__ T residual(const Rig& rig, int c, T x, T y, const T (&X)[3]) {
    const T(&P)[12] = rig.P[c];
    if constexpr (CENTRED) { x -= rig.pix0[c][0]; y -= rig.pix0[c][1]; }
    return dlt_residual<T>(P, x, y, X);
  }
  static __device__ __forceinline__ double error(T sum, int n) { return sqrt((double)sum / (double)(2 * n)); }
  static __device__ __forceinline__ void to_world(const Rig& rig, T (&X)[3]) {
    if constexpr (CENTRED) { X[0] += rig.origin[0]; X[1] += rig.origin[1]; X[2] += rig.origin[2]; }
  }
};

// ---- FP64 streaming tile: two frames per thread, 2..8 cameras ----
// Same operation order as DltPolicy<double> (which serves tails, unaligned rows and more than 8 cameras), so the
// points are bit-identical whichever kernel a frame lands in.
struct DltTile64 {
  static constexpr int FPT = 2;
  using S = DltPolicy<double, false, MASK_SELECT_HI>;
  using Rig = DltRig<double>;
  using Real = double;
  template <int NC, int PIX, bool WIDE, class RS>
  static __device__ __forceinline__ void run(const Rig& rig, const RS& raw, int, double (&X)[2][3], uint32_t (&mask)[2],
                                             double (&err)[2], int (&iters)[2]) {
    typename S::Acc acc[2];
    mask[0] = mask[1] = 0;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      double P[12];
      load12(rig.P[c], P);
      const Views<double, PIX, 2> q = decode<double, PIX, 2>(raw[c]);
#pragma unroll
      for (int j = 0; j < 2; j++) {
        mask[j] |= (q.v[j] ? 1u : 0u) << c;
        dlt_view<MASK_SELECT_HI>(P, q.x[j], q.y[j], q.v[j], acc[j].M, acc[j].v);
      }
    }
#pragma unroll
    for (int j = 0; j < 2; j++) {
      X[j][0] = X[j][1] = X[j][2] = 0;
      err[j] = 0;
      iters[j] = 0;
      const int n = __popc(mask[j]);
      if (n >= 2) {
        solve_sym3<double>(acc[j].M, acc[j].v, X[j]);
        if constexpr (WIDE) {
          double e = 0;
#pragma unroll
          for (int c = 0; c < NC; c++) {
            const Views<double, PIX, 2> q = decode<double, PIX, 2>(raw[c]);
            if (q.v[j]) e += S::residual(rig, c, q.x[j], q.y[j], X[j]);
          }
          err[j] = S::error(e, n);
        }
      }
    }
  }
};

// ---- FP32 main path: packed-pair SIMD (FFMA2 / FMUL2 / FADD2, new on sm_100) ----
// One thread owns frames (2g, 2g+1) as the two halves of a float2; every multiply-add of the
// accumulation is one FFMA2, so the solve needs half the issue slots of the scalar form (which was
// issue-bound: profiles/r1a, 80 % issue-active).  Same operation order as the scalar DltPolicy<float>
// path (which serves the tails), so the points are bit-identical.  Rig constants are pre-duplicated /
// pre-negated float2 so the operands come from the uniform datapath.
struct __align__(16) DltRigX2 {
  float2 A[TRI_MAX_CAMS][8];   // P0 P1 P2 -P3 | P4 P5 P6 -P7   (addends of the x row, the y row)
  float2 N[TRI_MAX_CAMS][4];   // -P8 -P9 -P10 P11              (multiplicands)
  float2 npix0[TRI_MAX_CAMS][2];
  float origin[3];
  const float* absent;  // DltRig<float>::absent
};

struct DltX2Tile {
  static constexpr int FPT = 2;
  using Rig = DltRigX2;
  using Real = float;
  template <int NC, int PIX, bool WIDE, class RS>
  static __device__ __forceinline__ void run(const Rig& rig, const RS& raw, int, float (&X)[2][3], uint32_t (&mask)[2],
                                             double (&err)[2], int (&iters)[2]) {
    float2 M[6] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}, v[3] = {{0, 0}, {0, 0}, {0, 0}};
    uint32_t mask0 = 0, mask1 = 0;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const Views<float, PIX, 2> q = decode<float, PIX, 2>(raw[c]);
      mask0 |= (q.v[0] ? 1u : 0u) << c;
      mask1 |= (q.v[1] ? 1u : 0u) << c;
      float2 K[14];  // this camera's constants
      const float4* kv = reinterpret_cast<const float4*>(rig.A[c]);
#pragma unroll
      for (int k = 0; k < 4; k++) { const float4 t = kv[k]; K[2 * k] = make_float2(t.x, t.y); K[2 * k + 1] = make_float2(t.z, t.w); }
      const float4* nv = reinterpret_cast<const float4*>(rig.N[c]);
#pragma unroll
      for (int k = 0; k < 2; k++) { const float4 t = nv[k]; K[8 + 2 * k] = make_float2(t.x, t.y); K[9 + 2 * k] = make_float2(t.z, t.w); }
      const float4 t = *reinterpret_cast<const float4*>(rig.npix0[c]);
      K[12] = make_float2(t.x, t.y); K[13] = make_float2(t.z, t.w);
      float2 x = __fadd2_rn(make_float2(q.x[0], q.x[1]), K[12]);
      float2 y = __fadd2_rn(make_float2(q.y[0], q.y[1]), K[13]);
      x = make_float2(q.v[0] ? x.x : 0.f, q.v[1] ? x.y : 0.f);  // absent view: the canonical pixel (the rig's pixel origin)
      y = make_float2(q.v[0] ? y.x : 0.f, q.v[1] ? y.y : 0.f);
#pragma unroll
      for (int r = 0; r < 2; r++) {
        const float2 u = r == 0 ? x : y;
        const float2 a0 = fma2(u, K[8], K[4 * r]), a1 = fma2(u, K[9], K[4 * r + 1]),
                     a2 = fma2(u, K[10], K[4 * r + 2]), b = fma2(u, K[11], K[4 * r + 3]);
        M[0] = fma2(a0, a0, M[0]); M[1] = fma2(a0, a1, M[1]); M[2] = fma2(a0, a2, M[2]); v[0] = fma2(a0, b, v[0]);
        M[3] = fma2(a1, a1, M[3]); M[4] = fma2(a1, a2, M[4]); v[1] = fma2(a1, b, v[1]);
        M[5] = fma2(a2, a2, M[5]); v[2] = fma2(a2, b, v[2]);
      }
    }
    {  // what the absent cameras added, one table row per frame
      const float4* r0 = reinterpret_cast<const float4*>(rig.absent + (size_t)(~mask0 & ((1u << NC) - 1u)) * DLT_TABLE_ROW);
      const float4* r1 = reinterpret_cast<const float4*>(rig.absent + (size_t)(~mask1 & ((1u << NC) - 1u)) * DLT_TABLE_ROW);
      const float4 s0 = __ldg(r0), s1 = __ldg(r0 + 1), s2 = __ldg(r0 + 2), t0 = __ldg(r1), t1 = __ldg(r1 + 1), t2 = __ldg(r1 + 2);
      M[0].x -= s0.x; M[1].x -= s0.y; M[2].x -= s0.z; M[3].x -= s0.w; M[4].x -= s1.x; M[5].x -= s1.y; v[0].x -= s1.z; v[1].x -= s1.w; v[2].x -= s2.x;
      M[0].y -= t0.x; M[1].y -= t0.y; M[2].y -= t0.z; M[3].y -= t0.w; M[4].y -= t1.x; M[5].y -= t1.y; v[0].y -= t1.z; v[1].y -= t1.w; v[2].y -= t2.x;
    }
    float2 X0, X1, X2;
    solve_sym3_x2(M, v, X0, X1, X2);
    const bool ok0 = __popc(mask0) >= 2, ok1 = __popc(mask1) >= 2;
    float Xr[2][3] = {{X0.x, X1.x, X2.x}, {X0.y, X1.y, X2.y}};
    mask[0] = mask0; mask[1] = mask1;
#pragma unroll
    for (int j = 0; j < 2; j++) {
      err[j] = 0;
      iters[j] = 0;
      const bool ok = j == 0 ? ok0 : ok1;
      if constexpr (WIDE) {
        if (ok) {  // the `error` of triangulatePoint in the tile's (centred) coordinates, as DltPolicy<float> computes it
          float e = 0;
#pragma unroll
          for (int c = 0; c < NC; c++) {
            const Views<float, PIX, 2> q = decode<float, PIX, 2>(raw[c]);
            if (q.v[j]) {  // the rig's P back from the .x halves (negation is exact)
              const float2 *A = rig.A[c], *N = rig.N[c];
              const float P[12] = {A[0].x, A[1].x, A[2].x, -A[3].x, A[4].x, A[5].x, A[6].x, -A[7].x, -N[0].x, -N[1].x, -N[2].x, N[3].x};
              e += dlt_residual<float>(P, q.x[j] + rig.npix0[c][0].x, q.y[j] + rig.npix0[c][1].x, Xr[j]);
            }
          }
          err[j] = DltPolicy<float, true, MASK_TABLE>::error(e, __popc(j == 0 ? mask0 : mask1));
        }
      }
      X[j][0] = ok ? Xr[j][0] + rig.origin[0] : 0.f; X[j][1] = ok ? Xr[j][1] + rig.origin[1] : 0.f; X[j][2] = ok ? Xr[j][2] + rig.origin[2] : 0.f;
    }
  }
};


static DltRigX2 make_x2(const DltRig<float>& r) {
  DltRigX2 x;
  for (int c = 0; c < TRI_MAX_CAMS; c++) {
    const float* P = r.P[c];
    const float A[8] = {P[0], P[1], P[2], -P[3], P[4], P[5], P[6], -P[7]};
    const float N[4] = {-P[8], -P[9], -P[10], P[11]};
    for (int k = 0; k < 8; k++) x.A[c][k] = make_float2(A[k], A[k]);
    for (int k = 0; k < 4; k++) x.N[c][k] = make_float2(N[k], N[k]);
    for (int k = 0; k < 2; k++) x.npix0[c][k] = make_float2(-r.pix0[c][k], -r.pix0[c][k]);
  }
  for (int k = 0; k < 3; k++) x.origin[k] = r.origin[k];
  x.absent = r.absent;
  return x;
}

cudaError_t launch_dlt(const LaunchCtx& ctx, bool f32, int pixfmt, const DltRig<double>& rig64_,
                       const DltRig<float>& rig32_, const void* d_xy, int n_use, int64_t n_frames,
                       int64_t cam_stride, const BatchOut& out) {
  if (n_frames <= 0) return cudaSuccess;
  using P32 = DltPolicy<float, true, MASK_TABLE>;
  using P64 = DltPolicy<double, false, MASK_SELECT_HI>;
  if (f32) {
    DltRig<float> rig32 = rig32_;
    rig32.n_use = n_use;
    const DltRigX2 x2 = make_x2(rig32);
    // float2 pixels: read from the slot camera by camera instead of pulled into registers on arrival -- fewer live registers,
    // 1.269 -> 1.224 ms per 100 M frames (profiles/r2_dlt_variants.log); the other solves measured slower that way
    if (pixfmt == PIX_F32) return launch_streamed<DltX2Tile, P32, PIX_F32, 2, 2, 3, true>(ctx, x2, rig32, d_xy, n_use, n_frames, cam_stride, out, 0);
    if (pixfmt == PIX_F64) return launch_streamed<DltX2Tile, P32, PIX_F64, 2, 2, 3>(ctx, x2, rig32, d_xy, n_use, n_frames, cam_stride, out, 0);
    return launch_streamed<DltX2Tile, P32, PIX_U16, 2, 2, 3>(ctx, x2, rig32, d_xy, n_use, n_frames, cam_stride, out, 0);
  }
  DltRig<double> rig64 = rig64_;
  rig64.n_use = n_use;
  if (pixfmt == PIX_F32) return launch_streamed<DltTile64, P64, PIX_F32, 2, 2, 2>(ctx, rig64, rig64, d_xy, n_use, n_frames, cam_stride, out, 0);
  if (pixfmt == PIX_F64) return launch_batch_policy<P64, PIX_F64, 1, 3>(ctx, rig64, d_xy, n_use, n_frames, cam_stride, out, 0);
  return launch_streamed<DltTile64, P64, PIX_U16, 2, 3, 2>(ctx, rig64, rig64, d_xy, n_use, n_frames, cam_stride, out, 0);
}

}  // namespace tri
