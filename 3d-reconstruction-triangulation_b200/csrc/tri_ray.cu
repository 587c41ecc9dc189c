// tri_ray.cu -- kernel 2: fused pixel-ray generation + quaternion rotation + nearest-point-to-rays
// solve (RayTriangulator::triangulatePoints, src/RayTriangulator.cpp:51-107) for sm_100a.
//
// Reference: ray_i = (camera position, q (0, normalise(v_i)) q*) with v_i the pixel ray of
// Triangulator.cpp:27-44; the point minimises S(p) = sum_i r_i(p)^2, r_i = |dir_i x (p - o_i)|
// (Triangulator.cpp:3-9, RayTriangulator.cpp:16-26), found by cv::LMSolver on the n scalar residuals
// r_i with a central-difference Jacobian.  S is QUADRATIC in p:
//     S(p) = p^T M p - 2 c^T p + k,  M = sum_i (|d_i|^2 I - d_i d_i^T),  c = sum_i M_i o_i.
// The fused kernel therefore runs Levenberg-Marquardt on the 3n residual components
// e_i = dir_i x (p - o_i), whose Jacobian [dir_i]_x is analytic and exact: J^T J = M, J^T e = M p - c.
// Same objective, same minimiser, same cv::LMSolver damping schedule -- but M, c, k are accumulated
// once per frame in registers (~40 FMA per view, rig constants from the constant bank) and each LM
// iteration is O(1).  (The scalar-residual form the reference uses has a rank-2 J^T J for two views,
// which is why its LM crawls there, SURVEY.md F5.)  opt bit 0: 1 = LM loop, 0 = closed form
// p = M^-1 c (one exact Newton step).  The trajectory-exact emulation of the reference's LM lives in
// tri_ray_ref.cu.
#include <float.h>

#include "tri_pipe.cuh"

namespace tri {

// a rig constant of one camera: the scalar of RayFold, or the low half of RayRigX2's pre-duplicated pair
__device__ __forceinline__ float lo(float v) { return v; }
__device__ __forceinline__ double lo(double v) { return v; }
__device__ __forceinline__ float lo(float2 v) { return v.x; }

template <typename T_>
struct RayPolicy {
  using T = T_;
  using Rig = RayFold<T>;
  // more than 8 cameras: chunk_kernel (tri_pipe.cuh) -- 32 cameras x 20 M frames: LM FP64 5.37 -> 3.30 ms, closed
  // form FP64 5.01 -> 2.81 ms, FP32 3.69 -> 1.81 ms against the generic kernel (profiles/r1_32cams.log)
  static constexpr bool CHUNKED = true;
  static constexpr int CHUNK_FPT = sizeof(T_) == 4 ? 2 : 1;
  struct Acc {
    T uu[6] = {0, 0, 0, 0, 0, 0};  // sum u u^T / |v|^2        (M = tr I - uu)
    T cu[3] = {0, 0, 0};           // sum u (s . ob)           (c = cn - cu)
    T cn[3] = {0, 0, 0};           // sum n4 ob
    T so[3] = {0, 0, 0};           // sum ob                   (LM start = mean of origins, :90-98)
    T tr = 0, ku = 0, kn = 0;      // k = kn - ku
  };
  // u (unnormalised rotated ray) and 1/|v|^2 of one view; R = RayFold<T>, or RayRigX2 for RayPolicy<float>
  template <class R>
  static __device__ __forceinline__ void ray(const R& r, int c, T x, T y, T (&u)[3], T& inv) {
    u[0] = fma_(lo(r.U0[c][0]), x, fma_(lo(r.U1[c][0]), y, lo(r.U2[c][0])));
    u[1] = fma_(lo(r.U0[c][1]), x, fma_(lo(r.U1[c][1]), y, lo(r.U2[c][1])));
    u[2] = fma_(lo(r.U0[c][2]), x, fma_(lo(r.U1[c][2]), y, lo(r.U2[c][2])));
    const T vx = fma_(lo(r.ax[c]), x, lo(r.bx[c])), vy = fma_(lo(r.ay[c]), y, lo(r.by[c]));
    inv = rcp_ray(fma_(vx, vx, fma_(vy, vy, lo(r.dd[c]))));
  }
  // the pixel-dependent terms of one view ...
  template <bool BRANCH = true>
  static __device__ __forceinline__ void add_pixel(const Rig& r, int c, T x, T y, bool valid, Acc& a) {
    if constexpr (BRANCH) { if (!valid) return; }
    T u[3], inv;
    ray(r, c, x, y, u, inv);
    if constexpr (!BRANCH) inv = valid ? inv : T(0);  // an absent view adds exact zeros (u is finite)
    const T s0 = mul_(u[0], inv), s1 = mul_(u[1], inv), s2 = mul_(u[2], inv);
    a.uu[0] = fma_(s0, u[0], a.uu[0]); a.uu[1] = fma_(s0, u[1], a.uu[1]); a.uu[2] = fma_(s0, u[2], a.uu[2]);
    a.uu[3] = fma_(s1, u[1], a.uu[3]); a.uu[4] = fma_(s1, u[2], a.uu[4]); a.uu[5] = fma_(s2, u[2], a.uu[5]);
    const T t = fma_(s0, r.ob[c][0], fma_(s1, r.ob[c][1], mul_(s2, r.ob[c][2])));
    const T w = fma_(u[0], r.ob[c][0], fma_(u[1], r.ob[c][1], mul_(u[2], r.ob[c][2])));
    a.cu[0] = fma_(u[0], t, a.cu[0]); a.cu[1] = fma_(u[1], t, a.cu[1]); a.cu[2] = fma_(u[2], t, a.cu[2]);
    a.ku = fma_(t, w, a.ku);
  }
  // ... and the ones that depend on its presence alone (the streaming tiles take these from rig.mask_table)
  static __device__ __forceinline__ void add_const(const Rig& r, int c, bool valid, Acc& a) {
    if (!valid) return;
    a.cn[0] += r.n4ob[c][0]; a.cn[1] += r.n4ob[c][1]; a.cn[2] += r.n4ob[c][2];
    a.so[0] += r.ob[c][0]; a.so[1] += r.ob[c][1]; a.so[2] += r.ob[c][2];
    a.tr += r.n4[c];
    a.kn += r.n4ob2[c];
  }
  static __device__ __forceinline__ void add(const Rig& r, int c, T x, T y, bool valid, Acc& a) {
    add_pixel(r, c, x, y, valid, a);
    add_const(r, c, valid, a);
  }
  // chunk_kernel: the pixel terms branch-free (views of a chunk can then overlap), the cheap presence terms skipped
  static __device__ __forceinline__ void add_chunk(const Rig& r, int c, T x, T y, bool valid, Acc& a) {
    add_pixel<false>(r, c, x, y, valid, a);
    add_const(r, c, valid, a);
  }
  static __device__ __forceinline__ T quad(const T (&M)[6], const T (&c)[3], T k, const T (&p)[3]) {
    const T Mp0 = fma_(M[0], p[0], fma_(M[1], p[1], mul_(M[2], p[2])));
    const T Mp1 = fma_(M[1], p[0], fma_(M[3], p[1], mul_(M[4], p[2])));
    const T Mp2 = fma_(M[2], p[0], fma_(M[4], p[1], mul_(M[5], p[2])));
    return fma_(p[0], fma_(T(-2), c[0], Mp0), fma_(p[1], fma_(T(-2), c[1], Mp1), fma_(p[2], fma_(T(-2), c[2], Mp2), k)));
  }
  static __device__ __forceinline__ void solve(const Rig&, const Acc& a, uint32_t, int n, T (&X)[3], int opt, int& iters) {
    const T M[6] = {a.tr - a.uu[0], -a.uu[1], -a.uu[2], a.tr - a.uu[3], -a.uu[4], a.tr - a.uu[5]};
    const T c[3] = {a.cn[0] - a.cu[0], a.cn[1] - a.cu[1], a.cn[2] - a.cu[2]};
    if (!(opt & 1)) {
      solve_sym3<T>(M, c, X);
      iters = 1;
      return;
    }
    // cv::LMSolver's loop (calib3d levmarq.cpp: lambda = 1, lc = 0.75, Rlo/Rhi = 0.25/0.75, diagonal
    // scaling fixed at the start point, eps = FLT_EPSILON, 1000 iterations: RayTriangulator.h:9-11,
    // RayTriangulator.cpp:100-104) on the analytic normal equations A = M, v = M p - c.
    const T k = a.kn - a.ku;
    const T rn = rcp_((T)n);
    T p[3] = {a.so[0] * rn, a.so[1] * rn, a.so[2] * rn};
    const T D[3] = {M[0], M[3], M[5]};
    T lambda = 1, lc = T(0.75);
    T S = quad(M, c, k, p);
    T g[3] = {M[0] * p[0] + M[1] * p[1] + M[2] * p[2] - c[0], M[1] * p[0] + M[3] * p[1] + M[4] * p[2] - c[1],
              M[2] * p[0] + M[4] * p[1] + M[5] * p[2] - c[2]};
    int it = 0;
    for (;;) {
      const T Ap[6] = {M[0] + lambda * D[0], M[1], M[2], M[3] + lambda * D[1], M[4], M[5] + lambda * D[2]};
      T d[3];
      solve_sym3<T>(Ap, g, d);
      const T pd[3] = {p[0] - d[0], p[1] - d[1], p[2] - d[2]};
      const T Sd = quad(M, c, k, pd);
      const T Md0 = M[0] * d[0] + M[1] * d[1] + M[2] * d[2], Md1 = M[1] * d[0] + M[3] * d[1] + M[4] * d[2],
              Md2 = M[2] * d[0] + M[4] * d[1] + M[5] * d[2];
      const T dS = d[0] * (2 * g[0] - Md0) + d[1] * (2 * g[1] - Md1) + d[2] * (2 * g[2] - Md2);
      const T R = (S - Sd) * rcp_(fabs(dS) > (T)DBL_EPSILON ? dS : T(1));
      if (R > T(0.75)) {
        lambda *= T(0.5);
        if (lambda < lc) lambda = 0;
      } else if (R < T(0.25)) {
        const T t = d[0] * g[0] + d[1] * g[1] + d[2] * g[2];
        T nu = (Sd - S) * rcp_(fabs(t) > (T)DBL_EPSILON ? t : T(1)) + 2;
        nu = fmin(fmax(nu, T(2)), T(10));
        if (lambda == 0) {  // re-inflate from diag(M^-1)
          const T c00 = M[3] * M[5] - M[4] * M[4], c11 = M[0] * M[5] - M[2] * M[2], c22 = M[0] * M[3] - M[1] * M[1];
          const T det = M[0] * c00 + M[1] * (M[2] * M[4] - M[1] * M[5]) + M[2] * (M[1] * M[4] - M[2] * M[3]);
          const T idet = rcp_(det);
          const T mx = fmax(fmax(fabs(c00 * idet), fabs(c11 * idet)), fmax(fabs(c22 * idet), (T)DBL_EPSILON));
          lambda = lc = rcp_(mx);
          nu *= T(0.5);
        }
        lambda *= nu;
      }
      if (Sd < S) {
        S = Sd;
        p[0] = pd[0]; p[1] = pd[1]; p[2] = pd[2];
        g[0] -= Md0; g[1] -= Md1; g[2] -= Md2;  // M (p - d) - c
      }
      it++;
      const T dmax = fmax(fabs(d[0]), fmax(fabs(d[1]), fabs(d[2])));
      if (!(it < 1000 && dmax >= (T)FLT_EPSILON)) break;
    }
    X[0] = p[0]; X[1] = p[1]; X[2] = p[2];
    iters = it;
  }
  // r_i = |dir_i x (p - o_i)| (Triangulator.cpp:3-9); the reported error is the mean (RayTriangulator.cpp:26)
  template <class R>
  static __device__ __forceinline__ T residual(const R& r, int c, T x, T y, const T (&X)[3]) {
    T u[3], inv;
    ray(r, c, x, y, u, inv);
    const T w0 = X[0] - lo(r.ob[c][0]), w1 = X[1] - lo(r.ob[c][1]), w2 = X[2] - lo(r.ob[c][2]);
    const T c0 = fma_(u[1], w2, -mul_(u[2], w1)), c1 = fma_(u[2], w0, -mul_(u[0], w2)), c2 = fma_(u[0], w1, -mul_(u[1], w0));
    return sqrt(mul_(fma_(c0, c0, fma_(c1, c1, mul_(c2, c2))), inv));
  }
  static __device__ __forceinline__ double error(T sum, int n) { return (double)sum / (double)n; }
  static __device__ __forceinline__ void to_world(const Rig& r, T (&X)[3]) {
    X[0] += r.origin[0]; X[1] += r.origin[1]; X[2] += r.origin[2];
  }
};

// ---- streaming tile of the scalar policy, one frame per thread: the validity mask first, its table row
// requested at once (it is needed only after the camera loop, so the load hides behind it), the solver a
// compile-time choice (the closed form then drops the terms only the LM loop reads) ----
template <typename T_, bool LM, int FPT_ = 1>
struct RayTableTile {
  static constexpr int FPT = FPT_;
  using S = RayPolicy<T_>;
  using Rig = typename S::Rig;
  using Real = T_;
  template <int NC, int PIX, bool WIDE, class RS>
  static __device__ __forceinline__ void run(const Rig& rig, const RS& raw, int, T_ (&X)[FPT][3],
                                             uint32_t (&mask)[FPT], double (&err)[FPT], int (&iters)[FPT]) {
    using T = T_;
    static_assert(NC <= TRI_RAY_TABLE_CAMS, "the mask table covers 8 cameras");
#pragma unroll
    for (int j = 0; j < FPT; j++) mask[j] = 0;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const Views<float, PIX, FPT> v = decode<float, PIX, FPT>(raw[c]);
#pragma unroll
      for (int j = 0; j < FPT; j++) mask[j] |= (v.v[j] ? 1u : 0u) << c;
    }
    T row[FPT][8];
#pragma unroll
    for (int j = 0; j < FPT; j++) {
      if constexpr (sizeof(T) == 8) {
        const double2* src = reinterpret_cast<const double2*>(rig.mask_table + 8 * mask[j]);
#pragma unroll
        for (int k = 0; k < (LM ? 4 : 2); k++) { const double2 t = __ldg(src + k); row[j][2 * k] = t.x; row[j][2 * k + 1] = t.y; }
      } else {
        const float4* src = reinterpret_cast<const float4*>(rig.mask_table + 8 * mask[j]);
#pragma unroll
        for (int k = 0; k < (LM ? 2 : 1); k++) { const float4 t = __ldg(src + k); row[j][4 * k] = t.x; row[j][4 * k + 1] = t.y; row[j][4 * k + 2] = t.z; row[j][4 * k + 3] = t.w; }
      }
    }
    typename S::Acc acc[FPT];
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const Views<T, PIX, FPT> w = decode<T, PIX, FPT>(raw[c]);
      // absent views: skipped by a branch in the closed form, masked branch-free under the LM loop (measured:
      // 2.54 vs 3.04 ms and 4.75 vs 4.98 ms per 100 M frames -- the branch-free closed form spills at 128 registers)
#pragma unroll
      for (int j = 0; j < FPT; j++) S::template add_pixel<!LM>(rig, c, w.x[j], w.y[j], w.v[j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < FPT; j++) {
      acc[j].cn[0] = row[j][0]; acc[j].cn[1] = row[j][1]; acc[j].cn[2] = row[j][2]; acc[j].tr = row[j][3];
      if constexpr (LM) { acc[j].so[0] = row[j][4]; acc[j].so[1] = row[j][5]; acc[j].so[2] = row[j][6]; acc[j].kn = row[j][7]; }
      X[j][0] = X[j][1] = X[j][2] = 0;
      err[j] = 0;
      iters[j] = 0;
      const int n = __popc(mask[j]);
      if (n >= 2) {
        S::solve(rig, acc[j], mask[j], n, X[j], LM ? 1 : 0, iters[j]);
        if constexpr (WIDE) {  // mean distance to the rays at the solution (RayTriangulator.cpp:26)
          T e = 0;
#pragma unroll
          for (int c = 0; c < NC; c++) {
            const Views<T, PIX, FPT> w = decode<T, PIX, FPT>(raw[c]);
            if (w.v[j]) e += S::residual(rig, c, w.x[j], w.y[j], X[j]);
          }
          err[j] = S::error(e, n);
        }
        S::to_world(rig, X[j]);
      }
    }
  }
};

// ---- FP32 closed form, packed-pair SIMD (the ray counterpart of DltX2Tile) ----
// Same operation order as RayPolicy<float> (which serves tails and optional outputs), so the points are
// bit-identical; an absent view is masked by zeroing 1/|v|^2 and the constant terms' weight.
struct __align__(16) RayRigX2 {
  float2 U0[TRI_MAX_CAMS][3], U1[TRI_MAX_CAMS][3], U2[TRI_MAX_CAMS][3];
  float2 ax[TRI_MAX_CAMS], bx[TRI_MAX_CAMS], ay[TRI_MAX_CAMS], by[TRI_MAX_CAMS], dd[TRI_MAX_CAMS], n4[TRI_MAX_CAMS];
  float2 ob[TRI_MAX_CAMS][3], n4ob[TRI_MAX_CAMS][3];
  float origin[3];
  const float* mask_table;  // RayFold<float>::mask_table
};

struct RayX2Tile {
  static constexpr int FPT = 2;
  using Rig = RayRigX2;
  using Real = float;
  template <int NC, int PIX, bool WIDE, class RS>
  static __device__ __forceinline__ void run(const Rig& r, const RS& raw, int, float (&X)[2][3],
                                             uint32_t (&mask)[2], double (&err)[2], int (&iters)[2]) {
    const float2 z = make_float2(0.f, 0.f);
    float2 uu[6] = {z, z, z, z, z, z}, cu[3] = {z, z, z};
    uint32_t mask0 = 0, mask1 = 0;
#pragma unroll
    for (int c = 0; c < NC; c++) {  // one pass over the views: the validity masks build up alongside the sums
      const Views<float, PIX, 2> q = decode<float, PIX, 2>(raw[c]);
      mask0 |= (q.v[0] ? 1u : 0u) << c;
      mask1 |= (q.v[1] ? 1u : 0u) << c;
      const float2 x = make_float2(q.x[0], q.x[1]), y = make_float2(q.y[0], q.y[1]);
      const float2 u0 = fma2(r.U0[c][0], x, fma2(r.U1[c][0], y, r.U2[c][0]));
      const float2 u1 = fma2(r.U0[c][1], x, fma2(r.U1[c][1], y, r.U2[c][1]));
      const float2 u2 = fma2(r.U0[c][2], x, fma2(r.U1[c][2], y, r.U2[c][2]));
      const float2 vx = fma2(r.ax[c], x, r.bx[c]), vy = fma2(r.ay[c], y, r.by[c]);
      const float2 vv = fma2(vx, vx, fma2(vy, vy, r.dd[c]));
      const float2 inv = make_float2(q.v[0] ? rcp_ray(vv.x) : 0.f, q.v[1] ? rcp_ray(vv.y) : 0.f);
      const float2 s0 = mul2(u0, inv), s1 = mul2(u1, inv), s2 = mul2(u2, inv);
      uu[0] = fma2(s0, u0, uu[0]); uu[1] = fma2(s0, u1, uu[1]); uu[2] = fma2(s0, u2, uu[2]);
      uu[3] = fma2(s1, u1, uu[3]); uu[4] = fma2(s1, u2, uu[4]); uu[5] = fma2(s2, u2, uu[5]);
      const float2 t = fma2(s0, r.ob[c][0], fma2(s1, r.ob[c][1], mul2(s2, r.ob[c][2])));
      cu[0] = fma2(u0, t, cu[0]); cu[1] = fma2(u1, t, cu[1]); cu[2] = fma2(u2, t, cu[2]);
    }
    // sum of n4 ob and of n4 over the valid cameras: one table row per frame (L1-resident, 8 KB)
    const float4 k0 = __ldg(reinterpret_cast<const float4*>(r.mask_table + 8 * mask0));
    const float4 k1 = __ldg(reinterpret_cast<const float4*>(r.mask_table + 8 * mask1));
    const float2 cn[3] = {make_float2(k0.x, k1.x), make_float2(k0.y, k1.y), make_float2(k0.z, k1.z)}, tr = make_float2(k0.w, k1.w);
    const float2 M[6] = {add2(tr, neg2(uu[0])), neg2(uu[1]), neg2(uu[2]), add2(tr, neg2(uu[3])), neg2(uu[4]), add2(tr, neg2(uu[5]))};
    const float2 cc[3] = {add2(cn[0], neg2(cu[0])), add2(cn[1], neg2(cu[1])), add2(cn[2], neg2(cu[2]))};
    float2 X0, X1, X2;
    solve_sym3_x2(M, cc, X0, X1, X2);
    const bool ok0 = __popc(mask0) >= 2, ok1 = __popc(mask1) >= 2;
    mask[0] = mask0; mask[1] = mask1;
    const float Xr[2][3] = {{X0.x, X1.x, X2.x}, {X0.y, X1.y, X2.y}};
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const bool ok = j == 0 ? ok0 : ok1;
      err[j] = 0;
      iters[j] = ok ? 1 : 0;
      if constexpr (WIDE) {
        if (ok) {  // mean distance to the rays
          float e = 0;
#pragma unroll
          for (int c = 0; c < NC; c++) {
            const Views<float, PIX, 2> q = decode<float, PIX, 2>(raw[c]);
            if (q.v[j]) e += RayPolicy<float>::residual(r, c, q.x[j], q.y[j], Xr[j]);
          }
          err[j] = RayPolicy<float>::error(e, __popc(j == 0 ? mask0 : mask1));
        }
      }
      X[j][0] = ok ? Xr[j][0] + r.origin[0] : 0.f; X[j][1] = ok ? Xr[j][1] + r.origin[1] : 0.f; X[j][2] = ok ? Xr[j][2] + r.origin[2] : 0.f;
    }
  }
};

static RayRigX2 make_ray_x2(const RayFold<float>& f) {
  RayRigX2 x;
  auto d = [](float v) { return make_float2(v, v); };
  for (int c = 0; c < TRI_MAX_CAMS; c++) {
    for (int k = 0; k < 3; k++) {
      x.U0[c][k] = d(f.U0[c][k]); x.U1[c][k] = d(f.U1[c][k]); x.U2[c][k] = d(f.U2[c][k]);
      x.ob[c][k] = d(f.ob[c][k]); x.n4ob[c][k] = d(f.n4ob[c][k]);
    }
    x.ax[c] = d(f.ax[c]); x.bx[c] = d(f.bx[c]); x.ay[c] = d(f.ay[c]); x.by[c] = d(f.by[c]); x.dd[c] = d(f.dd[c]); x.n4[c] = d(f.n4[c]);
  }
  for (int k = 0; k < 3; k++) x.origin[k] = f.origin[k];
  x.mask_table = f.mask_table;
  return x;
}

cudaError_t launch_ray_fold(const LaunchCtx& ctx, bool lm, bool f32, int pixfmt, const RayFold<double>& r64,
                            const RayFold<float>& r32, const void* d_xy, int n_use, int64_t n_frames,
                            int64_t cam_stride, const BatchOut& out) {
  if (n_frames <= 0) return cudaSuccess;
  using P32 = RayPolicy<float>;
  using P64 = RayPolicy<double>;
  const int opt = lm ? 1 : 0;
  if (f32) {  // FP32: closed form only (the gain ratio of the LM loop needs S to ~1e-9 relative)
    const RayRigX2 x2 = make_ray_x2(r32);
    switch (pixfmt) {
      case PIX_F32:
        // 3 stages x 2 CTAs per SM: 1.32 ms per 100 M frames; 2 stages x 3 CTAs (the DLT's choice): 1.47 ms -- with the
        // lighter solve the kernel waits on memory (ncu r1f: long_scoreboard on top), so depth beats occupancy
        // one pass over the views, pixels read from the slot as they are needed: 1.32 -> 1.26 ms per 100 M frames
        // (profiles/r2_dlt_variants.log; with the pixels pulled into registers on arrival the single pass measured 1.37)
        return launch_streamed<RayX2Tile, P32, PIX_F32, 2, 3, 2, true>(ctx, x2, r32, d_xy, n_use, n_frames, cam_stride, out, 0);
      case PIX_F64: return launch_streamed<RayX2Tile, P32, PIX_F64, 2, 3, 2>(ctx, x2, r32, d_xy, n_use, n_frames, cam_stride, out, 0);
      default: return launch_streamed<RayX2Tile, P32, PIX_U16, 2, 3, 2>(ctx, x2, r32, d_xy, n_use, n_frames, cam_stride, out, 0);
    }
  }
  // one frame per thread; the solver is a compile-time choice of the tile (the scalar policy serves the tails)
  // two frames per thread in both solvers (independent chains for the FP64 pipe): LM 4.70 -> 4.44 ms, closed form
  // 2.50 -> 2.41 ms per 100 M frames
  using LMT = RayTableTile<double, true, 2>;
  using CFT = RayTableTile<double, false, 2>;
  switch (pixfmt) {
    case PIX_F32:
      // (4- and 6-stage rings measured the same: these two are FP64-pipe-bound)
      return lm ? launch_streamed<LMT, P64, PIX_F32, 2, 2, 2>(ctx, r64, r64, d_xy, n_use, n_frames, cam_stride, out, opt)
                : launch_streamed<CFT, P64, PIX_F32, 2, 3, 2>(ctx, r64, r64, d_xy, n_use, n_frames, cam_stride, out, opt);
    case PIX_F64: return launch_streamed<LMT, P64, PIX_F64, 1, 3, 2>(ctx, r64, r64, d_xy, n_use, n_frames, cam_stride, out, opt);
    default:
      return lm ? launch_streamed<LMT, P64, PIX_U16, 2, 2, 2>(ctx, r64, r64, d_xy, n_use, n_frames, cam_stride, out, opt)
                : launch_streamed<CFT, P64, PIX_U16, 2, 3, 2>(ctx, r64, r64, d_xy, n_use, n_frames, cam_stride, out, opt);
  }
}

}  // namespace tri
