// tri_batch.cuh -- the streaming skeleton shared by the batched triangulatePoints kernels
// (kernel 4 of the north star: structure-of-arrays detections, validity bitmask, vector loads,
// shared-memory staged output).
//
// Layout in HBM: pixels xy[cam][frame] (float2 | double2 | ushort2), camera rows `row_bytes` apart;
// (-1,-1) -- or 0xFFFF,0xFFFF for ushort2 -- marks "no detection" (DetectionsContainer.cpp:145-171,
// MatrixTriangulator.cpp:86, RayTriangulator.cpp:66).  One thread owns two consecutive frames: one
// 16-byte load per camera (8 for ushort2), all cameras' loads issued before the first use.  The
// per-frame solve is a policy class S:
//     S::T, S::Rig (a __grid_constant__ parameter: operands come from the constant bank), S::Acc,
//     S::add(rig, c, x, y, valid, acc)     one view into the accumulator (a no-op when !valid)
//     S::solve(rig, acc, mask, n, X, opt, iters) the per-frame solve, X in rig coordinates (mask = validity bits:
//                                          the FP32 DLT takes its absent-view correction from a table row)
//     S::residual(rig, c, x, y, X)         that view's contribution to the reported error
//     S::error(sum, n)                     the reported error from the summed contributions
//     S::to_world(rig, X)
// Results: float3 packed (12 B) through a shared-memory tile -> coalesced 16-byte streaming stores;
// optional double3 / mask / err / iters outputs for parity tests and the classifier.
#pragma once
#include "tri_common.cuh"

namespace tri {

constexpr int BATCH_THREADS = 256;

template <typename T>
struct View2 {  // the pixels of two consecutive frames on one camera
  T x0, y0, x1, y1;
  bool v0, v1;
};

template <typename T, int PIX>
__device__ __forceinline__ View2<T> fetch2(const char* row, int64_t pair) {
  View2<T> r;
  if constexpr (PIX == PIX_F32) {
    float4 q = ld_stream(reinterpret_cast<const float4*>(row) + pair);
    r.v0 = pix_valid(q.x, q.y);
    r.v1 = pix_valid(q.z, q.w);
    r.x0 = to_real<T>(q.x); r.y0 = to_real<T>(q.y); r.x1 = to_real<T>(q.z); r.y1 = to_real<T>(q.w);
  } else if constexpr (PIX == PIX_F64) {
    double2 a = ld_stream(reinterpret_cast<const double2*>(row) + 2 * pair);
    double2 b = ld_stream(reinterpret_cast<const double2*>(row) + 2 * pair + 1);
    r.v0 = pix_valid(a.x, a.y);
    r.v1 = pix_valid(b.x, b.y);
    r.x0 = (T)a.x; r.y0 = (T)a.y; r.x1 = (T)b.x; r.y1 = (T)b.y;
  } else {
    uint2 q = ld_stream(reinterpret_cast<const uint2*>(row) + pair);
    r.v0 = q.x != 0xffffffffu;
    r.v1 = q.y != 0xffffffffu;
    if constexpr (sizeof(T) == 8) {  // integers < 2^16 -> double without touching the conversion pipe
      const double magic = 4503599627370496.0;  // 2^52
      r.x0 = __hiloint2double(0x43300000, (int)(q.x & 0xffffu)) - magic;
      r.y0 = __hiloint2double(0x43300000, (int)(q.x >> 16)) - magic;
      r.x1 = __hiloint2double(0x43300000, (int)(q.y & 0xffffu)) - magic;
      r.y1 = __hiloint2double(0x43300000, (int)(q.y >> 16)) - magic;
    } else {
      r.x0 = (T)(q.x & 0xffffu); r.y0 = (T)(q.x >> 16); r.x1 = (T)(q.y & 0xffffu); r.y1 = (T)(q.y >> 16);
    }
  }
  return r;
}

template <typename T, int PIX>
__device__ __forceinline__ void fetch1(const char* row, int64_t f, T& x, T& y, bool& v) {
  if constexpr (PIX == PIX_F32) {
    float2 q = ld_stream(reinterpret_cast<const float2*>(row) + f);
    v = pix_valid(q.x, q.y); x = (T)q.x; y = (T)q.y;
  } else if constexpr (PIX == PIX_F64) {
    double2 q = ld_stream(reinterpret_cast<const double2*>(row) + f);
    v = pix_valid(q.x, q.y); x = (T)q.x; y = (T)q.y;
  } else {
    unsigned q = ld_stream(reinterpret_cast<const unsigned*>(row) + f);
    v = q != 0xffffffffu; x = (T)(q & 0xffffu); y = (T)(q >> 16);
  }
}

// ---- FPT (1 or 2) consecutive frames per thread; NC > 0 unrolls the camera loop and keeps every
// pixel in registers.  FPT = 2 needs 16-byte aligned camera rows (8 for ushort2). ----
template <typename T, int PIX, int FPT>
struct Views {
  T x[FPT], y[FPT];
  bool v[FPT];
};

template <typename T, int PIX, int FPT>
__device__ __forceinline__ Views<T, PIX, FPT> fetch(const char* row, int64_t group) {
  Views<T, PIX, FPT> r;
  if constexpr (FPT == 2) {
    View2<T> w = fetch2<T, PIX>(row, group);
    r.x[0] = w.x0; r.y[0] = w.y0; r.v[0] = w.v0; r.x[1] = w.x1; r.y[1] = w.y1; r.v[1] = w.v1;
  } else {
    fetch1<T, PIX>(row, group, r.x[0], r.y[0], r.v[0]);
  }
  return r;
}

template <class S, int NC, int PIX, int FPT, int MINB>
__global__ void __launch_bounds__(BATCH_THREADS, MINB)
batch_kernel(const __grid_constant__ typename S::Rig rig, const char* __restrict__ xy, int64_t row_bytes,
             int64_t n_groups, int n_use, BatchOut out, int opt, unsigned long long* first_bad, int64_t frame_base) {
  using T = typename S::T;
  __shared__ __align__(16) float tile[BATCH_THREADS * 3 * FPT];
  const int64_t block_group0 = (int64_t)blockIdx.x * BATCH_THREADS;
  const int64_t group = block_group0 + threadIdx.x;
  const int nc = NC > 0 ? NC : n_use;
  T X[FPT][3];
#pragma unroll
  for (int j = 0; j < FPT; j++) X[j][0] = X[j][1] = X[j][2] = 0;

  if (group < n_groups) {
    typename S::Acc acc[FPT];
    uint32_t mask[FPT];
    T e[FPT];
    int it[FPT], n[FPT];
#pragma unroll
    for (int j = 0; j < FPT; j++) { mask[j] = 0; e[j] = 0; it[j] = 0; }
    if constexpr (NC > 0) {
      Views<T, PIX, FPT> w[NC];
#pragma unroll
      for (int c = 0; c < NC; c++) w[c] = fetch<T, PIX, FPT>(xy + c * row_bytes, group);  // all loads in flight
#pragma unroll
      for (int c = 0; c < NC; c++)
#pragma unroll
        for (int j = 0; j < FPT; j++)
          { S::add(rig, c, w[c].x[j], w[c].y[j], w[c].v[j], acc[j]); mask[j] |= (w[c].v[j] ? 1u : 0u) << c; }
#pragma unroll
      for (int j = 0; j < FPT; j++) {
        n[j] = __popc(mask[j]);
        if (n[j] >= 2) S::solve(rig, acc[j], mask[j], n[j], X[j], opt, it[j]);
      }
      if (out.err) {
#pragma unroll
        for (int c = 0; c < NC; c++)
#pragma unroll
          for (int j = 0; j < FPT; j++)
            if (w[c].v[j]) e[j] += S::residual(rig, c, w[c].x[j], w[c].y[j], X[j]);
      }
    } else {
#pragma unroll 4
      for (int c = 0; c < nc; c++) {
        Views<T, PIX, FPT> w = fetch<T, PIX, FPT>(xy + c * row_bytes, group);
#pragma unroll
        for (int j = 0; j < FPT; j++)
          { S::add(rig, c, w.x[j], w.y[j], w.v[j], acc[j]); mask[j] |= (w.v[j] ? 1u : 0u) << c; }
      }
#pragma unroll
      for (int j = 0; j < FPT; j++) {
        n[j] = __popc(mask[j]);
        if (n[j] >= 2) S::solve(rig, acc[j], mask[j], n[j], X[j], opt, it[j]);
      }
      if (out.err) {
        for (int c = 0; c < nc; c++) {
          Views<T, PIX, FPT> w = fetch<T, PIX, FPT>(xy + c * row_bytes, group);
#pragma unroll
          for (int j = 0; j < FPT; j++)
            if (w.v[j]) e[j] += S::residual(rig, c, w.x[j], w.y[j], X[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < FPT; j++) {
      const int64_t f = FPT * group + j;
      if (n[j] >= 2) S::to_world(rig, X[j]);
      else atomicMin(first_bad, (unsigned long long)(frame_base + f));
      if (out.xyz_f64) { double* o = out.xyz_f64 + 3 * f; o[0] = X[j][0]; o[1] = X[j][1]; o[2] = X[j][2]; }
      if (out.mask) out.mask[f] = mask[j];
      if (out.err) out.err[f] = n[j] >= 2 ? S::error(e[j], n[j]) : 0.0;
      if (out.iters) out.iters[f] = it[j];
    }
  }

  if (out.xyz_f32) {  // uniform branch: 12 B per frame into the tile, the tile out as 16 B vectors
    float* t = tile + 3 * FPT * threadIdx.x;
#pragma unroll
    for (int j = 0; j < FPT; j++) { t[3 * j] = (float)X[j][0]; t[3 * j + 1] = (float)X[j][1]; t[3 * j + 2] = (float)X[j][2]; }
    __syncthreads();
    const int64_t remaining = n_groups - block_group0;
    float* dst = out.xyz_f32 + 3 * FPT * block_group0;
    if (remaining >= BATCH_THREADS && ((uintptr_t)dst & 15) == 0) {
      float4* d4 = reinterpret_cast<float4*>(dst);
      const float4* s4 = reinterpret_cast<const float4*>(tile);
#pragma unroll
      for (int i = threadIdx.x; i < BATCH_THREADS * 3 * FPT / 4; i += BATCH_THREADS) __stcs(d4 + i, s4[i]);
    } else {
      const int cnt = (int)(remaining < BATCH_THREADS ? remaining : BATCH_THREADS) * 3 * FPT;
      for (int i = threadIdx.x; i < cnt; i += BATCH_THREADS) dst[i] = tile[i];
    }
  }
}

// ---- fallback: one frame per thread, scalar loads (unaligned rows, odd tail frame) ----
template <class S, int PIX>
__global__ void __launch_bounds__(BATCH_THREADS)
batch_single_kernel(const __grid_constant__ typename S::Rig rig, const char* __restrict__ xy, int64_t row_bytes,
                    int64_t f_begin, int64_t f_end, int n_use, BatchOut out, int opt, unsigned long long* first_bad,
                    int64_t frame_base) {
  using T = typename S::T;
  const int64_t f = f_begin + (int64_t)blockIdx.x * BATCH_THREADS + threadIdx.x;
  if (f >= f_end) return;
  typename S::Acc acc;
  T X[3] = {0, 0, 0}, e = 0;
  uint32_t mask = 0;
  int it = 0;
  for (int c = 0; c < n_use; c++) {
    T x, y; bool ok;
    fetch1<T, PIX>(xy + c * row_bytes, f, x, y, ok);
    { S::add(rig, c, x, y, ok, acc); mask |= (ok ? 1u : 0u) << c; }
  }
  const int n = __popc(mask);
  if (n >= 2) {
    S::solve(rig, acc, mask, n, X, opt, it);
    if (out.err)
      for (int c = 0; c < n_use; c++) {
        T x, y; bool ok;
        fetch1<T, PIX>(xy + c * row_bytes, f, x, y, ok);
        if (ok) e += S::residual(rig, c, x, y, X);
      }
    S::to_world(rig, X);
  } else {
    atomicMin(first_bad, (unsigned long long)(frame_base + f));
  }
  if (out.xyz_f32) { float* o = out.xyz_f32 + 3 * f; o[0] = (float)X[0]; o[1] = (float)X[1]; o[2] = (float)X[2]; }
  if (out.xyz_f64) { double* o = out.xyz_f64 + 3 * f; o[0] = X[0]; o[1] = X[1]; o[2] = X[2]; }
  if (out.mask) out.mask[f] = mask;
  if (out.err) out.err[f] = n >= 2 ? S::error(e, n) : 0.0;
  if (out.iters) out.iters[f] = it;
}

// FPT = frames per thread of the main kernel, MINB = resident blocks per SM asked of ptxas.
template <class S, int PIX, int FPT, int MINB>
static cudaError_t launch_batch_policy(const LaunchCtx& ctx, const typename S::Rig& rig, const void* d_xy, int n_use,
                                       int64_t n_frames, int64_t cam_stride, const BatchOut& out, int opt) {
  const char* xy = static_cast<const char*>(d_xy);
  const int64_t row_bytes = cam_stride * pix_bytes(PIX);
  const int64_t need = FPT * pix_bytes(PIX);  // every camera row must start vector-aligned
  const bool vec = FPT == 1 || (((uintptr_t)xy % need == 0) && (row_bytes % need == 0));
  const int64_t n_groups = vec ? n_frames / FPT : 0;
  if (n_groups > 0) {
    const unsigned grid = (unsigned)((n_groups + BATCH_THREADS - 1) / BATCH_THREADS);
#define TRI_CASE(N)                                                                                              \
  case N:                                                                                                        \
    batch_kernel<S, N, PIX, FPT, MINB><<<grid, BATCH_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, n_groups, n_use, \
                                                                               out, opt, ctx.d_first_bad,        \
                                                                               ctx.frame_base);                  \
    break;
    switch (n_use) {
      TRI_CASE(2) TRI_CASE(3) TRI_CASE(4) TRI_CASE(5) TRI_CASE(6) TRI_CASE(7) TRI_CASE(8)
      default:
        batch_kernel<S, 0, PIX, FPT, MINB><<<grid, BATCH_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, n_groups, n_use, out,
                                                                                   opt, ctx.d_first_bad, ctx.frame_base);
    }
#undef TRI_CASE
    ++*ctx.launches;
  }
  const int64_t done = FPT * n_groups;
  if (done < n_frames) {
    const unsigned grid = (unsigned)((n_frames - done + BATCH_THREADS - 1) / BATCH_THREADS);
    batch_single_kernel<S, PIX><<<grid, BATCH_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, done, n_frames, n_use, out,
                                                                        opt, ctx.d_first_bad, ctx.frame_base);
    ++*ctx.launches;
  }
  return cudaGetLastError();
}

}  // namespace tri
