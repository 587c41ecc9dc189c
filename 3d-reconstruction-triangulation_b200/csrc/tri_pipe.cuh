// tri_pipe.cuh -- persistent streaming kernels of the batched triangulatePoints hot path.
//
// grid = SMs x resident CTAs, each CTA walks tiles t = blockIdx.x, += gridDim.x of BATCH_THREADS x FPT frames; the
// pixels of the next STAGES tiles are always in flight into a shared-memory ring while the current tile is solved;
// the 12-byte points leave through a per-warp transpose as 16-byte streaming stores.  Every thread prefetches its own
// pixels with cp.async (LDGSTS) and waits on its own copy group -- no cross-warp synchronisation at all.  A
// warp-specialised TMA feeder (a producer warp issuing 1-D bulk copies onto per-stage mbarriers) was measured against it
// in round 2 (profiles/r2_dlt_variants.log): with a near-empty solve it is the faster feeder (1.10 ms per 100 M frames =
// 6.9 TB/s), but under every real solve it loses (FP32 DLT 1.295 vs 1.269 ms, FP32 ray 1.45 vs 1.32, FP64 DLT 1.96 vs
// 1.86): the ninth warp costs registers (288 threads per CTA) and the consumers of a CTA wake together on the stage's
// barrier instead of drifting apart.
// Algorithmic traffic: 8 B x cameras in, 12 B out per frame; nothing is re-read (profiles/: 7.59 GB per 100 M frames).
#pragma once
#include <type_traits>

#include "tri_batch.cuh"

namespace tri {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// raw pixels of FPT consecutive frames of one camera, as they sit in the shared-memory stage
template <int PIX, int FPT> struct RawPix;
template <> struct RawPix<PIX_F32, 2> { using type = float4; };
template <> struct RawPix<PIX_F32, 1> { using type = float2; };
template <> struct RawPix<PIX_U16, 2> { using type = uint2; };
template <> struct RawPix<PIX_U16, 1> { using type = unsigned; };

template <typename T, int PIX, int FPT>
__device__ __forceinline__ Views<T, PIX, FPT> decode(const typename RawPix<PIX, FPT>::type& q) {
  Views<T, PIX, FPT> r;
  if constexpr (PIX == PIX_F32 && FPT == 2) {
    r.v[0] = pix_valid(q.x, q.y); r.v[1] = pix_valid(q.z, q.w);
    r.x[0] = to_real<T>(q.x); r.y[0] = to_real<T>(q.y); r.x[1] = to_real<T>(q.z); r.y[1] = to_real<T>(q.w);
  } else if constexpr (PIX == PIX_F32 && FPT == 1) {
    r.v[0] = pix_valid(q.x, q.y); r.x[0] = to_real<T>(q.x); r.y[0] = to_real<T>(q.y);
  } else if constexpr (PIX == PIX_U16 && FPT == 2) {
    r.v[0] = q.x != 0xffffffffu; r.v[1] = q.y != 0xffffffffu;
    r.x[0] = (T)(q.x & 0xffffu); r.y[0] = (T)(q.x >> 16); r.x[1] = (T)(q.y & 0xffffu); r.y[1] = (T)(q.y >> 16);
  } else {
    r.v[0] = q != 0xffffffffu; r.x[0] = (T)(q & 0xffffu); r.y[0] = (T)(q >> 16);
  }
  return r;
}

// ---- packed-pair FP32 helpers (FFMA2 / FMUL2 / FADD2, sm_100): two frames in the halves of a float2 ----
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
// adjugate solve of two 3x3 symmetric systems at once; same operation order as solve_sym3<float>
__device__ __forceinline__ void solve_sym3_x2(const float2 (&M)[6], const float2 (&v)[3], float2& X0, float2& X1, float2& X2) {
  const float2 c00 = fma2(M[3], M[5], neg2(mul2(M[4], M[4]))), c01 = fma2(M[2], M[4], neg2(mul2(M[1], M[5]))),
               c02 = fma2(M[1], M[4], neg2(mul2(M[2], M[3]))), c11 = fma2(M[0], M[5], neg2(mul2(M[2], M[2]))),
               c12 = fma2(M[1], M[2], neg2(mul2(M[0], M[4]))), c22 = fma2(M[0], M[3], neg2(mul2(M[1], M[1])));
  const float2 det = fma2(M[0], c00, fma2(M[1], c01, mul2(M[2], c02)));
  const float2 inv = make_float2(1.0f / det.x, 1.0f / det.y);
  X0 = mul2(fma2(c00, v[0], fma2(c01, v[1], mul2(c02, v[2]))), inv);
  X1 = mul2(fma2(c01, v[0], fma2(c11, v[1], mul2(c12, v[2]))), inv);
  X2 = mul2(fma2(c02, v[0], fma2(c12, v[1], mul2(c22, v[2]))), inv);
}

// The pixels of one thread's frames, one RawPix per camera: either pulled into registers when the tile arrives (the slot
// is re-armed at once) or read from the thread's shared-memory slot camera by camera as the solve needs them (LAZY: fewer
// live registers, so more resident warps; the slot is re-armed after the solve).
template <typename Raw, int NC, bool LAZY>
struct RawSrc {
  Raw regs[LAZY ? 1 : NC];
  const Raw* slot;  // LAZY: camera c at slot[c * BATCH_THREADS]
  __device__ __forceinline__ Raw operator[](int c) const { if constexpr (LAZY) return slot[c * BATCH_THREADS]; else return regs[c]; }
};

// ---- tile interface of the streaming kernels ------------------------------------------------------
// A tile solver TS turns the raw pixels of FPT consecutive frames (one RawPix per camera) into points:
//     TS::FPT, TS::Rig (a __grid_constant__ parameter), TS::Real (the arithmetic type of the result)
//     TS::run<NC, PIX, WIDE>(rig, raw, opt, X, mask, err, iters)
// WIDE is a compile-time switch for the optional outputs of tri_batch_out (double3 points, the `error` of
// triangulatePoint, LM iterations): the lean instantiation (float3 + mask) is what the throughput metric runs,
// the wide one serves the C++ adapter, whose interface returns cv::Point3d (Triangulator.h:51-52).

// A tile's mask output is its frames' validity bits -- the too-few latch counts them -- unless the tile declares
// MASK_IS_VALIDITY = false (the robust tile: mask = the inlier set, `iters` carries the number of valid views).
template <class TS, class = void>
struct MaskIsValidity { static constexpr bool value = true; };
template <class TS>
struct MaskIsValidity<TS, std::void_t<decltype(TS::MASK_IS_VALIDITY)>> { static constexpr bool value = TS::MASK_IS_VALIDITY; };

// ---- barrier-free per-thread async pipeline ---------------------------------------------------------
// Nothing synchronises across warps: every thread prefetches ITS OWN pixels of the next STAGES tiles with
// cp.async (LDGSTS, 16 B per camera row, fully coalesced per warp) into a private shared-memory slot, waits only
// on its own cp.async group, pulls the slot into registers, re-arms it, and solves.  Warps drift apart freely, so
// one warp's memory wait hides under another warp's FMAs.  The 12-byte points are transposed through a
// per-warp shared tile (__syncwarp only) into coalesced 16-byte streaming stores.  (Measured against it in round
// 1 and dropped: one tile per CTA with up-front vector loads, and a CTA-synchronous TMA ring -- profiles/r1_*.)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// the optional per-frame outputs of FPT consecutive frames starting at f0 (per-thread stores; a warp covers a
// contiguous range, so every sector is fully written)
template <int FPT, typename Real>
__device__ __forceinline__ void store_wide(const BatchOut& out, int64_t f0, const Real (&X)[FPT][3], const double (&err)[FPT],
                                           const int (&iters)[FPT]) {
  if (out.xyz_f64) {
    double* o = out.xyz_f64 + 3 * f0;
    if constexpr (FPT == 2) {  // 48 B, 16-byte aligned (f0 is even)
      double2* o2 = reinterpret_cast<double2*>(o);
      o2[0] = make_double2((double)X[0][0], (double)X[0][1]); o2[1] = make_double2((double)X[0][2], (double)X[1][0]);
      o2[2] = make_double2((double)X[1][1], (double)X[1][2]);
    } else {
      o[0] = (double)X[0][0]; o[1] = (double)X[0][1]; o[2] = (double)X[0][2];
    }
  }
  if (out.err) {
    if constexpr (FPT == 2) reinterpret_cast<double2*>(out.err)[f0 / 2] = make_double2(err[0], err[1]);
    else out.err[f0] = err[0];
  }
  if (out.iters) {
    if constexpr (FPT == 2) reinterpret_cast<int2*>(out.iters)[f0 / 2] = make_int2(iters[0], iters[1]);
    else out.iters[f0] = iters[0];
  }
}

template <class TS, int NC, int PIX, int STAGES, int MINB, bool WIDE, bool LAZY = false>
__global__ void __launch_bounds__(BATCH_THREADS, WIDE ? 1 : MINB)  // the wide instantiation keeps the pixels live for the error pass
stream_kernel(const __grid_constant__ typename TS::Rig rig, const char* __restrict__ xy, int64_t row_bytes, int64_t n_tiles,
              BatchOut out, int opt, unsigned long long* first_bad, int64_t frame_base) {
  constexpr int FPT = TS::FPT;
  using Raw = typename RawPix<PIX, FPT>::type;
  using Real = typename TS::Real;
  constexpr int TILE = BATCH_THREADS * FPT;
  constexpr int RB = (int)sizeof(Raw);  // bytes per thread per camera per tile
  extern __shared__ __align__(128) unsigned char smem[];
  // layout: [STAGES][NC][BATCH_THREADS] Raw | [warps][32 * FPT * 3] float
  Raw* slots = reinterpret_cast<Raw*>(smem);
  float* outw = reinterpret_cast<float*>(smem + STAGES * NC * BATCH_THREADS * RB) + (threadIdx.x >> 5) * (32 * FPT * 3);
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t stride = gridDim.x;
  int64_t tile = blockIdx.x;

  auto prefetch = [&](int s, int64_t t) {
    const char* src = xy + (t * BATCH_THREADS + tid) * RB;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      Raw* dst = slots + (s * NC + c) * BATCH_THREADS + tid;
      if constexpr (RB == 16) cp_async16(dst, src + c * row_bytes);
      else if constexpr (RB == 8) cp_async8(dst, src + c * row_bytes);
      else cp_async4(dst, src + c * row_bytes);
    }
  };
#pragma unroll
  for (int s = 0; s < STAGES; s++) {
    if (tile + s * stride < n_tiles) prefetch(s, tile + s * stride);
    cp_async_commit();
  }

  for (int k = 0; tile < n_tiles; k++, tile += stride) {
    const int s = k % STAGES;
    cp_async_wait<STAGES - 1>();  // this thread's copies for tile k have landed
    RawSrc<Raw, NC, LAZY> raw;
    if constexpr (LAZY) {
      raw.slot = slots + (size_t)s * NC * BATCH_THREADS + tid;
    } else {
#pragma unroll
      for (int c = 0; c < NC; c++) raw.regs[c] = slots[(s * NC + c) * BATCH_THREADS + tid];
      if (tile + STAGES * stride < n_tiles) prefetch(s, tile + STAGES * stride);
      cp_async_commit();
    }

    Real X[FPT][3];
    uint32_t mask[FPT];
    double err[FPT];
    int iters[FPT];
    TS::template run<NC, PIX, WIDE>(rig, raw, opt, X, mask, err, iters);
    if constexpr (LAZY) {  // the slot is free only now
      if (tile + STAGES * stride < n_tiles) prefetch(s, tile + STAGES * stride);
      cp_async_commit();
    }

    const int64_t f0 = tile * TILE + (int64_t)tid * FPT;
#pragma unroll
    for (int j = 0; j < FPT; j++)
      if ((MaskIsValidity<TS>::value ? __popc(mask[j]) : iters[j]) < 2) atomicMin(first_bad, (unsigned long long)(frame_base + f0 + j));
    if (out.mask) {
      if constexpr (FPT == 2) reinterpret_cast<uint2*>(out.mask)[f0 / 2] = make_uint2(mask[0], mask[1]);
      else out.mask[f0] = mask[0];
    }
    if constexpr (WIDE) {
      store_wide<FPT, Real>(out, f0, X, err, iters);
      if (!out.xyz_f32) continue;  // uniform
    }
    // warp-level transpose: 32 x FPT x 12 B contiguous in global memory
    __syncwarp();  // the previous tile's reads of this warp's tile are done
    if constexpr (FPT == 2) {
      float2* o2 = reinterpret_cast<float2*>(outw) + 3 * lane;
      o2[0] = make_float2((float)X[0][0], (float)X[0][1]); o2[1] = make_float2((float)X[0][2], (float)X[1][0]);
      o2[2] = make_float2((float)X[1][1], (float)X[1][2]);
    } else {
      outw[3 * lane] = (float)X[0][0]; outw[3 * lane + 1] = (float)X[0][1]; outw[3 * lane + 2] = (float)X[0][2];
    }
    __syncwarp();
    float4* dst = reinterpret_cast<float4*>(out.xyz_f32 + 3 * (tile * TILE + (int64_t)(tid - lane) * FPT));
    const float4* src4 = reinterpret_cast<const float4*>(outw);
    constexpr int N4 = 32 * FPT * 3 / 4;  // 24 or 48 float4 per warp
#pragma unroll
    for (int i = lane; i < N4; i += 32) __stcs(dst + i, src4[i]);
  }
  cp_async_wait<0>();
}

// which optional outputs the caller wants -> the WIDE instantiation; alignment of whatever is written
static inline bool wants_wide(const BatchOut& out) { return out.xyz_f64 || out.err || out.iters; }
static inline bool stream_aligned(const void* xy, int64_t row_bytes, int align, const BatchOut& out) {
  return !(((uintptr_t)xy % align) || (row_bytes % align) || ((uintptr_t)out.xyz_f32 & 15) || ((uintptr_t)out.xyz_f64 & 15) ||
           ((uintptr_t)out.mask & 7) || ((uintptr_t)out.err & 15) || ((uintptr_t)out.iters & 7));
}

// LAZY: the pixels are read from the slot as the solve needs them (RawSrc) instead of pulled into registers on arrival
template <class TS, int PIX, int STAGES, int MINB, bool WIDE, bool LAZY>
static cudaError_t launch_stream_w(const LaunchCtx& ctx, const typename TS::Rig& rig, const char* xy, int n_use, int64_t n_tiles,
                                   int64_t row_bytes, const BatchOut& out, int opt) {
  constexpr int FPT = TS::FPT;
  using Raw = typename RawPix<PIX, FPT>::type;
  cudaError_t err = cudaSuccess;
#define TRI_CASE(N)                                                                                                     \
  case N: {                                                                                                             \
    auto kern = stream_kernel<TS, N, PIX, STAGES, MINB, WIDE, LAZY>;                                                    \
    constexpr int bytes = STAGES * N * BATCH_THREADS * (int)sizeof(Raw) + (BATCH_THREADS / 32) * 32 * FPT * 12;          \
    err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);                               \
    if (err != cudaSuccess) return err;                                                                                 \
    int per_sm = 1;                                                                                                     \
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, BATCH_THREADS, bytes);                           \
    if (err != cudaSuccess) return err;                                                                                 \
    const int64_t grid = std::min<int64_t>(n_tiles, (int64_t)ctx.sm_count * std::max(per_sm, 1));                       \
    kern<<<(unsigned)grid, BATCH_THREADS, bytes, ctx.stream>>>(rig, xy, row_bytes, n_tiles, out, opt, ctx.d_first_bad,  \
                                                         ctx.frame_base);                                               \
  } break;
  switch (n_use) { TRI_CASE(2) TRI_CASE(3) TRI_CASE(4) TRI_CASE(5) TRI_CASE(6) TRI_CASE(7) TRI_CASE(8) }
#undef TRI_CASE
  ++*ctx.launches;
  return cudaGetLastError();
}

// Launch the streaming kernel on the full tiles of [0, n_frames); *covered = the number of frames it took
// (0 if the layout does not qualify: unaligned rows or outputs, fewer frames than a tile).
template <class TS, int PIX, int STAGES, int MINB, bool LAZY = false>
static cudaError_t launch_stream(const LaunchCtx& ctx, const typename TS::Rig& rig, const void* d_xy, int n_use, int64_t n_frames,
                                 int64_t cam_stride, const BatchOut& out, int opt, int64_t* covered) {
  *covered = 0;
  constexpr int TILE = BATCH_THREADS * TS::FPT;
  using Raw = typename RawPix<PIX, TS::FPT>::type;
  const char* xy = static_cast<const char*>(d_xy);
  const int64_t row_bytes = cam_stride * pix_bytes(PIX);
  const int64_t n_tiles = n_frames / TILE;
  if (n_tiles == 0 || n_use < 2 || n_use > 8) return cudaSuccess;
  if (!stream_aligned(xy, row_bytes, (int)sizeof(Raw), out)) return cudaSuccess;
  const cudaError_t err = wants_wide(out) ? launch_stream_w<TS, PIX, STAGES, MINB, true, LAZY>(ctx, rig, xy, n_use, n_tiles, row_bytes, out, opt)
                                          : launch_stream_w<TS, PIX, STAGES, MINB, false, LAZY>(ctx, rig, xy, n_use, n_tiles, row_bytes, out, opt);
  if (err == cudaSuccess) *covered = n_tiles * TILE;
  return err;
}

// ---- more than 8 cameras: the same barrier-free pipeline over (tile, camera chunk) units -----------
// The generic batch_kernel indexes the rig with a runtime camera number, so every constant is an LDC (the ADU
// pipe then bounds the ray kernels: 22 constants per view) and nothing is prefetched.  Here a tile's cameras are
// walked in chunks of 8 with the accumulators carried in registers: one pipeline unit = 8 camera rows of one
// tile, the chunk number selects one of four fully unrolled bodies, so every camera index is static again and
// the constants come through uniform registers.
constexpr int CHUNK_CAMS = 8;

template <class S, int C0, int PIX, int FPT>
__device__ __forceinline__ void chunk_accumulate(const typename S::Rig& rig, const typename RawPix<PIX, FPT>::type (&raw)[CHUNK_CAMS],
                                                 int n_use, typename S::Acc (&acc)[FPT], uint32_t (&mask)[FPT]) {
  using T = typename S::T;
  if (C0 + CHUNK_CAMS <= n_use) {  // a full chunk: no per-camera test, so the views of the chunk can overlap
#pragma unroll
    for (int c = 0; c < CHUNK_CAMS; c++) {
      const Views<T, PIX, FPT> w = decode<T, PIX, FPT>(raw[c]);
#pragma unroll
      for (int j = 0; j < FPT; j++) { S::add_chunk(rig, C0 + c, w.x[j], w.y[j], w.v[j], acc[j]); mask[j] |= (w.v[j] ? 1u : 0u) << (C0 + c); }
    }
  } else {
#pragma unroll
    for (int c = 0; c < CHUNK_CAMS; c++) {
      if (C0 + c < n_use) {  // uniform
        const Views<T, PIX, FPT> w = decode<T, PIX, FPT>(raw[c]);
#pragma unroll
        for (int j = 0; j < FPT; j++) { S::add_chunk(rig, C0 + c, w.x[j], w.y[j], w.v[j], acc[j]); mask[j] |= (w.v[j] ? 1u : 0u) << (C0 + c); }
      }
    }
  }
}

template <class S, int PIX, int FPT, int STAGES, int MINB, bool WIDE>
__global__ void __launch_bounds__(BATCH_THREADS, MINB)
chunk_kernel(const __grid_constant__ typename S::Rig rig, const char* __restrict__ xy, int64_t row_bytes, int64_t n_tiles, int n_use,
             BatchOut out, int opt, unsigned long long* first_bad, int64_t frame_base) {
  using T = typename S::T;
  using Raw = typename RawPix<PIX, FPT>::type;
  constexpr int TILE = BATCH_THREADS * FPT;
  constexpr int RB = (int)sizeof(Raw);
  extern __shared__ __align__(128) unsigned char smem[];
  // layout: [STAGES][CHUNK_CAMS][BATCH_THREADS] Raw | [warps][32 * FPT * 3] float
  Raw* slots = reinterpret_cast<Raw*>(smem);
  float* outw = reinterpret_cast<float*>(smem + STAGES * CHUNK_CAMS * BATCH_THREADS * RB) + (threadIdx.x >> 5) * (32 * FPT * 3);
  const int tid = threadIdx.x, lane = tid & 31;
  const int n_chunks = (n_use + CHUNK_CAMS - 1) / CHUNK_CAMS;
  // this CTA's units: tiles blockIdx.x, + gridDim.x, ...; each tile = n_chunks consecutive units
  const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t my_units = my_tiles * n_chunks;

  auto prefetch = [&](int s, int64_t u) {
    const int64_t t = blockIdx.x + (u / n_chunks) * gridDim.x;
    const int ch = (int)(u % n_chunks);
    const char* src = xy + (t * BATCH_THREADS + tid) * RB + (int64_t)ch * CHUNK_CAMS * row_bytes;
#pragma unroll
    for (int c = 0; c < CHUNK_CAMS; c++) {
      if (ch * CHUNK_CAMS + c < n_use) {
        Raw* dst = slots + (s * CHUNK_CAMS + c) * BATCH_THREADS + tid;
        if constexpr (RB == 16) cp_async16(dst, src + c * row_bytes);
        else if constexpr (RB == 8) cp_async8(dst, src + c * row_bytes);
        else cp_async4(dst, src + c * row_bytes);
      }
    }
  };
#pragma unroll
  for (int s = 0; s < STAGES; s++) {
    if (s < my_units) prefetch(s, s);
    cp_async_commit();
  }

  typename S::Acc acc[FPT];
  uint32_t mask[FPT];
  int ch = 0;
  int64_t tile = blockIdx.x;
  for (int64_t u = 0; u < my_units; u++) {
    const int s = (int)(u % STAGES);
    cp_async_wait<STAGES - 1>();
    Raw raw[CHUNK_CAMS];
#pragma unroll
    for (int c = 0; c < CHUNK_CAMS; c++) raw[c] = slots[(s * CHUNK_CAMS + c) * BATCH_THREADS + tid];
    if (u + STAGES < my_units) prefetch(s, u + STAGES);
    cp_async_commit();

    if (ch == 0) {
#pragma unroll
      for (int j = 0; j < FPT; j++) { acc[j] = typename S::Acc(); mask[j] = 0; }
    }
    switch (ch) {
      case 0: chunk_accumulate<S, 0, PIX, FPT>(rig, raw, n_use, acc, mask); break;
      case 1: chunk_accumulate<S, 8, PIX, FPT>(rig, raw, n_use, acc, mask); break;
      case 2: chunk_accumulate<S, 16, PIX, FPT>(rig, raw, n_use, acc, mask); break;
      default: chunk_accumulate<S, 24, PIX, FPT>(rig, raw, n_use, acc, mask); break;
    }
    if (++ch < n_chunks) continue;
    ch = 0;

    T X[FPT][3];
    double err[FPT];
    int iters[FPT];
#pragma unroll
    for (int j = 0; j < FPT; j++) {
      X[j][0] = X[j][1] = X[j][2] = 0;
      err[j] = 0;
      iters[j] = 0;
      if (__popc(mask[j]) >= 2) { S::solve(rig, acc[j], mask[j], __popc(mask[j]), X[j], opt, iters[j]); S::to_world(rig, X[j]); }
    }
    const int64_t f0 = tile * TILE + (int64_t)tid * FPT;
    const int64_t warp_f0 = tile * TILE + (int64_t)(tid - lane) * FPT;
    tile += gridDim.x;
#pragma unroll
    for (int j = 0; j < FPT; j++)
      if (__popc(mask[j]) < 2) atomicMin(first_bad, (unsigned long long)(frame_base + f0 + j));
    if (out.mask) {
      if constexpr (FPT == 2) reinterpret_cast<uint2*>(out.mask)[f0 / 2] = make_uint2(mask[0], mask[1]);
      else out.mask[f0] = mask[0];
    }
    if constexpr (WIDE) {  // double3 points / iterations (the `error` output needs the pixels again: generic kernel)
      store_wide<FPT, T>(out, f0, X, err, iters);
      if (!out.xyz_f32) continue;
    }
    __syncwarp();
    if constexpr (FPT == 2) {
      float2* o2 = reinterpret_cast<float2*>(outw) + 3 * lane;
      o2[0] = make_float2((float)X[0][0], (float)X[0][1]); o2[1] = make_float2((float)X[0][2], (float)X[1][0]);
      o2[2] = make_float2((float)X[1][1], (float)X[1][2]);
    } else {
      outw[3 * lane] = (float)X[0][0]; outw[3 * lane + 1] = (float)X[0][1]; outw[3 * lane + 2] = (float)X[0][2];
    }
    __syncwarp();
    float4* dst = reinterpret_cast<float4*>(out.xyz_f32 + 3 * warp_f0);
    const float4* src4 = reinterpret_cast<const float4*>(outw);
    constexpr int N4 = 32 * FPT * 3 / 4;
#pragma unroll
    for (int i = lane; i < N4; i += 32) __stcs(dst + i, src4[i]);
  }
  cp_async_wait<0>();
}

template <class S, int PIX, int FPT, int STAGES, int MINB>
static cudaError_t launch_chunk(const LaunchCtx& ctx, const typename S::Rig& rig, const void* d_xy, int n_use, int64_t n_frames,
                                int64_t cam_stride, const BatchOut& out, int opt, int64_t* covered) {
  *covered = 0;
  constexpr int TILE = BATCH_THREADS * FPT;
  using Raw = typename RawPix<PIX, FPT>::type;
  const char* xy = static_cast<const char*>(d_xy);
  const int64_t row_bytes = cam_stride * pix_bytes(PIX);
  const int64_t n_tiles = n_frames / TILE;
  if (n_tiles == 0 || n_use <= CHUNK_CAMS || n_use > 4 * CHUNK_CAMS) return cudaSuccess;
  if (out.err) return cudaSuccess;
  if (!stream_aligned(xy, row_bytes, (int)sizeof(Raw), out)) return cudaSuccess;
  constexpr int bytes = STAGES * CHUNK_CAMS * BATCH_THREADS * (int)sizeof(Raw) + (BATCH_THREADS / 32) * 32 * FPT * 12;
  auto go = [&](auto kern) -> cudaError_t {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (err != cudaSuccess) return err;
    int per_sm = 1;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, BATCH_THREADS, bytes);
    if (err != cudaSuccess) return err;
    const int64_t grid = std::min<int64_t>(n_tiles, (int64_t)ctx.sm_count * std::max(per_sm, 1));
    kern<<<(unsigned)grid, BATCH_THREADS, bytes, ctx.stream>>>(rig, xy, row_bytes, n_tiles, n_use, out, opt, ctx.d_first_bad, ctx.frame_base);
    return cudaGetLastError();
  };
  const cudaError_t err = wants_wide(out) ? go(chunk_kernel<S, PIX, FPT, STAGES, MINB, true>) : go(chunk_kernel<S, PIX, FPT, STAGES, MINB, false>);
  if (err != cudaSuccess) return err;
  ++*ctx.launches;
  *covered = n_tiles * TILE;
  return cudaSuccess;
}

// Sub-range helper for the tail after the pipelined tiles.
inline BatchOut advance(const BatchOut& o, int64_t frames) {
  BatchOut r = o;
  if (r.xyz_f32) r.xyz_f32 += 3 * frames;
  if (r.xyz_f64) r.xyz_f64 += 3 * frames;
  if (r.mask) r.mask += frames;
  if (r.err) r.err += frames;
  if (r.iters) r.iters += frames;
  return r;
}


// streaming kernel on the full tiles, the scalar policy kernel on whatever is left (tails, unaligned rows)
template <class TS, class S, int PIX, int FPT, int STAGES, int MINB, bool LAZY = false>
static cudaError_t launch_streamed(const LaunchCtx& ctx, const typename TS::Rig& tile_rig, const typename S::Rig& rig,
                                   const void* d_xy, int n_use, int64_t n_frames, int64_t cam_stride, const BatchOut& out, int opt) {
  int64_t covered = 0;
  if constexpr (PIX != PIX_F64) {
    cudaError_t err;
    if (S::CHUNKED && n_use > CHUNK_CAMS)  // 9..32 cameras: camera-chunked pipeline over the scalar policy
      err = launch_chunk<S, PIX, S::CHUNK_FPT, 3, 2>(ctx, rig, d_xy, n_use, n_frames, cam_stride, out, opt, &covered);
    else
      err = launch_stream<TS, PIX, STAGES, MINB, LAZY>(ctx, tile_rig, d_xy, n_use, n_frames, cam_stride, out, opt, &covered);
    if (err != cudaSuccess || covered == n_frames) return err;
  }
  LaunchCtx rest = ctx;
  rest.frame_base += covered;
  return launch_batch_policy<S, PIX, FPT, (MINB > 3 ? 3 : MINB)>(rest, rig, static_cast<const char*>(d_xy) + covered * pix_bytes(PIX), n_use,
                                                n_frames - covered, cam_stride, advance(out, covered), opt);
}

}  // namespace tri
