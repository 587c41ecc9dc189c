// tri_classify.cu -- kernel 3: DroneClassifier::classifyDrones (src/DroneClassifier.cpp:96-332) as two
// kernels.  Compiled with -fmad=false: every compare that decides an index (error_ pruning, the
// MAX_STEP gates, the priority order) is evaluated in the reference's operation order.
//
// (A) enumerate_kernel -- frame-parallel.  fillCombinationQueue (:156-198) walks a tree whose level c
//     picks, for camera c, "none" (0) or detection k (1..n_c); every node with >= 2 detections is
//     triangulated and its subtree cut when error > error_ (:185-187); complete nodes with
//     >= MIN_CAMERAS detections are the candidate combinations (:190-196).  Whether a node survives
//     depends only on its own prefix, so the tree is expanded level-synchronously: one CTA owns a
//     frame, a level's children are evaluated one per thread and compacted IN ORDER (ballot + scan),
//     which reproduces the reference's DFS order of the leaves (lexicographic in the per-camera
//     choices).  A combination is one 64-bit word, 4 bits per camera.  The gated enumerations of
//     triangulateWithLastPos (:219-250) are subsets of this full-frame leaf list (same prefixes, same
//     pixels => same errors), so the tree is expanded ONCE per frame instead of once per path.
// (B) link_kernel -- frame-sequential (the reference's tracking state: last position + 3-point tail
//     per path, :119-135, :269-297).  One CTA walks the frames in order; per path it evaluates the
//     MAX_STEP ray gate of every detection in parallel, then takes the arg-min over the admissible
//     leaves of the key (fewest unused cameras, smallest error, DFS order) -- the first element the
//     reference's priority_queue would pop that passes :241-246.  Phase 2 (pickBestCombinations +
//     classifyPaths, :200-217, :262-332) is the same arg-min repeated greedily, then the tiny
//     path-assignment logic on one thread.  Ties on (unused cameras, error) are broken by DFS order
//     (the reference's heap order is an artefact of libstdc++); they are counted in stats.ties.
#include <float.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "tri_classify.cuh"

namespace tri {

// ---- (A) candidate generation ------------------------------------------------------------------
__global__ void __launch_bounds__(CLS_THREADS, TRI_ENUM_MIN_CTAS)
enumerate_kernel(const __grid_constant__ DltRig<double> dlt, const __grid_constant__ RayRig ray, ClsParams p,
                 const int32_t* __restrict__ offs, const double* __restrict__ dets, u64* __restrict__ front,
                 double* __restrict__ tmp_xyz, double* __restrict__ tmp_err, u64* __restrict__ leaf_rec,
                 long long* __restrict__ leaf_off, int* __restrict__ leaf_cnt, int* __restrict__ hdr,
                 unsigned char* __restrict__ fdet, long long* __restrict__ fdet_off, int* __restrict__ fdet_cnt, unsigned* __restrict__ sort_kb,
                 ClsCounters* ctr) {
  __shared__ int s_n[CLS_MAX_CAMS], s_pref[CLS_MAX_CAMS + 1], s_hist[CLS_MAX_CAMS + 2];
  __shared__ long long s_doff;
  __shared__ double s_px[CLS_MAX_CAMS][TRI_MAX_DETS], s_py[CLS_MAX_CAMS][TRI_MAX_DETS];
  __shared__ int s_warp[CLS_THREADS / 32];
  __shared__ long long s_off;
  extern __shared__ __align__(16) unsigned char enum_dyn[];  // the sort keys of a frame's leaves
  u64* s_ka = reinterpret_cast<u64*>(enum_dyn);                   // error bits
  unsigned* s_kb = reinterpret_cast<unsigned*>(s_ka + ENUM_SORT_CAP);  // (unused cameras, DFS index)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = p.n_cams;
  __shared__ double s_P[CLS_MAX_CAMS][12];  // the projection matrices: every thread solves a different camera subset
  for (int i = tid; i < C * 12; i += CLS_THREADS) s_P[i / 12][i % 12] = dlt.P[i / 12][i % 12];
  u64* buf0 = front + (size_t)blockIdx.x * 2 * p.cap;
  u64* buf1 = buf0 + p.cap;
  double* t_xyz = tmp_xyz + (size_t)blockIdx.x * 3 * p.cap;
  double* t_err = tmp_err + (size_t)blockIdx.x * p.cap;
  u64 st_nodes = 0, st_solves = 0, st_iters = 0;

  // Frames are handed out one at a time (their cost varies by orders of magnitude with the number of detections): the
  // first round by block index, then from a shared counter.
  __shared__ int s_frame;
  for (int f = p.f0 + blockIdx.x; f < p.f1;) {
    __syncthreads();
    for (int i = tid; i < C * TRI_MAX_DETS; i += CLS_THREADS) {
      const int c = i / TRI_MAX_DETS, d = i % TRI_MAX_DETS;
      const int a = offs[(size_t)c * (p.n_frames + 1) + f], b = offs[(size_t)c * (p.n_frames + 1) + f + 1];
      if (d == 0) {
        s_n[c] = min(b - a, TRI_MAX_DETS);
        if (b - a > TRI_MAX_DETS || b < a) atomicExch(&ctr->bad_input, 1);
      }
      if (d < b - a) { s_px[c][d] = dets[2 * (size_t)(a + d)]; s_py[c][d] = dets[2 * (size_t)(a + d) + 1]; }
    }
    __syncthreads();  // s_n is complete
    if (tid == 0) {
      buf0[0] = 0;
      int n = 0;
      for (int c = 0; c < C; c++) { s_pref[c] = n; n += s_n[c]; }
      s_pref[C] = n;
      s_doff = (long long)atomicAdd(&ctr->fdet_total, (u64)n);  // the buffer holds every detection of the batch: no overflow
      fdet_off[f - p.f0] = s_doff;
      fdet_cnt[f - p.f0] = n;
    }
    __syncthreads();
    // the frame's detections with their pixel rays, camera-major, as the block the linking pass stages: n x float4 (origin, dir.x),
    // n x float4 (dir.y, dir.z, camera), n x 4 doubles (dir): it gates them against every path
    {
      const int n = s_pref[C];
      float4* A = reinterpret_cast<float4*>(fdet + (size_t)s_doff * FDET_BYTES);
      float4* B = A + n;
      double* Dd = reinterpret_cast<double*>(B + n);
      for (int i = tid; i < C * TRI_MAX_DETS; i += CLS_THREADS) {
        const int c = i / TRI_MAX_DETS, d = i % TRI_MAX_DETS;
        if (d < s_n[c]) {
          double dir[3];
          ref::make_dir(ray, c, s_px[c][d], s_py[c][d], dir);
          const int k = s_pref[c] + d;
          A[k] = make_float4((float)ray.pos[c][0], (float)ray.pos[c][1], (float)ray.pos[c][2], (float)dir[0]);
          B[k] = make_float4((float)dir[1], (float)dir[2], __int_as_float(c), 0.f);
          Dd[4 * k] = dir[0]; Dd[4 * k + 1] = dir[1]; Dd[4 * k + 2] = dir[2]; Dd[4 * k + 3] = 0;
        }
      }
    }
    u64 *fin = buf0, *fout = buf1;
    int m = 1;
    for (int c = 0; c < C && m > 0; c++) {
      const int nch = s_n[c] + 1;
      const int total = m * nch;
      const bool last = c == C - 1;
      int out_base = 0;
      for (int j0 = 0; j0 < total; j0 += CLS_THREADS) {
        const int j = j0 + tid;
        bool keep = false;
        u64 comb = 0;
        double X[3] = {0, 0, 0}, err = 0;
        if (j < total) {
          const int parent = j / nch, k = j - parent * nch;
          comb = fin[parent] | ((u64)k << (4 * c));
          const int cnt = __popcll(nonzero_nibbles(comb));
          keep = true;
          st_nodes++;
          if (cnt >= 2) st_solves++;  // the reference re-solves the "none" children too (:166-181)
          if (cnt >= 2 && (k > 0 || last)) {  // a "none" child repeats its parent's subset: same error
            int it;
            err = solve_combination(s_P, ray, p.solver, comb, c + 1, s_px, s_py, X, it);
            st_iters += it;
            if (err > p.error_) keep = false;  // :185-187
          }
          if (last && cnt < MIN_CAMERAS) keep = false;  // complete but too few detections: no candidate
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(ballot);
        __syncthreads();
        int before = 0, chunk = 0;
#pragma unroll
        for (int w = 0; w < CLS_THREADS / 32; w++) {
          if (w < warp) before += s_warp[w];
          chunk += s_warp[w];
        }
        const int pos = out_base + before + __popc(ballot & ((1u << lane) - 1));
        if (keep) {
          if (pos < p.cap) {
            fout[pos] = comb;
            if (last) { t_xyz[3 * pos] = X[0]; t_xyz[3 * pos + 1] = X[1]; t_xyz[3 * pos + 2] = X[2]; t_err[pos] = err; }
          } else {
            atomicExch(&ctr->overflow_frontier, 1);
          }
        }
        out_base += chunk;
        __syncthreads();
      }
      m = min(out_base, p.cap);
      if (tid == 0) atomicMax(&ctr->max_frontier, out_base);
      u64* t = fin; fin = fout; fout = t;
      if (m == 0) break;
      if (last) {
        // publish this frame's leaves as records into a contiguous range of the global leaf array
        if (tid == 0) {
          long long off = (long long)atomicAdd(&ctr->leaf_total, (u64)m);
          if (off + m > p.leaf_cap) { atomicExch(&ctr->overflow_leaves, 1); off = -1; }
          s_off = off;
        }
        for (int i = tid; i < CLS_MAX_CAMS + 2; i += CLS_THREADS) s_hist[i] = 0;
        __syncthreads();
        const long long off = s_off;
        if (off >= 0) {
          // ... in PRIORITY order: the order in which the reference's priority_queue pops them = fewer unused cameras first,
          // then smaller error (Combination::operator<, :12-20), ties by DFS order.  The errors are >= +0, so their bit
          // patterns order like the values: the leaves are sorted by (unused cameras, error bits, DFS index) with a bitonic
          // network (round 1 ranked by counting, O(m^2): three quarters of this kernel's time).
          const u64 cam_bits = C == 16 ? ~0ull : ((1ull << (4 * C)) - 1);
          const int RW = rec_words(p.W);
          u64 n_tie = 0;
          auto publish = [&](int i, int rank, u64 ci, double ei) {  // leaf i is the rank-th to be popped
            // the frame's block: m masks of W words, then m x (point, combination)
            u64* mrow = leaf_rec + (size_t)off * RW + (size_t)rank * p.W;
            u64* prow = leaf_rec + (size_t)off * RW + (size_t)m * p.W + (size_t)rank * 4;
            u64 mk[4] = {0, 0, 0, 0};
            for (int c = 0; c < C; c++) {
              const int k = (int)((ci >> (4 * c)) & 15);
              if (k) { const int bit = s_pref[c] + k - 1; mk[bit >> 6] |= 1ull << (bit & 63); }
            }
            if (!(ei < p.error_)) mk[p.W - 1] |= 1ull << 63;  // poison: a leaf (:185-196) that no acceptance test passes (:209, :243)
            for (int w = 0; w < p.W; w++) mrow[w] = mk[w];
            prow[0] = (u64)__double_as_longlong(t_xyz[3 * i]);
            prow[1] = (u64)__double_as_longlong(t_xyz[3 * i + 1]);
            prow[2] = (u64)__double_as_longlong(t_xyz[3 * i + 2]);
            prow[3] = ci;
          };
          // keys in shared memory, or -- a frame with more than ENUM_SORT_CAP leaves -- in this CTA's scratch in global memory
          // (the frontier buffer that is free after the last level; __syncthreads orders the CTA's global accesses as well)
          auto sort_and_publish = [&](u64* ka, unsigned* kb) {
            int n = 2;
            while (n < m) n <<= 1;
            for (int i = tid; i < n; i += CLS_THREADS) {
              if (i < m) {
                const int zi = C - __popcll(nonzero_nibbles(fin[i] & cam_bits));
                ka[i] = (u64)__double_as_longlong(t_err[i]);
                kb[i] = ((unsigned)zi << ENUM_IDX_BITS) | (unsigned)i;
                atomicAdd(&s_hist[zi + 1], 1);
              } else {
                ka[i] = ~0ull; kb[i] = ~0u;  // padding sorts last
              }
            }
            __syncthreads();
            for (int k = 2; k <= n; k <<= 1)
              for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < (n >> 1); t += CLS_THREADS) {
                  const int lo = 2 * t - (t & (j - 1)), hi = lo + j;  // the t-th pair of this step
                  const u64 a = ka[lo], b = ka[hi];
                  const unsigned ab = kb[lo], bb = kb[hi];
                  const unsigned za = ab >> ENUM_IDX_BITS, zb = bb >> ENUM_IDX_BITS;
                  const bool a_after_b = za != zb ? za > zb : (a != b ? a > b : ab > bb);
                  if (a_after_b == ((lo & k) == 0)) { ka[lo] = b; ka[hi] = a; kb[lo] = bb; kb[hi] = ab; }
                }
                __syncthreads();
              }
            for (int r = tid; r < m; r += CLS_THREADS) {
              const u64 a = ka[r];
              const unsigned ab = kb[r], z = ab >> ENUM_IDX_BITS;
              const int i = (int)(ab & ((1u << ENUM_IDX_BITS) - 1));
              n_tie += (r > 0 && ka[r - 1] == a && (kb[r - 1] >> ENUM_IDX_BITS) == z) ||
                       (r + 1 < m && ka[r + 1] == a && (kb[r + 1] >> ENUM_IDX_BITS) == z);
              publish(i, r, fin[i], __longlong_as_double((long long)a));
            }
          };
          if (m <= ENUM_SORT_CAP) sort_and_publish(s_ka, s_kb);
          else sort_and_publish(fout, sort_kb + (size_t)blockIdx.x * p.cap);
          if (n_tie) atomicAdd(&ctr->ties, n_tie);
          __syncthreads();
          if (tid == 0) {
            leaf_off[f - p.f0] = off; leaf_cnt[f - p.f0] = m; atomicAdd(&ctr->leaves, (u64)m);
            int run = 0;
            int* zs = hdr + (size_t)(f - p.f0) * HDR_INTS;
            for (int z = 0; z <= C + 1; z++) { run += s_hist[z]; zs[z] = run; }  // zs[z] = leaves with fewer than z unused cameras
            for (int c = 0; c <= C; c++) zs[HDR_PREF + c] = s_pref[c];
            *reinterpret_cast<long long*>(zs + HDR_OFF) = off;
          }
        } else if (tid == 0) {
          leaf_off[f - p.f0] = 0; leaf_cnt[f - p.f0] = 0;
        }
        m = -1;  // done
      }
    }
    if (m >= 0 && tid == 0) {  // the tree died out (or no cameras)
      leaf_off[f - p.f0] = 0; leaf_cnt[f - p.f0] = 0;
      for (int z = 0; z <= C + 1; z++) hdr[(size_t)(f - p.f0) * HDR_INTS + z] = 0;
      for (int c = 0; c <= C; c++) hdr[(size_t)(f - p.f0) * HDR_INTS + HDR_PREF + c] = s_pref[c];
    }
    if (tid == 0) s_frame = p.f0 + (int)gridDim.x + (int)atomicAdd(&ctr->next_frame, 1ull);
    __syncthreads();
    f = s_frame;
  }
  // block totals of the per-thread statistics
  for (int o = 16; o > 0; o >>= 1) {
    st_nodes += __shfl_down_sync(0xffffffffu, st_nodes, o);
    st_solves += __shfl_down_sync(0xffffffffu, st_solves, o);
    st_iters += __shfl_down_sync(0xffffffffu, st_iters, o);
  }
  if (lane == 0) { atomicAdd(&ctr->nodes, st_nodes); atomicAdd(&ctr->solves, st_solves); atomicAdd(&ctr->lm_iters, st_iters); }
}

// ---- (B) linking -------------------------------------------------------------------------------
// One CTA of sixteen warps per sequence; two block barriers per frame, plus one per kept combination when the frame has a
// phase 2.  Everything that does not depend on the tracking state was prepared by (A): the leaves in priority order -- their
// detection masks as one dense array, points + combination words as another --, the number of leaves per count of unused
// cameras, the frame's detections with their pixel rays.  A frame's leaves, detections and header arrive in shared memory
// as three bulk async copies (cp.async.bulk -> UBLKCP) that complete on an mbarrier, issued one frame ahead into the other
// buffer by the last warp (which also reads the frame table two frames ahead, off every other warp's path).  Per frame:
//   speculative phase 1, all tracked paths at once, LINK_WARPS / paths warps per path:
//     gate    the MAX_STEP ray gate (:228-236) with lane <-> detection: the ballot of one 32-detection test IS a slice
//             of the path's gate mask.  The distance runs in single precision first and in the reference's
//             double-precision operation order only where single precision cannot decide.  (Each warp of a path
//             computes the gate for itself: cheaper than handing it over.)
//     scan    the FIRST leaf (priority order) whose mask lies inside the gate and whose point is within MAX_STEP of the
//             path's last point (:241-246), ignoring earlier paths' picks; it starts at the first leaf with at least
//             as many unused cameras as the gate leaves empty; a warp tests 128 leaves per step, the warps of a path
//             take the 128-leaf blocks in turn and keep the smallest hit with a shared-memory atomicMin.
//   confirmation, every warp for itself (lane <-> path; the same registers in every warp, so nothing is handed over): if
//     the picks' masks are pairwise disjoint -- one OR-reduction against one sum of popcounts -- every pick is also the
//     first of the list filtered by the earlier paths' picks (:119-135).  Otherwise (404 of 14 738 picks on S09_D6)
//     warp 0 walks the paths in order, scans the colliding ones again with the used mask and publishes the result.
//   phase 2, pickBestCombinations (:200-217), the reference's pop loop in parallel: every warp keeps the masks of its
//     128-leaf blocks in registers; a round finds the first leaf of the whole list that misses the used mask (REDUX.MIN
//     in the warp, atomicMin across the warps, one block barrier), adds its mask to the used mask and strikes the leaves
//     it collides with.
//   classifyPaths (:262-332) on one warp (LINK_SERIAL_WARP), lane <-> kept combination: tail distances, nearest open path, then the ordered
//     assignment by warp-wide minimum extraction (three REDUX operations per step).  Phase 1's pushes run on the last warp
//     meanwhile: phase 2 and classifyPaths only touch the paths phase 1 did not serve.  (Both are warps that usually have
//     no path of their own to gate.)
// The kernel is one latency-bound CTA per sequence: what a frame costs is the length of its chain of dependent
// instructions (a lone warp issues one every 6-10 cycles here: LDS 30, VOTE 28, SHFL 33, REDUX 50 cycles, tools/micro/redux.cu;
// instruction fetch is not the limit, tools/micro/ifetch.cu).  Round 1 ran it with ~15 block barriers per frame, the pixel rays
// and the whole phase-2 filter inside (29 ms for S09_D6's 3000 frames); the steps since, and the variants that lost, are in
// profiles/r2_link_kernel.log.
__device__ __forceinline__ uint32_t cls_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cls_mbar_init(u64* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cls_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void cls_mbar_expect_tx(u64* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cls_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cls_mbar_wait(u64* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(cls_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void cls_bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, u64* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(cls_smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(cls_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ double dist3(const double* a, double bx, double by, double bz) {  // cv::norm(a - b)
  const double x = a[0] - bx, y = a[1] - by, z = a[2] - bz;
  return sqrt(x * x + y * y + z * z);
}
// sqrt(s) < MAX_STEP without the square root unless s is within rounding reach of MAX_STEP^2 (sqrt is monotonic and
// correctly rounded, so away from the boundary the two compares agree)
__device__ __forceinline__ bool sqrt_below_step(double s) {
  const double t = MAX_STEP * MAX_STEP;
  if (s < t * (1 - 1e-12)) return true;
  if (s > t * (1 + 1e-12)) return false;
  return sqrt(s) < MAX_STEP;
}

template <int W>
struct LinkLayout {
  static constexpr int RW = rec_words(W);
  static constexpr int MAX_LEAVES = W == 2 ? 1664 : 960;  // staged leaves per frame; longer lists are read from global memory
  static constexpr int REC_BYTES = MAX_LEAVES * RW * 8;
  static constexpr int DET_BYTES = LINK_MAX_DETS * FDET_BYTES;
  static constexpr int HDR_BYTES = HDR_INTS * 4;
  static constexpr int BUF_BYTES = REC_BYTES + DET_BYTES + HDR_BYTES;
  static constexpr int BYTES = 2 * BUF_BYTES + 16;  // + the two mbarriers
};

#ifndef TRI_LINK_WARPS
#define TRI_LINK_WARPS 16
#endif
constexpr int LINK_WARPS = TRI_LINK_WARPS;  // >= TRI_MAX_DRONES
constexpr int LINK_THREADS = 32 * LINK_WARPS;
constexpr int LINK_BLOCKS = 2 * LINK_WARPS;  // phase 2 holds the first LINK_BLOCKS x 128 leaves of a frame in registers, two blocks per warp (the rest is walked in place)
constexpr int LINK_NONE = 0x7fffffff;
constexpr int LINK_SERIAL_WARP = LINK_WARPS - 2;  // runs phase 2's bookkeeping and classifyPaths: a warp that usually has no path to gate (S09_D6 4.47 -> 4.43 us per frame against warp 0)

// ALL_STAGED: no frame of the batch has more than MAX_LEAVES leaves (the host knows the longest list), so the body that reads
// leaves from global memory is not even compiled in -- the kernel is latency-bound on one SM and its instruction footprint counts.
template <int W, bool ALL_STAGED>
__global__ void __launch_bounds__(LINK_THREADS, 1)
link_kernel(const __grid_constant__ RayRig ray, ClsParams p, const int2* __restrict__ seq_bounds,
            const u64* __restrict__ leaf_rec, const long long* __restrict__ leaf_off, const int* __restrict__ leaf_cnt,
            const int* __restrict__ hdr, const unsigned char* __restrict__ fdet, const long long* __restrict__ fdet_off,
            const int* __restrict__ fdet_cnt, LinkState* state, double* __restrict__ out_paths, int8_t* __restrict__ out_assign,
            uint8_t* __restrict__ out_phase, ClsCounters* ctr) {
  using L_ = LinkLayout<W>;
  constexpr int RW = L_::RW;
  constexpr u64 POISON = 1ull << 63;  // in word W - 1
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(128) unsigned char link_dyn[];
  __shared__ LinkState S;
  __shared__ float s_lastf[TRI_MAX_DRONES][4];        // single-precision copy of each path's last point
  __shared__ unsigned s_gate[TRI_MAX_DRONES][2 * W];  // 32-bit slices of each tracked path's gate mask
  __shared__ int s_spec[2][TRI_MAX_DRONES];           // each tracked path's speculative pick (leaf index), by frame parity
  __shared__ u64 s_used[W];                           // a frame with colliding picks: what warp 0 confirmed
  __shared__ unsigned s_processed;
  __shared__ int s_win[3];                            // phase 2: the first leaf still in the list, by round mod 3
  __shared__ int s_fin_idx[LINK_MAX_FINAL];
  u64* full = reinterpret_cast<u64*>(link_dyn + 2 * L_::BUF_BYTES);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, C = p.n_cams, D = p.n_drones;
  const int fa = seq_bounds ? seq_bounds[blockIdx.x].x : p.f0, fb = seq_bounds ? seq_bounds[blockIdx.x].y : p.f1;
  LinkState* st = state + blockIdx.x;
  for (int i = tid; i < (int)(sizeof(LinkState) / sizeof(int)); i += LINK_THREADS) ((int*)&S)[i] = ((const int*)st)[i];
  if (tid < 2 * TRI_MAX_DRONES) (&s_spec[0][0])[tid] = LINK_NONE;
  if (tid < 3) s_win[tid] = LINK_NONE;
  if (tid == 0) {
    cls_mbar_init(&full[0], 1); cls_mbar_init(&full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid < D) {
    const double* last = S.tail[tid][min(max(S.n[tid], 1), PATH_TAIL) - 1];
    s_lastf[tid][0] = (float)last[0]; s_lastf[tid][1] = (float)last[1]; s_lastf[tid][2] = (float)last[2];
  }
  u64 n_phase1 = 0, n_phase2 = 0;  // lane 0 of the serial warp
  bool overflow_final = false;

  // ---- the stager: lane 0 of the last warp.  Frame table two frames ahead in registers, the staged copy one frame ahead ----
  const bool stager = tid == LINK_THREADS - 32;
  const int nf = fb - fa;
  int L_n1 = 0, nd_n1 = 0, L_n2 = 0, nd_n2 = 0;
  long long off_n1 = 0, doff_n1 = 0, off_n2 = 0, doff_n2 = 0;
  auto meta = [&](int k, int& L, long long& off, int& nd, long long& doff) {
    L = 0; off = 0; nd = 0; doff = 0;
    if (k < nf) { const int g = fa + k - p.f0; L = leaf_cnt[g]; off = leaf_off[g]; nd = fdet_cnt[g]; doff = fdet_off[g]; }
  };
  auto stage = [&](int b, int f, int L, long long off, int nd, long long doff) {
    unsigned char* base = link_dyn + (size_t)b * L_::BUF_BYTES;
    const uint32_t rec_bytes = L <= L_::MAX_LEAVES ? (uint32_t)L * RW * 8 : 0, det_bytes = (uint32_t)nd * FDET_BYTES;
    cls_mbar_expect_tx(&full[b], rec_bytes + det_bytes + L_::HDR_BYTES);
    if (rec_bytes) cls_bulk_load(base, leaf_rec + (size_t)off * RW, rec_bytes, &full[b]);
    if (det_bytes) cls_bulk_load(base + L_::REC_BYTES, fdet + (size_t)doff * FDET_BYTES, det_bytes, &full[b]);
    cls_bulk_load(base + L_::REC_BYTES + L_::DET_BYTES, hdr + (size_t)(f - p.f0) * HDR_INTS, L_::HDR_BYTES, &full[b]);
  };
  if (stager) {
    meta(0, L_n1, off_n1, nd_n1, doff_n1);
    meta(1, L_n2, off_n2, nd_n2, doff_n2);
    if (nf > 0) stage(0, fa, L_n1, off_n1, nd_n1, doff_n1);
  }

  // which warp works on which path: recomputed only when the set of tracked paths changes
  unsigned map_mask = FULL;
  int map_nseg = 0, map_seg = 0, map_np = -1;

  // One frame.  `staged` says the leaves are in shared memory (a compile-time fact, so that they are read with LDS
  // instead of generic loads); a frame with more than MAX_LEAVES leaves reads them from global memory.
  auto frame = [&](auto staged, const int k, const int L) {
    const int f = fa + k, b = k & 1;
    const unsigned char* base = link_dyn + (size_t)b * L_::BUF_BYTES;
    const int* zs = reinterpret_cast<const int*>(base + L_::REC_BYTES + L_::DET_BYTES);
    const int nd = zs[HDR_PREF + C];
    const u64* msk = decltype(staged)::value ? reinterpret_cast<const u64*>(base)
                                             : leaf_rec + (size_t)(*reinterpret_cast<const long long*>(zs + HDR_OFF)) * RW;
    const u64* pts = msk + (size_t)L * W;
    const float4* detA = reinterpret_cast<const float4*>(base + L_::REC_BYTES);
    const float4* detB = detA + nd;
    const double* detD = reinterpret_cast<const double*>(detB + nd);
    int* spec = s_spec[b];

    // The first leaf (priority order) from index `start` on whose mask lies inside the gate g, misses `used`, and whose point
    // is within MAX_STEP of (lx, ly, lz): what the reference's priority_queue pops first that passes :241-246.  This warp
    // takes the 128-leaf blocks seg, seg + nseg, ...; `best` (shared, or nullptr) holds the smallest hit of the other warps.
    auto scan = [&](int start, int seg, int nseg, const u64 (&g)[W], const u64 (&used)[W], double lx, double ly, double lz, const int* best) {
      int pick = LINK_NONE;
      for (int i0 = (start & ~31) + 128 * seg; i0 < L; i0 += 128 * nseg) {
        if (best && *reinterpret_cast<const volatile int*>(best) < i0) break;  // an earlier block already has one
        unsigned cand[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int i = i0 + 32 * u + lane;
          bool ok = i < L;
          const u64* r = msk + (size_t)(ok ? i : 0) * W;
#pragma unroll
          for (int w = 0; w < W; w += 2) {
            const ulonglong2 m = *reinterpret_cast<const ulonglong2*>(r + w);
            ok = ok && !(m.x & ~g[w]) && !(m.x & used[w]) && !(m.y & ~g[w + 1]) && !(m.y & used[w + 1]);
          }
          cand[u] = __ballot_sync(FULL, ok);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (cand[u] && pick == LINK_NONE) {  // cv::norm(c.point - pos) < MAX_STEP, :244
            bool ok = (cand[u] >> lane) & 1u;
            if (ok) {
              const u64* r = pts + (size_t)(i0 + 32 * u + lane) * 4;
              const double x = __longlong_as_double((long long)r[0]) - lx, y = __longlong_as_double((long long)r[1]) - ly,
                           z = __longlong_as_double((long long)r[2]) - lz;
              ok = sqrt_below_step(x * x + y * y + z * z);
            }
            const unsigned hit = __ballot_sync(FULL, ok);
            if (hit) pick = i0 + 32 * u + __ffs(hit) - 1;
          }
        }
        if (pick != LINK_NONE) break;
      }
      return pick;
    };
    auto emit = [&](int path, int leaf, int phase) {  // one thread: push a leaf's point to a path
      const u64* r = pts + (size_t)leaf * 4;
      const double x = __longlong_as_double((long long)r[0]), y = __longlong_as_double((long long)r[1]), z = __longlong_as_double((long long)r[2]);
      const u64 comb = r[3];
      const int n = S.n[path];
      double(*t)[3] = S.tail[path];
      if (n >= PATH_TAIL) {
        for (int q = 0; q < PATH_TAIL - 1; q++) for (int j = 0; j < 3; j++) t[q][j] = t[q + 1][j];
        t[PATH_TAIL - 1][0] = x; t[PATH_TAIL - 1][1] = y; t[PATH_TAIL - 1][2] = z;
      } else {
        t[n][0] = x; t[n][1] = y; t[n][2] = z;
      }
      s_lastf[path][0] = (float)x; s_lastf[path][1] = (float)y; s_lastf[path][2] = (float)z;
      if (n < 0x3fffffff) S.n[path] = n + 1;
      double* o = out_paths + ((size_t)path * p.n_frames + f) * 3;
      o[0] = x; o[1] = y; o[2] = z;
      if (out_assign) {
        int8_t* dst = out_assign + ((size_t)path * p.n_frames + f) * C;
        if (C == 8) {  // the 8 nibbles spread to 8 bytes, one store (rows of 8 bytes are 8-byte aligned)
          u64 v = comb & 0xffffffffull;
          v = (v | (v << 16)) & 0x0000ffff0000ffffull;
          v = (v | (v << 8)) & 0x00ff00ff00ff00ffull;
          v = (v | (v << 4)) & 0x0f0f0f0f0f0f0f0full;
          *reinterpret_cast<u64*>(dst) = v;
        } else {
          for (int c = 0; c < C; c++) dst[c] = (int8_t)((comb >> (4 * c)) & 15);
        }
      }
      if (out_phase) out_phase[(size_t)path * p.n_frames + f] = (uint8_t)phase;
    };

    // ---- which paths track (:121-123): every warp computes the same list ----
    bool act = false;
    int my_n = 0;
    if (lane < D) {
      my_n = S.n[lane];
      const double* last = S.tail[lane][min(max(my_n, 1), PATH_TAIL) - 1];
      act = my_n != 0 && !(last[0] == 0 && last[1] == 0 && last[2] == 0);
    }
    const unsigned act_mask = __ballot_sync(FULL, act);
    const int n_act = __popc(act_mask);

    // ---- speculative phase 1: path ai = warp mod n_act, block phase seg = warp div n_act of nseg (warps beyond nseg * n_act rest) ----
    if (act_mask != map_mask) {
      map_mask = act_mask; map_nseg = 0; map_seg = 0; map_np = -1;
      if (n_act > 0) {
        for (int t = n_act; t <= LINK_WARPS; t += n_act) map_nseg++;  // n_act <= TRI_MAX_DRONES = LINK_WARPS
        int ai = warp;
        while (ai >= n_act) { ai -= n_act; map_seg++; }
        if (map_seg < map_nseg) { unsigned rem = act_mask; for (int q = 0; q < ai; q++) rem &= rem - 1; map_np = __ffs(rem) - 1; }
      }
    }
    {
      const int np = map_np, seg = map_seg, nseg = map_nseg;
      if (np >= 0) {
        const int n_slices = (nd + 31) >> 5;
        const float lfx = s_lastf[np][0], lfy = s_lastf[np][1], lfz = s_lastf[np][2];
        const double* last = S.tail[np][min(S.n[np], PATH_TAIL) - 1];
        unsigned slice[2 * W], cam_set = 0;
#pragma unroll
        for (int t = 0; t < 2 * W; t++) {
          slice[t] = 0;
          if (t < n_slices) {
            const int di = 32 * t + lane;
            const bool have = di < nd;
            const float4 A = detA[have ? di : 0], B = detB[have ? di : 0];  // A = origin, dir.x; B = dir.y, dir.z, camera
            const float wx = lfx - A.x, wy = lfy - A.y, wz = lfz - A.z;
            const float cx = B.x * wz - B.y * wy, cy = B.y * wx - A.w * wz, cz = A.w * wy - B.x * wx;
            const float sf = cx * cx + cy * cy + cz * cz;
            bool gated = sf < (float)(MAX_STEP * MAX_STEP);
            // single precision decides unless sf is within its own error of the threshold: |error of a cross-product component|
            // <= ~6e-7 (|w|_1 |d|_1), and near the threshold d sf = 2 sqrt(sf) d c ~ 700 d c  (taken 3x wider)
            const float tol = 4.f + 2.1e-3f * (fabsf(wx) + fabsf(wy) + fabsf(wz));  // |d|_1 <= sqrt(3)
            if (have && fabsf(sf - (float)(MAX_STEP * MAX_STEP)) < tol) {
              const double* dd = detD + 4 * di;
              const double* org = ray.pos[__float_as_int(B.z)];
              const double ex = last[0] - org[0], ey = last[1] - org[1], ez = last[2] - org[2];  // distToRay, Triangulator.cpp:3-9
              const double fx = dd[1] * ez - dd[2] * ey, fy = dd[2] * ex - dd[0] * ez, fz = dd[0] * ey - dd[1] * ex;
              gated = sqrt_below_step(fx * fx + fy * fy + fz * fz);
            }
            slice[t] = __ballot_sync(FULL, have && gated);
            if (have && gated) cam_set |= 1u << __float_as_int(B.z);
          }
        }
        u64 g[W], none[W];
#pragma unroll
        for (int w = 0; w < W; w++) { g[w] = ((u64)slice[2 * w + 1] << 32) | slice[2 * w]; none[w] = w == W - 1 ? POISON : 0ull; }
        const int cams_in_gate = __popc(__reduce_or_sync(FULL, cam_set));  // cameras with a detection inside the gate
        if (seg == 0 && lane < 2 * W) {
          unsigned v = 0;
#pragma unroll
          for (int t = 0; t < 2 * W; t++) v = lane == t ? slice[t] : v;
          s_gate[np][lane] = v;
        }
        if (cams_in_gate >= MIN_CAMERAS) {  // else fillCombinationQueue on the gated container yields nothing
          // leaves with fewer unused cameras than the gate leaves empty cannot lie inside it
          const int pick = scan(zs[C - cams_in_gate], seg, nseg, g, none, last[0], last[1], last[2], nseg > 1 ? &spec[np] : nullptr);
          if (lane == 0 && pick != LINK_NONE) atomicMin(&spec[np], pick);
        }
      }
    }
    __syncthreads();  // barrier 2: the speculative picks are in

    // ---- confirm the picks (:119-135), lane <-> path, every warp for itself ----
    u64 used[W];
    unsigned processed;
    int cand = (lane < D && ((act_mask >> lane) & 1u)) ? spec[lane] : LINK_NONE;
    {
      u64 mk[W];
      unsigned bits = 0, any = 0;
#pragma unroll
      for (int w = 0; w < W; w++) {
        mk[w] = cand != LINK_NONE ? msk[(size_t)cand * W + w] : 0ull;
        bits += __popcll(mk[w]);
        const unsigned lo = __reduce_or_sync(FULL, (unsigned)mk[w]), hi = __reduce_or_sync(FULL, (unsigned)(mk[w] >> 32));
        used[w] = ((u64)hi << 32) | lo;
        any += __popc(lo) + __popc(hi);
      }
      used[W - 1] |= POISON;
      processed = __ballot_sync(FULL, cand != LINK_NONE);
      if (__reduce_add_sync(FULL, bits) != any) {  // two picks share a detection: walk the paths in order (warp 0), rare
        if (warp == 0) {
#pragma unroll
          for (int w = 0; w < W; w++) used[w] = w == W - 1 ? POISON : 0ull;
          processed = 0;
          for (unsigned rem = act_mask; rem; rem &= rem - 1) {
            const int np = __ffs(rem) - 1;
            int c_np = __shfl_sync(FULL, cand, np);
            if (c_np == LINK_NONE) continue;
            bool clash = false;
#pragma unroll
            for (int w = 0; w < W; w++) clash = clash || (__shfl_sync(FULL, mk[w], np) & used[w]);
            if (clash) {  // walk the list again with the used filter; nothing before the unfiltered pick can pass
              u64 g[W];
#pragma unroll
              for (int w = 0; w < W; w++) g[w] = ((u64)s_gate[np][2 * w + 1] << 32) | s_gate[np][2 * w];
              const double* last = S.tail[np][min(S.n[np], PATH_TAIL) - 1];
              c_np = scan(c_np, 0, 1, g, used, last[0], last[1], last[2], nullptr);
              if (lane == np) {
                cand = c_np;
                spec[np] = c_np;  // (the warp that pushes reads the picks back)
#pragma unroll
                for (int w = 0; w < W; w++) mk[w] = c_np != LINK_NONE ? msk[(size_t)c_np * W + w] : 0ull;
              }
              if (c_np == LINK_NONE) continue;
            }
#pragma unroll
            for (int w = 0; w < W; w++) used[w] |= __shfl_sync(FULL, mk[w], np);
            processed |= 1u << np;
          }
          if (lane == 0) {
#pragma unroll
            for (int w = 0; w < W; w++) s_used[w] = used[w];
            s_processed = processed;
          }
        }
        __syncthreads();  // (only in such frames)
#pragma unroll
        for (int w = 0; w < W; w++) used[w] = s_used[w];
        processed = s_processed;
        cand = (lane < D && ((processed >> lane) & 1u)) ? spec[lane] : LINK_NONE;
      }
    }
    // phase 1's pushes, all confirmed paths at once (lane <-> path), on the last warp: warp 0 goes straight on to phase 2 and
    // classifyPaths, which only touch the paths phase 1 did not serve
    if (warp == LINK_WARPS - 1 && ((processed >> lane) & 1u)) emit(lane, cand, 1);
    if (tid == 32 * LINK_SERIAL_WARP) n_phase1 += __popc(processed);
    if (__popc(processed) == D) return;  // :137

    // ---- phase 2: pickBestCombinations (:200-217), the reference's pop loop in parallel.  Every warp keeps the masks of
    // its 128-leaf blocks in registers (block = warp + 16 j); a round finds the first leaf of the whole list that misses
    // the used mask (REDUX.MIN in the warp, atomicMin across the warps, one block barrier), adds its mask to the used
    // mask and strikes the leaves it collides with; the loop ends with the round that finds nothing. ----
    int n_fin = 0;
    {
      constexpr int NB = LINK_BLOCKS / LINK_WARPS;
      u64 m[NB][4][W];
      unsigned ok = 0;  // bit 4 j + u: leaf 128 (warp + 16 j) + 32 u + lane is still in the list
#pragma unroll
      for (int j = 0; j < NB; j++) {
        const int i0 = 128 * (warp + LINK_WARPS * j);
        if (i0 < L) {
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int i = i0 + 32 * u + lane;
            bool o = i < L;
            const u64* r = msk + (size_t)(o ? i : 0) * W;
#pragma unroll
            for (int w = 0; w < W; w += 2) {
              const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(r + w);
              m[j][u][w] = v.x; m[j][u][w + 1] = v.y;
              o = o && !(v.x & used[w]) && !(v.y & used[w + 1]);
            }
            ok |= (unsigned)o << (4 * j + u);
          }
        }
      }
      for (int round = 0;; round++) {
        int* win = &s_win[round % 3];
        unsigned mine = (unsigned)LINK_NONE;  // this lane's first leaf still in the list (blocks and words in rising order)
#pragma unroll
        for (int j = NB - 1; j >= 0; j--)
#pragma unroll
          for (int u = 3; u >= 0; u--) mine = (ok >> (4 * j + u) & 1u) ? (unsigned)(128 * (warp + LINK_WARPS * j) + 32 * u + lane) : mine;
        const unsigned first = __reduce_min_sync(FULL, mine);
        if (lane == 0 && first != (unsigned)LINK_NONE) atomicMin(win, (int)first);
        __syncthreads();
        const int pick = *reinterpret_cast<volatile int*>(win);
        if (tid == 0) s_win[(round + 2) % 3] = LINK_NONE;  // read last in round - 1, used next in round + 2
        if (pick == LINK_NONE) break;
        u64 mj[W];
#pragma unroll
        for (int w = 0; w < W; w++) { mj[w] = msk[(size_t)pick * W + w]; used[w] |= mj[w]; }
#pragma unroll
        for (int j = 0; j < NB; j++)
#pragma unroll
          for (int u = 0; u < 4; u++) {
            bool clash = false;
#pragma unroll
            for (int w = 0; w < W; w++) clash = clash || (m[j][u][w] & mj[w]);
            if (clash) ok &= ~(1u << (4 * j + u));  // (the pick collides with itself)
          }
        if (n_fin < LINK_MAX_FINAL) { if (tid == 32 * LINK_SERIAL_WARP) s_fin_idx[n_fin] = pick; n_fin++; }
        else overflow_final = true;
      }
    }
    if (warp != LINK_SERIAL_WARP) return;
    // (leaves beyond the blocks held in registers: walked in place, 32 at a time)
    for (int i0 = 128 * LINK_BLOCKS; i0 < L; i0 += 32) {
      const int li = i0 + lane < L ? i0 + lane : -1;
      u64 m[W];
      bool o = li >= 0;
#pragma unroll
      for (int w = 0; w < W; w++) { m[w] = o ? msk[(size_t)li * W + w] : 0ull; }
#pragma unroll
      for (int w = 0; w < W; w++) o = o && !(m[w] & used[w]);
      unsigned hit = __ballot_sync(FULL, o);
      while (hit) {
        const int j = __ffs(hit) - 1;
        bool clash = false;
#pragma unroll
        for (int w = 0; w < W; w++) {
          const u64 mj = __shfl_sync(FULL, m[w], j);
          used[w] |= mj;
          clash = clash || (m[w] & mj);
        }
        if (n_fin < LINK_MAX_FINAL) { if (lane == 0) s_fin_idx[n_fin] = i0 + j; n_fin++; }
        else overflow_final = true;
        o = o && !clash;  // lane j clashes with itself
        hit = __ballot_sync(FULL, o);
      }
    }
    __syncwarp();

    // ---- classifyPaths (:262-332), lane <-> kept combination (four rounds of 32 at most) ----
    const unsigned nonempty = __ballot_sync(FULL, lane < D && S.n[lane] != 0);  // S.n after phase 1's pushes
    const unsigned d_mask = D >= 32 ? FULL : ((1u << D) - 1);
    const unsigned open_paths = nonempty & ~processed;  // not processed and not empty: the only ones :269-297 measures
    const int one_open = (n_fin == 1 && __popc(open_paths) == 1) ? __ffs(open_paths) - 1 : -1;
    double e[LINK_MAX_FINAL / 32];
    int bp[LINK_MAX_FINAL / 32];
#pragma unroll
    for (int q = 0; q < LINK_MAX_FINAL / 32; q++) {
      e[q] = -1; bp[q] = 0;
      const int i = lane + 32 * q;
      if (i < n_fin && one_open >= 0) bp[q] = one_open;  // a single kept combination and a single open path: nothing to measure or to order
      else if (i < n_fin) {  // :269-297 (the processed set does not change until the assignment loop)
        const u64* r = pts + (size_t)s_fin_idx[i] * 4;
        const double px = __longlong_as_double((long long)r[0]), py = __longlong_as_double((long long)r[1]), pz = __longlong_as_double((long long)r[2]);
        for (unsigned rem = open_paths; rem; rem &= rem - 1) {
          const int j = __ffs(rem) - 1;
          const int npc = min(S.n[j], PATH_TAIL);
          double dist = 0;
          for (int t = 0; t < npc; t++) dist += dist3(S.tail[j][t], px, py, pz);
          dist = dist / (double)npc;
          if (dist < e[q] || e[q] == -1) { e[q] = dist; bp[q] = j; }
        }
      }
    }
    // The reference sorts the (combination, nearest path, distance) triples by distance -- std::sort(greater<>) of <= 16
    // elements is libstdc++'s insertion sort: stable, ascending -- and walks them in that order (:299-321).  A triple only
    // acts while an open or an empty path is left, so instead of sorting, the warp extracts the next triple (smallest
    // distance, then smallest index) and stops as soon as no path can take a point any more.  Distances are >= 0 (or all
    // -1 when no path is open), so their bit patterns order like the values: the minimum is two 32-bit REDUX.MIN.
    {
      unsigned done = processed;
      unsigned empty_paths = d_mask & ~nonempty;
      unsigned taken = 0;  // bit q: this lane's triple lane + 32 q is consumed
      for (int step = 0; step < n_fin; step++) {
        if (!(open_paths & ~done) && !empty_paths) break;  // every remaining triple would find its path taken and no empty one
        u64 key = ~0ull;
        int idx = LINK_NONE;
#pragma unroll
        for (int q = 0; q < LINK_MAX_FINAL / 32; q++) {
          const int i = lane + 32 * q;
          const u64 kq = (u64)__double_as_longlong(e[q]);
          if (i < n_fin && !(taken >> q & 1u) && (idx == LINK_NONE || kq < key)) { key = kq; idx = i; }
        }
        const unsigned hi = (unsigned)(key >> 32), mh = __reduce_min_sync(FULL, hi);
        const unsigned lo = hi == mh ? (unsigned)key : 0xffffffffu, ml = __reduce_min_sync(FULL, lo);
        const unsigned mine = (hi == mh && lo == ml) ? (unsigned)idx : (unsigned)LINK_NONE;
        const int win = (int)__reduce_min_sync(FULL, mine);
        const int wq = win >> 5;
        if ((win & 31) == lane) taken |= 1u << wq;
        int pth_l = bp[0];
#pragma unroll
        for (int q = 1; q < LINK_MAX_FINAL / 32; q++) pth_l = wq == q ? bp[q] : pth_l;
        const int pth = __shfl_sync(FULL, pth_l, win & 31);
        int target = -1;
        if (done >> pth & 1u) { if (empty_paths) target = __ffs(empty_paths) - 1; }  // the first empty path (:305-311)
        else target = pth;
        if (target != -1) {
          if (lane == 0) { emit(target, s_fin_idx[win], 2); n_phase2++; }
          done |= 1u << target;
          empty_paths &= ~(1u << target);
          __syncwarp();
        }
      }
    }
    __syncwarp();
  };

  for (int k = 0; k < nf; k++) {
    const int b = k & 1;
    __syncthreads();  // barrier 1: frame k - 1 is linked (state, its buffer free)
    if (stager) {
      L_n1 = L_n2; off_n1 = off_n2; nd_n1 = nd_n2; doff_n1 = doff_n2;
      if (k + 1 < nf) stage(b ^ 1, fa + k + 1, L_n1, off_n1, nd_n1, doff_n1);
      meta(k + 2, L_n2, off_n2, nd_n2, doff_n2);
    }
    if (warp == 0 && lane < D) s_spec[b ^ 1][lane] = LINK_NONE;  // last read in frame k - 1, next written in frame k + 1
    cls_mbar_wait(&full[b], (uint32_t)((k >> 1) & 1));
    const int L = reinterpret_cast<const int*>(link_dyn + (size_t)b * L_::BUF_BYTES + L_::REC_BYTES + L_::DET_BYTES)[C + 1];
    if constexpr (ALL_STAGED) {
      frame(std::true_type{}, k, L);
    } else {
      if (L <= L_::MAX_LEAVES) frame(std::true_type{}, k, L);
      else frame(std::false_type{}, k, L);
    }
  }
  __syncthreads();
  for (int i = tid; i < (int)(sizeof(LinkState) / sizeof(int)); i += LINK_THREADS) ((int*)st)[i] = ((const int*)&S)[i];
  if (tid == 32 * LINK_SERIAL_WARP) {
    atomicAdd(&ctr->phase1, n_phase1); atomicAdd(&ctr->phase2, n_phase2);
    if (overflow_final) atomicExch(&ctr->overflow_final, 1);
  }
}

// What (A) hands to (B) for one batch of frames.  Two sets: (A) fills one while (B) reads the other.
struct LinkInput {
  DevBuf lrec, loff, lcnt, hdr, fdet, fdoff, fdcnt;
  cudaEvent_t begin = nullptr, end = nullptr;  // of the linking pass that reads this set
  bool linking = false;                        // a linking pass on this set has been launched and not yet collected
  ~LinkInput() { if (begin) cudaEventDestroy(begin); if (end) cudaEventDestroy(end); }
};

struct ClsWork {
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  cudaStream_t link_stream = nullptr;    // (B) runs here, next to the enumeration of the following batch on the engine's stream
  double enumerate_ms = 0, link_ms = 0;  // of the call in progress
  ~ClsWork() {
    for (cudaEvent_t v : ev) if (v) cudaEventDestroy(v);
    if (link_stream) cudaStreamDestroy(link_stream);
  }
  cudaError_t events() {
    for (cudaEvent_t& v : ev)
      if (!v) { cudaError_t err = cudaEventCreate(&v); if (err != cudaSuccess) return err; }
    for (LinkInput& in : in)
      for (cudaEvent_t* v : {&in.begin, &in.end})
        if (!*v) { cudaError_t err = cudaEventCreate(v); if (err != cudaSuccess) return err; }
    if (!link_stream) { cudaError_t err = cudaStreamCreateWithFlags(&link_stream, cudaStreamNonBlocking); if (err != cudaSuccess) return err; }
    return cudaSuccess;
  }
  // the linking pass on set k has finished (wait for it if need be): its time is added to link_ms, the set is free again
  cudaError_t collect(int k) {
    LinkInput& I = in[k];
    if (!I.linking) return cudaSuccess;
    I.linking = false;
    cudaError_t err = cudaEventSynchronize(I.end);
    if (err != cudaSuccess) return err;
    float ms = 0;
    if ((err = cudaEventElapsedTime(&ms, I.begin, I.end)) != cudaSuccess) return err;
    link_ms += ms;
    return cudaSuccess;
  }
  DevBuf offs, dets, paths, assign, phase, state, ctr, ctr_link, front, txyz, terr, sortkb, seq;
  LinkInput in[2];
  // tri_classify_begin / tri_classify_finish: the enumerated shard waiting for its linking pass
  bool pending = false;
  ClsParams job;
  int job_max_frontier = 0;
};
static void free_cls_work(void* w) { delete static_cast<ClsWork*>(w); }

}  // namespace tri

using namespace tri;

namespace tri {
cudaError_t launch_lazy_link(cudaStream_t s, const DltRig<double>& dlt, const RayRig& ray, const ClsParams& p, int n_seq, const int2* d_seq,
                             const int32_t* d_offs, const double* d_dets, LinkState* d_state, double* d_paths, int8_t* d_assign,
                             uint8_t* d_phase, ClsCounters* d_ctr);
}

namespace {

// argument checks shared by the entry points; *n_det = detections in the CSR
int cls_check(tri_engine* e, int mode, int n_drones, const int32_t* det_offsets, const double* dets_xy, int n_frames, int64_t* n_det,
              bool lazy = false) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (mode != TRI_MATRIX && mode != TRI_RAY) return fail(TRI_ERR_ARG, "mode must be TRI_MATRIX or TRI_RAY");
  const int C = e->n_cams;
  if (C > CLS_MAX_CAMS && !lazy)
    return fail(TRI_ERR_ARG, "the frame-sharded classifier enumerates the candidate combinations, which is exponential in the camera count: at most "
                             "16 cameras (tri_classify / tri_classify_sequences take up to 32 through the lazy search)");
  if (n_drones < 1 || n_drones > TRI_MAX_DRONES) return fail(TRI_ERR_ARG, "n_drones must be in [1, TRI_MAX_DRONES]");
  if (n_frames < 0) return fail(TRI_ERR_ARG, "bad frame count");
  *n_det = 0;
  if (n_frames == 0) return TRI_OK;
  if (!det_offsets) return fail(TRI_ERR_ARG, "null detection offsets");
  for (int c = 0; c < C; c++) {
    const int32_t* o = det_offsets + (size_t)c * (n_frames + 1);
    for (int f = 0; f < n_frames; f++) {
      if (o[f + 1] < o[f]) return fail(TRI_ERR_ARG, "detection offsets must be non-decreasing");
      if (o[f + 1] - o[f] > TRI_MAX_DETS) return fail(TRI_ERR_CAPACITY, "more than TRI_MAX_DETS detections on one camera in one frame");
    }
    *n_det = std::max<int64_t>(*n_det, o[n_frames]);
  }
  if (*n_det > 0 && !dets_xy) return fail(TRI_ERR_ARG, "null detections");
  return TRI_OK;
}

ClsParams cls_params(const tri_engine* e, int mode, unsigned flags, int n_drones, int n_frames) {
  ClsParams p{};
  p.n_cams = e->n_cams; p.n_drones = n_drones; p.n_frames = n_frames;
  p.solver = mode == TRI_MATRIX ? 0 : (flags & TRI_RAY_CLOSED_FORM) ? 2 : 1;  // ray: the reference's LM trajectory unless the fast solver is asked for
  p.error_ = mode == TRI_MATRIX ? MAX_ERROR_MATRIX : MAX_ERROR_RAY;  // DroneClassifier.cpp:3-10
  p.W = e->n_cams <= 8 ? 2 : 4;
  return p;
}

int cls_grid(const tri_engine* e, int frames) {
  // every resident CTA slot gets a frame: the tree expansion is latency-bound (dependent FP64 chains, idle
  // lanes on narrow levels), so occupancy is what hides it -- 4 CTAs per SM instead of 2: S09_D6 with the
  // exact LM 3.88 -> 2.82 s (profiles/r1_cls_grid_sweep.log)
  int per_sm = 2;
  if (cudaFuncSetAttribute(enumerate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ENUM_SMEM_BYTES) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, enumerate_kernel, CLS_THREADS, ENUM_SMEM_BYTES) != cudaSuccess || per_sm < 1) per_sm = 2;
  return std::max(1, std::min(frames, per_sm * e->sm_count));
}

// (A) on frames [p.f0, p.f1) with the work buffers sized by (cap, leaf_cap); *h = the counters after the launch
int cls_enumerate(tri_engine* e, ClsWork& W, int k, ClsParams& p, int cap, long long leaf_cap, int64_t n_det_batch, ClsCounters* h) {
  cudaStream_t s = e->stream;
  const int frames = p.f1 - p.f0, grid = cls_grid(e, frames);
  TRI_CUDA(W.front.alloc(sizeof(u64) * 2 * (size_t)cap * grid));
  TRI_CUDA(W.txyz.alloc(sizeof(double) * 3 * (size_t)cap * grid));
  TRI_CUDA(W.terr.alloc(sizeof(double) * (size_t)cap * grid));
  TRI_CUDA(W.sortkb.alloc(sizeof(unsigned) * (size_t)cap * grid));
  TRI_CUDA(W.events());
  TRI_CUDA(W.collect(k));  // the linking pass that read this set before
  LinkInput& I = W.in[k];
  TRI_CUDA(I.lrec.alloc(sizeof(u64) * rec_words(p.W) * (size_t)leaf_cap));
  TRI_CUDA(I.loff.alloc(sizeof(long long) * frames));
  TRI_CUDA(I.lcnt.alloc(sizeof(int) * frames));
  TRI_CUDA(I.hdr.alloc(sizeof(int) * HDR_INTS * (size_t)frames));
  TRI_CUDA(I.fdet.alloc((size_t)FDET_BYTES * (size_t)std::max<int64_t>(n_det_batch, 1)));
  TRI_CUDA(I.fdoff.alloc(sizeof(long long) * frames));
  TRI_CUDA(I.fdcnt.alloc(sizeof(int) * frames));
  p.cap = cap; p.leaf_cap = leaf_cap;
  ClsCounters* ctr = W.ctr.as<ClsCounters>();
  TRI_CUDA(cudaMemsetAsync(&ctr->leaf_total, 0, 3 * sizeof(u64), s));  // leaf_total, fdet_total, next_frame: within this batch
  TRI_CUDA(cudaEventRecord(W.ev[0], s));
  enumerate_kernel<<<grid, CLS_THREADS, ENUM_SMEM_BYTES, s>>>(e->rig64, e->ray, p, W.offs.as<int32_t>(), W.dets.as<double>(), W.front.as<u64>(),
                                                 W.txyz.as<double>(), W.terr.as<double>(), I.lrec.as<u64>(), I.loff.as<long long>(),
                                                 I.lcnt.as<int>(), I.hdr.as<int>(), I.fdet.as<unsigned char>(), I.fdoff.as<long long>(),
                                                 I.fdcnt.as<int>(), W.sortkb.as<unsigned>(), ctr);
  e->launches++;
  TRI_CUDA(cudaGetLastError());
  TRI_CUDA(cudaEventRecord(W.ev[1], s));
  TRI_CUDA(cudaMemcpyAsync(h, ctr, sizeof(*h), cudaMemcpyDeviceToHost, s));
  TRI_CUDA(cudaStreamSynchronize(s));
  float ms = 0;
  TRI_CUDA(cudaEventElapsedTime(&ms, W.ev[0], W.ev[1]));
  W.enumerate_ms += ms;
  return TRI_OK;
}

// (B) on the batch enumerated into set k: one CTA per sequence (seq == nullptr: the single sequence [p.f0, p.f1)), launched on the
// link stream -- the caller goes on to enumerate the next batch into the other set; W.collect(k) waits for this pass.
int cls_link(tri_engine* e, ClsWork& W, int k, const ClsParams& p, int n_seq, const int2* d_seq, int first_seq, bool want_assign, bool want_phase, int max_leaves) {
  cudaStream_t s = W.link_stream;
  LinkInput& I = W.in[k];
  auto go = [&](auto kern, int bytes) -> int {
    TRI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    TRI_CUDA(cudaEventRecord(I.begin, s));
    kern<<<n_seq, LINK_THREADS, bytes, s>>>(e->ray, p, d_seq, I.lrec.as<u64>(), I.loff.as<long long>(), I.lcnt.as<int>(), I.hdr.as<int>(),
                                  I.fdet.as<unsigned char>(), I.fdoff.as<long long>(), I.fdcnt.as<int>(), W.state.as<LinkState>() + first_seq,
                                  W.paths.as<double>(), want_assign ? W.assign.as<int8_t>() : nullptr,
                                  want_phase ? W.phase.as<uint8_t>() : nullptr, W.ctr_link.as<ClsCounters>());
    e->launches++;
    TRI_CUDA(cudaGetLastError());
    TRI_CUDA(cudaEventRecord(I.end, s));
    I.linking = true;
    return TRI_OK;
  };
  if (p.W == 2) return max_leaves <= LinkLayout<2>::MAX_LEAVES ? go(link_kernel<2, true>, LinkLayout<2>::BYTES) : go(link_kernel<2, false>, LinkLayout<2>::BYTES);
  return max_leaves <= LinkLayout<4>::MAX_LEAVES ? go(link_kernel<4, true>, LinkLayout<4>::BYTES) : go(link_kernel<4, false>, LinkLayout<4>::BYTES);
}

int64_t dets_in_frames(const int32_t* det_offsets, int C, int n_frames, int f0, int f1) {
  int64_t n = 0;
  for (int c = 0; c < C; c++) { const int32_t* o = det_offsets + (size_t)c * (n_frames + 1); n += o[f1] - o[f0]; }
  return n;
}

void cls_stats(tri_classify_stats* stats, const ClsCounters& h, int max_frontier, const ClsWork& W) {
  if (!stats) return;
  stats->enumerate_us = (int64_t)(W.enumerate_ms * 1e3); stats->link_us = (int64_t)(W.link_ms * 1e3);
  stats->nodes = (int64_t)h.nodes; stats->solves = (int64_t)h.solves; stats->leaves = (int64_t)h.leaves;
  stats->lm_iters = (int64_t)h.lm_iters; stats->phase1 = (int64_t)h.phase1; stats->phase2 = (int64_t)h.phase2;
  stats->ties = (int64_t)h.ties; stats->max_frontier = max_frontier;
}

// The engine's classifier work space, created on first use.
ClsWork& cls_work(tri_engine* e) {
  if (!e->cls_work) { e->cls_work = new ClsWork(); e->cls_work_free = free_cls_work; }
  return *static_cast<ClsWork*>(e->cls_work);
}

// The detection CSR of n_frames frames onto the device, and room for the enumeration's counters.
int cls_upload(tri_engine* e, ClsWork& W, const int32_t* det_offsets, const double* dets_xy, int n_frames, int64_t n_det) {
  cudaStream_t s = e->stream;
  const size_t n_offs = (size_t)e->n_cams * (n_frames + 1);
  TRI_CUDA(W.offs.alloc(sizeof(int32_t) * n_offs));
  TRI_CUDA(W.dets.alloc(sizeof(double) * 2 * n_det));
  TRI_CUDA(W.ctr.alloc(sizeof(ClsCounters)));
  TRI_CUDA(cudaMemcpyAsync(W.offs.p, det_offsets, sizeof(int32_t) * n_offs, cudaMemcpyHostToDevice, s));
  if (n_det) TRI_CUDA(cudaMemcpyAsync(W.dets.p, dets_xy, sizeof(double) * 2 * n_det, cudaMemcpyHostToDevice, s));
  return TRI_OK;
}

// Output bytes: paths [drone][frame][xyz] doubles, assign [drone][frame][camera] and phase [drone][frame] bytes.
struct ClsOutBytes {
  size_t paths, assign, phase;
};
ClsOutBytes cls_out_bytes(const ClsParams& p) {
  return {sizeof(double) * 3 * p.n_drones * (size_t)p.n_frames, (size_t)p.n_drones * p.n_frames * p.n_cams, (size_t)p.n_drones * p.n_frames};
}

// The linking pass's outputs, cleared (assign to -1), and its n_state link states, copied from state_in or zeroed.
int cls_outputs(tri_engine* e, ClsWork& W, const ClsParams& p, int n_state, const void* state_in) {
  cudaStream_t s = e->stream;
  const ClsOutBytes b = cls_out_bytes(p);
  TRI_CUDA(W.paths.alloc(b.paths));
  TRI_CUDA(W.assign.alloc(b.assign));
  TRI_CUDA(W.phase.alloc(b.phase));
  TRI_CUDA(W.state.alloc(sizeof(LinkState) * (size_t)n_state));
  TRI_CUDA(W.ctr_link.alloc(sizeof(ClsCounters)));
  TRI_CUDA(cudaMemsetAsync(W.ctr_link.p, 0, sizeof(ClsCounters), s));
  TRI_CUDA(cudaMemsetAsync(W.paths.p, 0, b.paths, s));
  TRI_CUDA(cudaMemsetAsync(W.assign.p, 0xff, b.assign, s));
  TRI_CUDA(cudaMemsetAsync(W.phase.p, 0, b.phase, s));
  if (state_in) TRI_CUDA(cudaMemcpyAsync(W.state.p, state_in, sizeof(LinkState) * (size_t)n_state, cudaMemcpyHostToDevice, s));
  else TRI_CUDA(cudaMemsetAsync(W.state.p, 0, sizeof(LinkState) * (size_t)n_state, s));
  return TRI_OK;
}

// D2H of the outputs asked for (paths always), queued on the engine's stream.
int cls_copy_out(tri_engine* e, ClsWork& W, const ClsParams& p, double* out_paths, int8_t* out_assign, uint8_t* out_phase) {
  cudaStream_t s = e->stream;
  const ClsOutBytes b = cls_out_bytes(p);
  TRI_CUDA(cudaMemcpyAsync(out_paths, W.paths.p, b.paths, cudaMemcpyDeviceToHost, s));
  if (out_assign) TRI_CUDA(cudaMemcpyAsync(out_assign, W.assign.p, b.assign, cudaMemcpyDeviceToHost, s));
  if (out_phase) TRI_CUDA(cudaMemcpyAsync(out_phase, W.phase.p, b.phase, cudaMemcpyDeviceToHost, s));
  return TRI_OK;
}

// After the linking passes: the outputs (and the last link state, if state_out is given) to the host, the
// combination-capacity check, the statistics.
int cls_collect(tri_engine* e, ClsWork& W, const ClsParams& p, double* out_paths, int8_t* out_assign, uint8_t* out_phase,
                void* state_out, int max_frontier, tri_classify_stats* stats) {
  cudaStream_t s = e->stream;
  const int st = cls_copy_out(e, W, p, out_paths, out_assign, out_phase);
  if (st != TRI_OK) return st;
  if (state_out) TRI_CUDA(cudaMemcpyAsync(state_out, W.state.p, sizeof(LinkState), cudaMemcpyDeviceToHost, s));
  ClsCounters h{}, hl{};
  TRI_CUDA(cudaMemcpyAsync(&h, W.ctr.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  TRI_CUDA(cudaMemcpyAsync(&hl, W.ctr_link.p, sizeof(hl), cudaMemcpyDeviceToHost, s));
  TRI_CUDA(cudaStreamSynchronize(s));
  if (hl.overflow_final) return fail(TRI_ERR_CAPACITY, "more than 128 disjoint combinations kept in one frame");
  h.phase1 = hl.phase1; h.phase2 = hl.phase2;
  cls_stats(stats, h, max_frontier, W);
  return TRI_OK;
}

// Classify n_seq independent sequences laid back to back in one CSR of n_frames frames (seq_bounds[s] .. seq_bounds[s+1]).
int cls_run(tri_engine* e, int mode, unsigned flags, int n_drones, const int32_t* det_offsets, const double* dets_xy, int n_frames,
            int n_seq, const int32_t* seq_bounds, double* out_paths, int8_t* out_assign, uint8_t* out_phase, tri_classify_stats* stats) {
  int64_t n_det = 0;
  const bool lazy = e && (e->n_cams > CLS_MAX_CAMS || (flags & TRI_CLS_LAZY));
  int st = cls_check(e, mode, n_drones, det_offsets, dets_xy, n_frames, &n_det, lazy);
  if (st != TRI_OK) return st;
  if (!out_paths && n_frames > 0) return fail(TRI_ERR_ARG, "bad output arguments");
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n_frames == 0) return TRI_OK;
  const int C = e->n_cams;
  DeviceGuard g(e->device);
  cudaStream_t s = e->stream;
  ClsParams p = cls_params(e, mode, flags, n_drones, n_frames);
  ClsWork& W = cls_work(e);
  W.pending = false;
  TRI_CUDA(W.collect(0));  // (a linking pass left behind by a call that failed half-way)
  TRI_CUDA(W.collect(1));
  W.enumerate_ms = W.link_ms = 0;
  const bool multi = n_seq > 1;
  if ((st = cls_upload(e, W, det_offsets, dets_xy, n_frames, n_det)) != TRI_OK) return st;
  if ((st = cls_outputs(e, W, p, std::max(n_seq, 1), nullptr)) != TRI_OK) return st;
  TRI_CUDA(cudaMemsetAsync(W.ctr.p, 0, sizeof(ClsCounters), s));
  std::vector<int2> seq;
  if (multi) {  // every sequence links on its own warp: all frames are enumerated first, in one batch
    for (int q = 0; q < n_seq; q++) {
      if (seq_bounds[q] < 0 || seq_bounds[q + 1] < seq_bounds[q] || seq_bounds[q + 1] > n_frames) return fail(TRI_ERR_ARG, "sequence bounds must be non-decreasing within [0, n_frames]");
      seq.push_back(make_int2(seq_bounds[q], seq_bounds[q + 1]));
    }
    TRI_CUDA(W.seq.alloc(sizeof(int2) * n_seq));
    TRI_CUDA(cudaMemcpyAsync(W.seq.p, seq.data(), sizeof(int2) * n_seq, cudaMemcpyHostToDevice, s));
  }

  if (lazy) {  // more than 16 cameras, or on request: no enumeration, the lazy best-first search of tri_classify_lazy.cu
    p.f0 = 0; p.f1 = n_frames;
    TRI_CUDA(W.events());
    TRI_CUDA(cudaEventRecord(W.ev[1], s));
    TRI_CUDA(launch_lazy_link(s, e->rig64, e->ray, p, multi ? n_seq : 1, multi ? W.seq.as<int2>() : nullptr, W.offs.as<int32_t>(), W.dets.as<double>(),
                              W.state.as<LinkState>(), W.paths.as<double>(), out_assign ? W.assign.as<int8_t>() : nullptr,
                              out_phase ? W.phase.as<uint8_t>() : nullptr, W.ctr.as<ClsCounters>()));
    e->launches++;
    TRI_CUDA(cudaEventRecord(W.ev[2], s));
    if ((st = cls_copy_out(e, W, p, out_paths, out_assign, out_phase)) != TRI_OK) return st;
    ClsCounters hz{};
    TRI_CUDA(cudaMemcpyAsync(&hz, W.ctr.p, sizeof(hz), cudaMemcpyDeviceToHost, s));
    TRI_CUDA(cudaStreamSynchronize(s));
    float ms = 0;
    TRI_CUDA(cudaEventElapsedTime(&ms, W.ev[1], W.ev[2]));
    W.link_ms = ms;
    if (hz.bad_input) return fail(TRI_ERR_ARG, "malformed detection offsets");
    if (hz.overflow_frontier) return fail(TRI_ERR_CAPACITY, "the lazy search visited more than 2^20 nodes for one combination");
    if (hz.overflow_final) return fail(TRI_ERR_CAPACITY, "more than 128 disjoint combinations kept in one frame");
    cls_stats(stats, hz, 0, W);
    return TRI_OK;
  }

  // Work is cut into batches of frames: (A) enumerates a batch, (B) links it -- on its own stream, while (A) already works on the
  // next batch into the other set of buffers (everything this stream has queued so far is complete by then: cls_enumerate ends
  // with a synchronisation).  One sequence: 8192 frames per batch, the state carried from batch to batch.  Many sequences:
  // whole sequences per batch (about 128 k frames), one CTA each.
  int batch = std::min(n_frames, 8192);
  int cap = 1 << 14;
  long long leaf_cap = 4ll << 20;
  ClsCounters h{};
  int max_frontier = 0;
  int q0 = 0;  // first sequence of the batch (multi)
  int set = 0;  // the buffers this batch is enumerated into
  for (int f0 = 0; f0 < n_frames;) {
    int f1 = std::min(n_frames, f0 + batch), q1 = q0;
    if (multi) {
      q1 = q0 + 1;
      while (q1 < n_seq && seq_bounds[q1 + 1] - seq_bounds[q0] <= (128 << 10)) q1++;
      f1 = seq_bounds[q1];
      if (f1 == f0) { q0 = q1; continue; }  // empty sequences
      leaf_cap = std::max<long long>(leaf_cap, 1024ll * (f1 - f0));
    }
    p.f0 = f0; p.f1 = f1;
    ClsCounters before;
    TRI_CUDA(cudaMemcpyAsync(&before, W.ctr.p, sizeof(before), cudaMemcpyDeviceToHost, s));
    TRI_CUDA(cudaStreamSynchronize(s));
    if ((st = cls_enumerate(e, W, set, p, cap, leaf_cap, dets_in_frames(det_offsets, C, n_frames, f0, f1), &h)) != TRI_OK) return st;
    if (h.bad_input) return fail(TRI_ERR_ARG, "malformed detection offsets");
    if (h.overflow_frontier || h.overflow_leaves) {
      // grow the work buffers (or shrink the batch) and redo this batch; the statistics of the aborted attempt are rolled back
      if (h.overflow_frontier) { if (cap >= (1 << 22)) return fail(TRI_ERR_CAPACITY, "combination frontier exceeds 4M nodes in one frame"); cap *= 4; if (!multi) batch = std::max(1, batch / 4); }
      if (h.overflow_leaves) { if (!multi && batch > 64) batch /= 4; else if (leaf_cap < (1ll << 30)) leaf_cap *= 4; else return fail(TRI_ERR_CAPACITY, "candidate list exceeds device buffer"); }
      before.overflow_frontier = before.overflow_leaves = 0;
      TRI_CUDA(cudaMemcpyAsync(W.ctr.p, &before, sizeof(before), cudaMemcpyHostToDevice, s));
      TRI_CUDA(cudaStreamSynchronize(s));
      continue;
    }
    max_frontier = std::max(max_frontier, h.max_frontier);
    if ((st = cls_link(e, W, set, p, multi ? q1 - q0 : 1, multi ? W.seq.as<int2>() + q0 : nullptr, multi ? q0 : 0, out_assign != nullptr, out_phase != nullptr, h.max_frontier)) != TRI_OK) return st;
    set ^= 1;
    f0 = f1;
    q0 = q1;
  }
  TRI_CUDA(W.collect(0));
  TRI_CUDA(W.collect(1));
  return cls_collect(e, W, p, out_paths, out_assign, out_phase, nullptr, max_frontier, stats);
}

}  // namespace

extern "C" int tri_classify(tri_engine* e, int mode, unsigned flags, int n_drones, const int32_t* det_offsets,
                            const double* dets_xy, int n_frames, double* out_paths, int8_t* out_assign, uint8_t* out_phase,
                            tri_classify_stats* stats) {
  return cls_run(e, mode, flags, n_drones, det_offsets, dets_xy, n_frames, 1, nullptr, out_paths, out_assign, out_phase, stats);
}

// Many independent sequences (recordings) in one call: sequence q holds the frames [seq_bounds[q], seq_bounds[q+1]) of the
// CSR; every frame of every sequence is enumerated in one launch and each sequence is linked by its own warp.
extern "C" int tri_classify_sequences(tri_engine* e, int mode, unsigned flags, int n_drones, int n_seq, const int32_t* seq_bounds,
                                      const int32_t* det_offsets, const double* dets_xy, int n_frames, double* out_paths,
                                      int8_t* out_assign, uint8_t* out_phase, tri_classify_stats* stats) {
  if (n_seq < 1 || !seq_bounds) return fail(TRI_ERR_ARG, "no sequences");
  if (seq_bounds[0] != 0 || seq_bounds[n_seq] != n_frames) return fail(TRI_ERR_ARG, "sequence bounds must cover [0, n_frames]");
  if (n_seq == 1) return cls_run(e, mode, flags, n_drones, det_offsets, dets_xy, n_frames, 1, nullptr, out_paths, out_assign, out_phase, stats);
  return cls_run(e, mode, flags, n_drones, det_offsets, dets_xy, n_frames, n_seq, seq_bounds, out_paths, out_assign, out_phase, stats);
}

// ---- frame-sharded classification (SURVEY 8e): candidate generation is independent per frame, linking is a
// chain.  tri_classify_begin enumerates a contiguous shard of the sequence and keeps every frame's candidate
// list on the device; tri_classify_finish links the shard starting from the tracking state the previous shard
// ended with (n_drones x (last point + 3-point tail) + counters, an opaque tri_classify_state_bytes() blob) and
// returns the state for the next one.  All ranks enumerate at once; only the small state travels along the chain.
extern "C" int tri_classify_state_bytes(void) { return (int)sizeof(LinkState); }

extern "C" int tri_classify_begin(tri_engine* e, int mode, unsigned flags, int n_drones, const int32_t* det_offsets,
                                  const double* dets_xy, int n_frames) {
  int64_t n_det = 0;
  int st = cls_check(e, mode, n_drones, det_offsets, dets_xy, n_frames, &n_det);
  if (st != TRI_OK) return st;
  DeviceGuard g(e->device);
  cudaStream_t s = e->stream;
  ClsWork& W = cls_work(e);
  W.pending = false;
  W.enumerate_ms = W.link_ms = 0;
  ClsParams p = cls_params(e, mode, flags, n_drones, n_frames);
  p.f0 = 0; p.f1 = n_frames;
  W.job = p;
  W.job_max_frontier = 0;
  if (n_frames == 0) { W.pending = true; return TRI_OK; }
  if ((st = cls_upload(e, W, det_offsets, dets_xy, n_frames, n_det)) != TRI_OK) return st;
  int cap = 1 << 14;
  long long leaf_cap = std::max<long long>(4ll << 20, 1024ll * n_frames);
  for (;;) {  // the whole shard's candidates stay resident: on overflow grow the buffers and enumerate again
    TRI_CUDA(cudaMemsetAsync(W.ctr.p, 0, sizeof(ClsCounters), s));
    ClsCounters h{};
    if ((st = cls_enumerate(e, W, 0, p, cap, leaf_cap, n_det, &h)) != TRI_OK) return st;
    if (h.bad_input) return fail(TRI_ERR_ARG, "malformed detection offsets");
    if (h.overflow_frontier) { if (cap >= (1 << 22)) return fail(TRI_ERR_CAPACITY, "combination frontier exceeds 4M nodes in one frame"); cap *= 4; continue; }
    if (h.overflow_leaves) { if (leaf_cap >= (1ll << 30)) return fail(TRI_ERR_CAPACITY, "candidate list exceeds device buffer"); leaf_cap *= 4; continue; }
    W.job_max_frontier = h.max_frontier;
    break;
  }
  W.job = p;
  W.pending = true;
  return TRI_OK;
}

extern "C" int tri_classify_finish(tri_engine* e, const void* state_in, void* state_out, double* out_paths, int8_t* out_assign,
                                   uint8_t* out_phase, tri_classify_stats* stats) {
  if (!e || !e->cls_work) return fail(TRI_ERR_ARG, "tri_classify_finish without tri_classify_begin");
  ClsWork& W = *static_cast<ClsWork*>(e->cls_work);
  if (!W.pending) return fail(TRI_ERR_ARG, "tri_classify_finish without tri_classify_begin");
  W.pending = false;
  const ClsParams p = W.job;
  if (stats) memset(stats, 0, sizeof(*stats));
  if (p.n_frames == 0) {
    if (state_out) { if (state_in) memcpy(state_out, state_in, sizeof(LinkState)); else memset(state_out, 0, sizeof(LinkState)); }
    return TRI_OK;
  }
  if (!out_paths) return fail(TRI_ERR_ARG, "bad output arguments");
  DeviceGuard g(e->device);
  int st = cls_outputs(e, W, p, 1, state_in);
  if (st != TRI_OK) return st;
  TRI_CUDA(cudaStreamSynchronize(e->stream));  // the linking pass runs on its own stream
  if ((st = cls_link(e, W, 0, p, 1, nullptr, 0, out_assign != nullptr, out_phase != nullptr, W.job_max_frontier)) != TRI_OK) return st;
  TRI_CUDA(W.collect(0));
  return cls_collect(e, W, p, out_paths, out_assign, out_phase, state_out, W.job_max_frontier, stats);
}

// One C++ process driving several GPUs: every engine enumerates its contiguous frame range on its own host thread,
// then the shards are linked in order on the caller's thread with the state handed along.  Same outputs as
// tri_classify on the whole sequence.
extern "C" int tri_classify_multi(tri_engine* const* engines, int n_engines, int mode, unsigned flags, int n_drones,
                                  const int32_t* det_offsets, const double* dets_xy, int n_frames, double* out_paths,
                                  int8_t* out_assign, uint8_t* out_phase, tri_classify_stats* stats) {
  if (!engines || n_engines < 1) return fail(TRI_ERR_ARG, "no engines");
  for (int g = 0; g < n_engines; g++)
    if (!engines[g] || engines[g]->n_cams != engines[0]->n_cams) return fail(TRI_ERR_ARG, "engines must hold the same rig");
  if (n_engines == 1) return tri_classify(engines[0], mode, flags, n_drones, det_offsets, dets_xy, n_frames, out_paths, out_assign, out_phase, stats);
  if (n_frames < 0 || !out_paths || (n_frames > 0 && !det_offsets)) return fail(TRI_ERR_ARG, "bad arguments");
  if (n_drones < 1 || n_drones > TRI_MAX_DRONES) return fail(TRI_ERR_ARG, "n_drones must be in [1, TRI_MAX_DRONES]");
  if (n_frames == 0) { if (stats) memset(stats, 0, sizeof(*stats)); return TRI_OK; }
  const int C = engines[0]->n_cams;
  auto cut = [&](int g) { return (int)((int64_t)n_frames * g / n_engines); };
  // per-shard CSR: offsets rebased to the shard, detections gathered camera by camera
  std::vector<std::vector<int32_t>> offs(n_engines);
  std::vector<std::vector<double>> dets(n_engines);
  for (int g = 0; g < n_engines; g++) {
    const int f0 = cut(g), f1 = cut(g + 1);
    offs[g].assign((size_t)C * (f1 - f0 + 1), 0);
    int32_t base = 0;
    for (int c = 0; c < C; c++) {
      const int32_t* o = det_offsets + (size_t)c * (n_frames + 1);
      const int32_t a = o[f0], b = o[f1];
      if (b < a) return fail(TRI_ERR_ARG, "detection offsets must be non-decreasing");
      for (int f = f0; f <= f1; f++) offs[g][(size_t)c * (f1 - f0 + 1) + (f - f0)] = o[f] - a + base;
      if (b > a) {
        if (!dets_xy) return fail(TRI_ERR_ARG, "null detections");
        dets[g].insert(dets[g].end(), dets_xy + 2 * (size_t)a, dets_xy + 2 * (size_t)b);
      }
      base += b - a;
    }
  }
  const int rc = fan_out(n_engines, [&](int g) {
    return tri_classify_begin(engines[g], mode, flags, n_drones, offs[g].data(), dets[g].empty() ? nullptr : dets[g].data(), cut(g + 1) - cut(g));
  });
  if (rc != TRI_OK) return rc;
  if (stats) memset(stats, 0, sizeof(*stats));
  std::vector<unsigned char> state(sizeof(LinkState), 0);
  for (int g = 0; g < n_engines; g++) {
    const int f0 = cut(g), nf = cut(g + 1) - f0;
    std::vector<double> paths((size_t)3 * n_drones * nf);
    std::vector<int8_t> assign(out_assign ? (size_t)n_drones * nf * C : 0);
    std::vector<uint8_t> phase(out_phase ? (size_t)n_drones * nf : 0);
    tri_classify_stats st{};
    const int rc = tri_classify_finish(engines[g], g == 0 ? nullptr : state.data(), state.data(), nf ? paths.data() : out_paths,
                                       out_assign ? assign.data() : nullptr, out_phase ? phase.data() : nullptr, &st);
    if (rc != TRI_OK) return rc;
    for (int d = 0; d < n_drones; d++) {  // [drone][frame] rows of the shard into the whole sequence's rows
      if (nf) memcpy(out_paths + ((size_t)d * n_frames + f0) * 3, paths.data() + (size_t)d * nf * 3, sizeof(double) * 3 * nf);
      if (out_assign && nf) memcpy(out_assign + ((size_t)d * n_frames + f0) * C, assign.data() + (size_t)d * nf * C, (size_t)nf * C);
      if (out_phase && nf) memcpy(out_phase + (size_t)d * n_frames + f0, phase.data() + (size_t)d * nf, nf);
    }
    if (stats) {
      stats->nodes += st.nodes; stats->solves += st.solves; stats->leaves += st.leaves; stats->lm_iters += st.lm_iters;
      stats->phase1 += st.phase1; stats->phase2 += st.phase2; stats->ties += st.ties;
      stats->enumerate_us = std::max(stats->enumerate_us, st.enumerate_us); stats->link_us += st.link_us;
      stats->max_frontier = std::max(stats->max_frontier, st.max_frontier);
    }
  }
  return TRI_OK;
}
