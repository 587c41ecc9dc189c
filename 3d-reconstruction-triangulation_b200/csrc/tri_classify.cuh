// tri_classify.cuh -- declarations shared by the classifier's translation units (tri_classify.cu: enumeration + linking for
// up to 16 cameras; tri_classify_lazy.cu: the lazy best-first search for up to 32).  Include only from -fmad=false units.
#pragma once
#include <float.h>

#include "tri_engine.cuh"
#include "tri_ref.cuh"

namespace tri {

constexpr int CLS_MAX_CAMS = 16;   // 4 bits per camera in a 64-bit combination
constexpr int CLS_THREADS = 128;
#ifndef TRI_ENUM_SORT_CAP
#define TRI_ENUM_SORT_CAP 4096
#endif
#ifndef TRI_ENUM_MIN_CTAS
#define TRI_ENUM_MIN_CTAS 4
#endif
constexpr int ENUM_SORT_CAP = TRI_ENUM_SORT_CAP;   // leaves of one frame sorted in shared memory (12 bytes each); longer lists are sorted in global memory
constexpr int ENUM_IDX_BITS = 22;                  // a frame's leaves are numbered below the frontier capacity, at most 2^22
constexpr int ENUM_SMEM_BYTES = ENUM_SORT_CAP * 12;
constexpr int LINK_MAX_FINAL = 128;  // combinations pickBestCombinations can keep in one frame: <= 15 * C / 2 = 120 disjoint ones
typedef unsigned long long u64;

// DroneClassifier.h:11-17
constexpr double MAX_ERROR_MATRIX = 1e+5, MAX_ERROR_RAY = 120, MAX_STEP = 200;
constexpr int MIN_CAMERAS = 2, PATH_TAIL = 3;

// ---- what (A) hands to (B), per frame, all of it independent of the tracking state ------------------------
// The frame's detections are numbered camera-major (pref[c] + d); a detection MASK has one bit per such number.
// A candidate ("leaf") record, stored in PRIORITY order (Combination::operator<, :12-20):
//   mask[W]   the leaf's detections.  Two combinations collide (isCombinationUnique, :32-41) <=> their masks
//             intersect; a combination is inside a path's ray gate <=> its mask is a subset of the gate mask.  The top
//             bit of the last word is a poison bit: set on a leaf whose error is not < error_ (it can never be
//             accepted, :209, :243) and in every "used" mask.
//   xyz[3]    the triangulated point, comb = the 4-bit-per-camera combination word (for the assignment output)
// A frame's leaves are one block: the masks of all leaves ([L][W], dense: a warp tests 32 leaves with conflict-free 16-byte
// shared-memory loads), then [L][4] = point, combination.  W = 2 (<= 8 cameras) or 4 (<= 16 cameras).
__host__ __device__ constexpr int rec_words(int W) { return W + 4; }
// per frame: [0 .. C+1] zstart[z] = leaves with fewer than z unused cameras (so [C+1] = all leaves); [20 .. 20+C] pref[c]
// (so [20+C] = detections); [38..39] the frame's offset into the leaf array (a long long)
constexpr int HDR_INTS = 40;
constexpr int HDR_PREF = 20;
constexpr int HDR_OFF = 38;
// A frame's n detections with their pixel rays (Triangulator.cpp:27-55) are one block of n * FDET_BYTES bytes:
// n x float4 {origin, dir.x}, n x float4 {dir.y, dir.z, camera (int bits), 0} -- single precision for the gate's fast path --,
// n x 4 doubles {dir, 0}
constexpr int FDET_BYTES = 64;
constexpr int LINK_MAX_DETS = CLS_MAX_CAMS * TRI_MAX_DETS;  // 240

struct ClsParams {
  int n_cams, n_drones, solver;  // solver: 0 matrix, 1 ray reference LM, 2 ray closed form
  int n_frames;                  // whole sequence (row length of the CSR offsets is n_frames + 1)
  int f0, f1;                    // frame batch [f0, f1)
  int cap;                       // frontier capacity per CTA
  int W;                         // mask words per leaf
  long long leaf_cap;            // leaf records
  double error_;
};

struct ClsCounters {
  u64 leaf_total, fdet_total, next_frame, nodes, solves, leaves, lm_iters, phase1, phase2, ties;
  int max_frontier, overflow_frontier, overflow_leaves, overflow_final, bad_input;
};

struct LinkState {
  double tail[TRI_MAX_DRONES][PATH_TAIL][3];  // oldest .. newest of the last min(n,3) points
  int n[TRI_MAX_DRONES];                      // points pushed so far (saturating)
};

__device__ __forceinline__ u64 nonzero_nibbles(u64 v) { return (v | (v >> 1) | (v >> 2) | (v >> 3)) & 0x1111111111111111ull; }

// isCombinationUnique (DroneClassifier.cpp:32-41): no camera where both use the same detection
__device__ __forceinline__ bool conflicts(u64 a, u64 b) { return (nonzero_nibbles(a) & ~nonzero_nibbles(a ^ b)) != 0; }

// RayTriangulator::triangulatePoint on rays already built (solver 1: cv::LMSolver's trajectory; 2: the minimiser in closed form)
__device__ inline double solve_rays(const RayRig& ray, int solver, const ref::RaySet& rs, double X[3], int& iters) {
  iters = 0;
  if (solver == 1) return ref::lm_point(ray, rs, X, iters);
  // closed form about the mean origin (the minimiser the reference's LM converges to)
  const int n = rs.n;
  double m[3] = {0, 0, 0};
  for (int k = 0; k < n; k++) for (int j = 0; j < 3; j++) m[j] += ray.pos[rs.cam[k]][j] / n;
  double M[6] = {0, 0, 0, 0, 0, 0}, c[3] = {0, 0, 0};
  for (int k = 0; k < n; k++) {
    const double* d = rs.d[k];
    const double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
    const double o[3] = {ray.pos[rs.cam[k]][0] - m[0], ray.pos[rs.cam[k]][1] - m[1], ray.pos[rs.cam[k]][2] - m[2]};
    const double dot = d[0] * o[0] + d[1] * o[1] + d[2] * o[2];
    M[0] += dd - d[0] * d[0]; M[1] -= d[0] * d[1]; M[2] -= d[0] * d[2];
    M[3] += dd - d[1] * d[1]; M[4] -= d[1] * d[2]; M[5] += dd - d[2] * d[2];
    for (int j = 0; j < 3; j++) c[j] += dd * o[j] - d[j] * dot;
  }
  solve_sym3<double>(M, c, X);
  for (int j = 0; j < 3; j++) X[j] += m[j];
  double S, rmax, e;
  ref::residual_pass(ray, rs, X, S, rmax, e);
  iters = 1;
  return e;
}

template <typename Rows>
__device__ inline double solve_combination(const Rows& dlt_P, const RayRig& ray, int solver, u64 comb, int n_cams,
                                           const double (*px)[TRI_MAX_DETS], const double (*py)[TRI_MAX_DETS], double X[3],
                                           int& iters) {
  iters = 0;
  if (solver == 0) {
    // ref::dlt_point_rows on the combination's detections, camera by camera: the same operations in the same order, without
    // the compacted (camera, x, y) arrays -- indexed at run time they would live in local memory
    double M[6] = {0, 0, 0, 0, 0, 0}, v[3] = {0, 0, 0};
    int n = 0;
    for (int i = 0; i < n_cams; i++) {
      const int k = (int)((comb >> (4 * i)) & 15);
      if (!k) continue;
      n++;
      const double* P = dlt_P[i];
      const double x = px[i][k - 1], y = py[i][k - 1];
      double a0 = P[0] - x * P[8], a1 = P[1] - x * P[9], a2 = P[2] - x * P[10], b = x * P[11] - P[3];
      M[0] += a0 * a0; M[1] += a0 * a1; M[2] += a0 * a2; M[3] += a1 * a1; M[4] += a1 * a2; M[5] += a2 * a2;
      v[0] += a0 * b; v[1] += a1 * b; v[2] += a2 * b;
      a0 = P[4] - y * P[8]; a1 = P[5] - y * P[9]; a2 = P[6] - y * P[10]; b = y * P[11] - P[7];
      M[0] += a0 * a0; M[1] += a0 * a1; M[2] += a0 * a2; M[3] += a1 * a1; M[4] += a1 * a2; M[5] += a2 * a2;
      v[0] += a0 * b; v[1] += a1 * b; v[2] += a2 * b;
    }
    solve_sym3<double>(M, v, X);
    double ss = 0;
    for (int i = 0; i < n_cams; i++) {
      const int k = (int)((comb >> (4 * i)) & 15);
      if (!k) continue;
      const double* P = dlt_P[i];
      const double x = px[i][k - 1], y = py[i][k - 1];
      const double e0 = ((P[0] - x * P[8]) * X[0] + (P[1] - x * P[9]) * X[1] + (P[2] - x * P[10]) * X[2]) - (x * P[11] - P[3]);
      const double e1 = ((P[4] - y * P[8]) * X[0] + (P[5] - y * P[9]) * X[1] + (P[6] - y * P[10]) * X[2]) - (y * P[11] - P[7]);
      ss += e0 * e0;
      ss += e1 * e1;
    }
    return sqrt(ss / (2 * n));
  }
  ref::RaySet rs;
  rs.n = 0;
  for (int i = 0; i < n_cams; i++) {
    const int k = (int)((comb >> (4 * i)) & 15);
    if (k) { rs.cam[rs.n] = i; ref::make_dir(ray, i, px[i][k - 1], py[i][k - 1], rs.d[rs.n]); rs.n++; }
  }
  return solve_rays(ray, solver, rs, X, iters);
}

}  // namespace tri
