/* tri_oracle_robust.c -- CPU restatement of the CUDA engine's outlier-robust batch (tri_triangulate_points_robust).
 * TEST INFRASTRUCTURE ONLY, like tri_oracle.c (whose orc_matrix_point it builds on; the two are linked together into
 * liboracle_robust.so).  Not a reference function: the contract of include/tri_b200.h restated serially in FP64.
 * Hypotheses and the refit are orc_matrix_point solves (the reference's pinv-SVD DLT). */
#include "tri_oracle_robust.h"

#include <math.h>
#include <stdlib.h>

#define ROBUST_MAX_CAMS 32 /* validity / inlier masks are one uint32 per frame */

static void robust_project(const orc_camera* cam, const double X[3], double x, double y, double* w, double* r2) {
  const double* P = cam->P;
  *w = P[8] * X[0] + P[9] * X[1] + P[10] * X[2] + P[11];
  const double px = (P[0] * X[0] + P[1] * X[1] + P[2] * X[2] + P[3]) / *w;
  const double py = (P[4] * X[0] + P[5] * X[1] + P[6] * X[2] + P[7]) / *w;
  *r2 = (px - x) * (px - x) + (py - y) * (py - y);
}

typedef struct { int usable, count; uint32_t inl; double sum; double r[ROBUST_MAX_CAMS], w[ROBUST_MAX_CAMS]; } robust_hyp;

int orc_triangulate_points_robust(const orc_camera* cams, int n_cams, int n_point_cams, const double* xy, int64_t n_frames,
                                  double tau, int allow_too_few, double* out_xyz, double* out_err, uint32_t* out_mask,
                                  double* out_margin, int64_t* first_bad) {
  const int n = n_point_cams < n_cams ? n_point_cams : n_cams;
  if (n > ROBUST_MAX_CAMS) return ORC_ERR_DIM;
  robust_hyp* hyp = (robust_hyp*)malloc(sizeof(robust_hyp) * (ROBUST_MAX_CAMS * (ROBUST_MAX_CAMS - 1) / 2));
  if (first_bad) *first_bad = -1;
  for (int64_t f = 0; f < n_frames; f++) {
    double px[ROBUST_MAX_CAMS], py[ROBUST_MAX_CAMS];
    uint32_t V = 0;
    for (int c = 0; c < n; c++) {
      px[c] = xy[2 * ((size_t)c * n_frames + f)];
      py[c] = xy[2 * ((size_t)c * n_frames + f) + 1];
      if (px[c] != -1 && py[c] != -1) V |= 1u << c;
    }
    double* X = out_xyz + 3 * f;
    X[0] = X[1] = X[2] = 0;
    out_mask[f] = V;
    out_err[f] = 0;
    out_margin[f] = HUGE_VAL;
    if (__builtin_popcount(V) < 2) {
      if (first_bad && *first_bad < 0) *first_bad = f;
      if (!allow_too_few) { free(hyp); return ORC_ERR_TOO_FEW; }
      continue;
    }
    int nh = 0, best = -1;
    for (int i = 0; i < n; i++) {
      if (!(V >> i & 1)) continue;
      for (int j = i + 1; j < n; j++) {
        if (!(V >> j & 1)) continue;
        robust_hyp* h = &hyp[nh++];
        const int idx[2] = {i, j};
        const double pix[4] = {px[i], py[i], px[j], py[j]};
        double H[3];
        orc_matrix_point(cams, 2, idx, pix, H);
        h->inl = 0; h->sum = 0; h->usable = 1;
        for (int c = 0; c < n; c++) {
          if (!(V >> c & 1)) continue;
          double w, r2;
          robust_project(&cams[c], H, px[c], py[c], &w, &r2);
          h->w[c] = w;
          h->r[c] = sqrt(r2);
          if ((c == i || c == j) && !(w > 0)) h->usable = 0;
          if (w > 0 && r2 <= tau * tau) { h->inl |= 1u << c; h->sum += r2; }
        }
        h->count = __builtin_popcount(h->inl);
        if (!h->usable || h->count < 2) continue;
        if (best < 0 || h->count > hyp[best].count || (h->count == hyp[best].count && h->sum < hyp[best].sum)) best = nh - 1;
      }
    }
    /* margin: threshold tests of the hypotheses that one flipped test could make tie or win, and the sum-of-squares gap
     * to the best different set with the winner's count */
    const int need = best >= 0 ? hyp[best].count - 1 : 0;
    double margin = HUGE_VAL;
    for (int k = 0; k < nh; k++) {
      const robust_hyp* h = &hyp[k];
      if (!h->usable || h->count < need) continue;
      for (int c = 0; c < n; c++)
        if ((V >> c & 1) && h->w[c] > 0) margin = fmin(margin, fabs(h->r[c] - tau) / tau);
      if (best >= 0 && h->count == hyp[best].count && h->inl != hyp[best].inl) {
        const double s = fmax(h->sum, hyp[best].sum);
        margin = fmin(margin, s > 0 ? fabs(h->sum - hyp[best].sum) / s : 0.0);
      }
    }
    out_margin[f] = margin;
    if (best < 0) { out_mask[f] = 0; out_err[f] = NAN; continue; }
    const uint32_t I = hyp[best].inl;
    int idx[ROBUST_MAX_CAMS], m = 0;
    double pix[2 * ROBUST_MAX_CAMS];
    for (int c = 0; c < n; c++)
      if (I >> c & 1) { idx[m] = c; pix[2 * m] = px[c]; pix[2 * m + 1] = py[c]; m++; }
    orc_matrix_point(cams, m, idx, pix, X);
    double s = 0;
    for (int k = 0; k < m; k++) {
      double w, r2;
      robust_project(&cams[idx[k]], X, pix[2 * k], pix[2 * k + 1], &w, &r2);
      s += r2;
    }
    out_mask[f] = I;
    out_err[f] = sqrt(s / m);
  }
  free(hyp);
  return ORC_OK;
}
