/* tri_oracle_robust.h -- CPU restatement of the outlier-robust batch (tri_triangulate_points_robust).
 * TEST INFRASTRUCTURE ONLY (see tri_oracle.h). */
#ifndef TRI_ORACLE_ROBUST_H
#define TRI_ORACLE_ROBUST_H
#include "tri_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

/* Two-view consensus over the valid views with threshold tau (pixels), refit over the winner's inliers, serially in FP64.
 * xy as in orc_triangulate_points (double pairs, (-1,-1) = missing), at most 32 camera rows.  out_mask = inlier set,
 * out_err = RMS pixel reprojection error (NaN without consensus, 0 on a frame with < 2 views).  out_margin[f]: the
 * smallest |r_c - tau| / tau over the threshold tests of the hypotheses whose inlier count is at least the winner's minus
 * one, and the relative sum-of-squares gap between the winner and the best different set with its count -- a frame with a
 * small margin may legitimately decide differently under other rounding.  Without allow_too_few, returns ORC_ERR_TOO_FEW
 * at the first frame with < 2 views (*first_bad = that frame). */
int orc_triangulate_points_robust(const orc_camera* cams, int n_cams, int n_point_cams, const double* xy, int64_t n_frames,
                                  double tau, int allow_too_few, double* out_xyz, double* out_err, uint32_t* out_mask,
                                  double* out_margin, int64_t* first_bad);

#ifdef __cplusplus
}
#endif
#endif
