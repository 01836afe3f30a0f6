/* spn_verify.h - geometric verification of descriptor matches (part of libspn_b200.so).
 *
 * spn_verify_pairs fits one fundamental matrix or one homography to the matches of every image pair with RANSAC and
 * marks the matches that agree with it (cv2.findFundamentalMat(FM_RANSAC) / cv2.findHomography(RANSAC), COLMAP's
 * two-view geometry step).  Its inputs are the keypoint pool of spn_detect_describe and the compacted output of
 * spn_match_pairs, so it runs straight after matching without a host round trip.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`.  The pair list lives in the context's scratch buffer (guard-banded,
 * spn_check_guards).
 *
 * Geometry.  A keypoint (row, col) is the point x = (col, row, 1) in the network-input frame of features.npz.
 *   fundamental (model 0): x_b^T F x_a = 0 for a match (x_a, x_b).  F is scaled to ||F||_F = 1 with its largest-
 *       magnitude element positive (ties: the first in row-major order).  A match is an inlier iff its squared
 *       Sampson error is <= t^2, evaluated without a division as
 *           (x_b^T F x_a)^2 <= t^2 ((F x_a)_0^2 + (F x_a)_1^2 + (F^T x_b)_0^2 + (F^T x_b)_1^2).
 *   homography (model 1): x_b ~ H x_a, scaled so that H[2][2] = 1.  With p = H x_a a match is an inlier iff its
 *       squared forward transfer error is <= t^2, evaluated as (p_0 - col_b p_2)^2 + (p_1 - row_b p_2)^2 <= t^2 p_2^2.
 *
 * The rule (fp64 throughout; oracle/verify_oracle.py restates it in numpy):
 *   - Coordinates are Hartley-normalised per pair and per image (centroid at 0, mean distance sqrt(2), over all of the
 *     pair's matches); the solvers work in normalised coordinates, models are scored in pixels.  A pair whose points
 *     all coincide in a or in b gets no model.
 *   - Samples.  Hypothesis h (0, 1, 2, ...) of pair (a, b) draws s = 7 (F) or 4 (H) distinct match indices from n:
 *         key = splitmix64(seed ^ splitmix64(a << 32 | b)),  r_j = splitmix64(key ^ splitmix64(h << 32 | j)),
 *         index_j = ((r_j >> 32) * n) >> 32,   j = 0, 1, 2, ...  (64-bit unsigned arithmetic)
 *     a repeated index is skipped and the next j drawn; a sample that is not complete after 1024 draws gives no model.
 *     The key is (a, b), not the pair's position, so a pair's result does not depend on the other pairs of the call.
 *   - 7-point F: the 2-dimensional null space (F1, F2) of the 7 x 9 system from a Householder QR of its transpose, the
 *     real roots of det(alpha F1 + (1 - alpha) F2) (closed form, two Newton steps, ascending), one model per root.
 *     No model when a diagonal element of R is below 1e-9 in magnitude or the cubic's leading coefficient is below
 *     1e-12 of its largest coefficient.
 *     4-point H: the 8 x 8 DLT with h33 = 1 solved by Householder QR (same pivot rule); no model when three of the
 *     four points are collinear in a or in b (exact integer test) or |H[2][2]| < 1e-12 max |H_ij| in pixels.
 *   - Rounds of 256 hypotheses.  Each model is scored against every match of the pair; the best model is the one with
 *     the most inliers, ties to the lower hypothesis, then to the lower root.  After each round RANSAC stops once the
 *     hypotheses drawn reach log(1 - confidence) / log(1 - w^s) (w = best count / n, w^s by repeated multiplication)
 *     or max_iters rounded up to a whole round.
 *   - Refinement.  Refit on the inliers of the current model (normalised 8-point with rank-2 enforcement for F, the
 *     normalised DLT for H): the eigenvector of the smallest eigenvalue of the 9 x 9 normal matrix, summed in match
 *     order, from 12 cyclic Jacobi sweeps.  The refit replaces the model if it has at least as many inliers; this
 *     repeats while the count rises, at most 3 refits, and needs at least 8 (F) or 4 (H) inliers.
 *
 * Arguments:
 *   d_kp [N][cap][2]     int32 (row, col) keypoints: matching.extract_features' pool
 *   h_pairs [P][2]       HOST (a, b) image indices, 0 <= a, b < N, as given to spn_match_pairs
 *   d_offsets [P+1]      int64: pair p's matches are rows offsets[p] .. offsets[p+1] - 1 of d_matches
 *   d_matches [M][2]     int32 (keypoint of a, keypoint of b): matching.match_pairs' compacted output
 *   model                0 = fundamental (7-point), 1 = homography (4-point)
 *   threshold_px         t > 0, finite;  confidence in (0, 1);  1 <= max_iters <= 16777216;  seed any 64-bit value
 * Outputs (may be NULL when P == 0; d_inlier may be NULL when M == 0):
 *   d_model [P][9]       fp64 row-major model, zeros when there is none
 *   d_num_inliers [P]    int32 inliers of the final model; 0 without a model; -1 when the pair's offsets are out of
 *                        range (not 0 <= offsets[p] <= offsets[p+1] <= M, or more than cap matches), a keypoint index
 *                        is outside [0, cap) or a coordinate outside [0, 32767]
 *   d_hypotheses [P]     int32 hypotheses drawn (a multiple of 256; 0 when RANSAC did not run)
 *   d_best [P]           int32 hypothesis index of the winning minimal sample, -1 when there is none
 *   d_inlier [M]         uint8 1 where the match is an inlier of its pair's final model, else 0; rows of a pair whose
 *                        offsets are out of range are not written
 * A pair with fewer than 8 (F) or 4 (H) matches gets no model and 0 inliers.
 * Limits: 0 < N <= 1048576, 0 < cap <= 16384, 0 <= P <= 65535, M >= 0.  P == 0 is a no-op.  One 256-thread CTA per
 * pair; no atomics, bit-identical from run to run.  Scratch: P x 2 int32. */
#ifndef SPN_VERIFY_H
#define SPN_VERIFY_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

SPN_API int spn_verify_pairs(spn_ctx* ctx, const int32_t* d_kp, int N, int cap, const int32_t* h_pairs, int P,
                             const int64_t* d_offsets, const int32_t* d_matches, int64_t M, int model, double threshold_px,
                             double confidence, int max_iters, uint64_t seed, double* d_model, int32_t* d_num_inliers,
                             int32_t* d_hypotheses, int32_t* d_best, uint8_t* d_inlier, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_VERIFY_H */
