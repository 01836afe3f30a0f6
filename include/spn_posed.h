/* spn_posed.h - keypoint reprojection between posed views for the posed-view evaluation (part of libspn_b200.so).
 *
 * evaluations/posed_evaluation.py measures detectors and descriptors on posed multi-view scenes (data/PosedViews.py):
 * repeatability, match accuracy and relative-pose AUC.  spn_posed_reproject is its geometric ground truth: it maps every
 * keypoint of view a into view b through a's ray depth and both camera poses, decides whether the point is visible in b
 * (in front of the camera, inside the image, not occluded), and compacts the visible points into the two sets that
 * spn_repeatability_counts takes.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`.  The pair list is uploaded into the context's scratch buffer (guard-banded,
 * spn_check_guards).
 */
#ifndef SPN_POSED_H
#define SPN_POSED_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Reprojection of the keypoints of P view pairs (a, b) of one chunk of V views of H x W pixels.
 *   d_kp [V][max_kp][2]     int32 (row, col) keypoints, d_kp_count [V] their counts (counts above max_kp are clamped;
 *                           keypoints outside the image are never visible) - spn_detect_describe's lists
 *   d_depth [V][H][W]       distance along each pixel's ray
 *   d_K [V][9], d_R [V][9], d_t [V][3]   each view's intrinsics and camera-to-world pose (X_world = R X_cam + t)
 *   h_pairs [P][2]          HOST list of (a, b); a == b is allowed
 *   depth_tol               relative tolerance of the occlusion test
 * Geometry of keypoint (r, c) of view a in view b, in fp64 with every product, sum, quotient and square root rounded
 * on its own (no FMA contraction), in this order:
 *   Kinv_a, Rinv_b          adjugate / determinant (torch.linalg.inv's 3x3 formula, not rounded to float)
 *   ray = Kinv_a (c, r, 1)  row i: (m0 c + m1 r) + m2
 *   X = ray / |ray| * d_a(r, c)                     |v| = sqrt((v0^2 + v1^2) + v2^2)
 *   Y = Rinv_b ((R_a X + t_a) - t_b)                matrix row i: (m0 x + m1 y) + m2 z
 *   p = K_b Y, row' = p1 / p2, col' = p0 / p2
 * The keypoint is visible in b when d_a(r, c) is finite and > 0, Y2 > 0, 0 <= row' <= H-1, 0 <= col' <= W-1, and at
 * the nearest pixel (floor(row' + 0.5), floor(col' + 0.5)) b's depth d_b is finite, > 0 and ||Y| - d_b| <= depth_tol d_b.
 * Outputs (may be NULL when P == 0: nothing is written):
 *   d_proj [P][max_kp][2]   double (row', col') of a's keypoints in b; NaN where the chain is not finite, for
 *                           keypoints outside the image and for slots at or past the count
 *   d_vis [P][2][max_kp]    int32 flags: [q][0][i] keypoint i of a visible in b, [q][1][i] keypoint i of b visible in a
 *   d_set1 [P][max_kp][2]   double: a's visible keypoints at (row', col') in b, in keypoint order
 *   d_set2 [P][max_kp][2]   double: b's keypoints that are visible in a, at their own (row, col), in keypoint order
 *   d_set_count [P][2]      int32 sizes of set 1 and set 2; set slots past the size hold NaN
 * The two sets are in b's pixel frame and feed spn_repeatability_counts as they are.
 * Limits: 0 < H, W <= 32767, V > 0, max_kp > 0, 0 <= P <= 65535, pair indices in [0, V), depth_tol finite and >= 0.
 * P == 0 is a no-op.  Deterministic: no float atomics. */
SPN_API int spn_posed_reproject(spn_ctx* ctx, const int32_t* d_kp, const int32_t* d_kp_count, int max_kp, const float* d_depth,
                                const float* d_K, const float* d_R, const float* d_t, int V, int H, int W, int P,
                                const int32_t* h_pairs, double depth_tol, double* d_proj, int32_t* d_vis, double* d_set1,
                                double* d_set2, int32_t* d_set_count, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_POSED_H */
