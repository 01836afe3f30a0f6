/* spn_match.h - descriptor matching over a pool of descriptor sets (part of libspn_b200.so).
 *
 * spn_match_pairs matches the sparse descriptors of many image pairs in one call without gathering them first: the
 * descriptor sets of N images sit in one pool - the desc_sparse / kp_count layout spn_detect_describe returns - and a
 * host list of (a, b) pairs says which sets to match.  Every keypoint of a gets its nearest row of b, filtered by any
 * combination of the mutual check, the ratio test and a distance threshold (cv2.BFMatcher(NORM_L2) with crossCheck,
 * knnMatch(k=2) + Lowe's ratio test, and a max-distance cut).
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`.  The pair list and the mutual check's scratch live in the context's scratch buffer
 * (guard-banded, spn_check_guards).
 */
#ifndef SPN_MATCH_H
#define SPN_MATCH_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Matches of P pairs (a, b) of a pool of N descriptor sets.
 *   d_desc [N][cap][C]   fp32 descriptors, row i of set n valid for i < d_count[n] (counts are clamped to [0, cap])
 *   d_count [N]          int32
 *   h_pairs [P][2]       HOST list of (a, b), 0 <= a, b < N; a == b is allowed
 * Distances: d^2(i, j) = max(|a_i|^2 + |b_j|^2 - 2 a_i.b_j, 0) with the dot product on the tensor cores from fp16
 * (hi, lo) splits of the fp32 values (hi.hi + hi.lo + lo.hi, fp32 accumulation), exactly as spn_mutual_nn_match.
 * For keypoint i of a: best = the smallest d over the rows of b (ties to the lower index), second = the smallest over
 * the other rows (+inf when b has one row).  i -> best_j is kept iff
 *   mutual == 0, or i is the nearest row of a to b's row best_j (same rule in the other direction);
 *   ratio == 0, or d_best < ratio * d_second   (fp32, each operation rounded on its own; cv2's strict test);
 *   d_best <= max_dist                         (+inf: no threshold)
 * where d = sqrt(d^2) in fp32.
 * Outputs (may be NULL when P == 0: nothing is written):
 *   d_match [P][cap]     int32 index into b, or -1 (not kept, or i >= count of a)
 *   d_dist  [P][cap]     fp32 d_best of kept matches, 0 elsewhere
 * With mutual = 1, ratio = 0, max_dist = +inf the outputs equal spn_mutual_nn_match's on the gathered pairs.
 * Limits: 0 < N <= 1048576, 0 < cap <= 16384, C > 0 a multiple of 64, 0 <= P <= 65535, 0 <= ratio <= 1, max_dist not
 * NaN.  P == 0 is a no-op.  Scratch: P x (2 + cap) int32 with mutual, P x 2 without.  Deterministic: no atomics. */
SPN_API int spn_match_pairs(spn_ctx* ctx, const float* d_desc, const int32_t* d_count, int N, int cap, int C,
                            const int32_t* h_pairs, int P, int mutual, float ratio, float max_dist, int32_t* d_match,
                            float* d_dist, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_MATCH_H */
