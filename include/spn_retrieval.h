/* spn_retrieval.h - image retrieval over descriptor pools (part of libspn_b200.so).
 *
 * Two building blocks of vocabulary-based retrieval (VLAD) and of the k-means that learns the vocabulary:
 *   spn_knn            the k nearest rows of a train set for every row of a query set (word assignment: k = 1 against
 *                      the vocabulary; image retrieval: k neighbours of every global descriptor among the others);
 *   spn_residual_sums  per image and word, the sum of the residuals x - c_w of the keypoints assigned to word w.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`, the caller's device saved and restored.  No float atomics: every result is the
 * same run to run.  Neither call uploads anything from the host.
 */
#ifndef SPN_RETRIEVAL_H
#define SPN_RETRIEVAL_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The k nearest train rows of every query row.
 *   d_query [nq][C], d_train [nt][C]   fp32, row-major
 *   d_index [nq][k]                    int32 train row, ascending distance; -1 in slots past the usable train rows
 *   d_dist2 [nq][k]                    fp32 squared distance; +inf in those slots
 * Distances are spn_match_pairs's: d^2 = max(|q|^2 + |t|^2 - 2 q.t, 0) with the dot product on the tensor cores from
 * fp16 (hi, lo) splits (hi.hi + hi.lo + lo.hi, fp32 accumulation), so a pair of rows gets the same d^2 bits in both
 * calls.  Rows are taken in ascending train index and enter the list only on a strict '<': equal distances keep the
 * lower index first.  exclude_self = 1 (requires nq == nt: the same set) skips train row i for query row i.
 * Limits: 1 <= k <= 128, C a positive multiple of 64 up to 65536, 0 <= nq, nt <= 2^26.  nq == 0 is a no-op (pointers
 * may be NULL); nt == 0 fills every row with -1 / +inf (d_train may be NULL). */
SPN_API int spn_knn(spn_ctx* ctx, const float* d_query, int nq, const float* d_train, int nt, int C, int k, int exclude_self,
                    int32_t* d_index, float* d_dist2, spn_stream stream);

/* Residual sums of a descriptor pool against a vocabulary.
 *   d_desc [N][cap][C]   fp32, row i of image n valid for i < clamp(d_count[n], 0, cap) (spn_detect_describe's layout)
 *   d_count [N]          int32
 *   d_assign [N][cap]    int32 word of every row; values outside [0, K) are skipped
 *   d_words [K][C]       fp32 vocabulary
 *   d_sums [N][K][C]     fp32: sums[n][w] = sum over the valid rows i with assign[n][i] == w, in ascending i, of
 *                        (x_i - c_w); every subtraction and addition is a separately rounded fp32 operation (0 when w
 *                        has no rows)
 *   d_n [N][K]           int32 number of those rows
 * VLAD is the normalised sums; a k-means step is c_w + sum_n sums[n][w] / sum_n n[n][w].
 * Limits: 0 <= N <= 2^26, 1 <= cap <= 2^20, 1 <= C <= 65536, 1 <= K <= 65536.  N == 0 is a no-op. */
SPN_API int spn_residual_sums(spn_ctx* ctx, const float* d_desc, const int32_t* d_count, const int32_t* d_assign,
                              const float* d_words, int N, int cap, int C, int K, float* d_sums, int32_t* d_n,
                              spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_RETRIEVAL_H */
