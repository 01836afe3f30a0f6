/* spn_nerf.h - multi-view label fusion of ExportNeRFDetections (part of libspn_b200.so).
 *
 * ExportNeRFDetections (engine_solvers/export.py:225-366 of the reference) averages, for every target view j of a batch,
 * the heatmap of j with the heatmaps of source views k re-projected into j (spn_nerf_splat after warp_points_NeRF and
 * filter_points).  spn_nerf_fuse does that for every target of a batch in one pass: no per-pair launches, no per-pair
 * H x W maps in memory, no host synchronisation.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`.  Scratch lives in the context's scratch buffer (guard-banded, spn_check_guards).
 */
#ifndef SPN_NERF_H
#define SPN_NERF_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Fused NeRF pseudo-label heatmaps of one batch of V views of H x W pixels.
 *   d_prob [V][H][W]        each view's prob_heatmap
 *   d_kp [V][max_kp][2]     int32 (row, col) post-NMS keypoints in row-major order, d_kp_count [V] their counts (counts
 *                           above max_kp are clamped; keypoints outside the image are ignored) - spn_detect_describe's lists
 *   d_depth [V][H][W]       distance along each pixel's ray
 *   d_K [V][9], d_R [V][9], d_t [V][3]   intrinsics and camera-to-world poses (X_world = R X_cam + t)
 *   h_targets [n_targets]   HOST: view index j of every target
 *   h_pair_offsets [n_targets+1], h_pair_src [h_pair_offsets[n_targets]]   HOST CSR list: the source views k of target t
 *                           are h_pair_src[h_pair_offsets[t] .. h_pair_offsets[t+1]), in summation order, repeats allowed
 *   d_out [n_targets][H][W] (may be NULL when n_targets == 0: nothing is written)
 * For target t with view j and sources k_1..k_n:
 *   out[t] = (prob[j] + splat(j,k_1) + ... + splat(j,k_n)) / float(1 + n)        (sum left to right; the division is
 *                                                      evaluated as a multiplication by the fp32 reciprocal, as torch does)
 * splat(j,k) = ExportNeRFDetections.reproject(prob[k], kp[k], depth[k], K[j], R[k], t[k], R[j], t[j]): the keypoints of k
 * through the depth rule of warp_points_NeRF (the pixel's own depth on the border, row <= 2 | col <= 2 | row >= H-2 |
 * col >= W-2, or where its 5x5 patch spans < 0.03, else the patch minimum) and its fp32 chain K^-1 (x,y,1) -> unit ray
 * -> x depth -> R_k X + t_k -> R_j^-1 X - R_j^-1 t_j -> K X -> / z, with K[j] on both sides; filter_points
 * (0 <= row < H-1, 0 <= col < W-1); the i-th surviving point paired with the i-th ORIGINAL keypoint (the reference's
 * quirk); spn_nerf_splat's ordered 3x3 / single-pixel copy (later points overwrite earlier ones).
 * The pair list is checked on the host (indices in [0, V), offsets starting at 0 and non-decreasing) and uploaded with
 * one asynchronous copy.  Limits: 2 < H, W <= 32767, max_kp > 0, 0 <= n_targets <= 65535.  Deterministic: no float
 * atomics. */
SPN_API int spn_nerf_fuse(spn_ctx* ctx, const float* d_prob, const int32_t* d_kp, const int32_t* d_kp_count, int max_kp,
                          const float* d_depth, const float* d_K, const float* d_R, const float* d_t, int V, int H, int W,
                          int n_targets, const int32_t* h_targets, const int32_t* h_pair_offsets, const int32_t* h_pair_src,
                          float* d_out, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_NERF_H */
