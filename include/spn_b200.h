/* spn_b200.h - C ABI of the B200-native SuperPoint/MagicPoint inference hot path.
 *
 * The reference (AliYoussef97/SuperPoint-NeRF-Pytorch) is pure Python; the functions below are what a
 * ctypes/cffi binding inside the reference would call in place of the PyTorch/kornia/torchvision calls
 * cited next to each entry point (paths relative to superpoint/superpoint/ in the reference).
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; h_* is a HOST pointer;
 *   - shapes are explicit ints, tensors are dense row-major in the order written in the comment;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no implicit synchronisation
 *     except when the context's internal workspace has to grow (first call with a bigger shape);
 *   - return 0 on success, a negative SPN_E_* code on failure; spn_last_error() gives the message
 *     (thread-local); no C++ exception crosses the boundary;
 *   - CUDA only, sm_100a only: there is no CPU fallback.
 */
#ifndef SPN_B200_H
#define SPN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SPN_API __attribute__((visibility("default")))
#else
#define SPN_API
#endif

typedef struct spn_ctx spn_ctx;
typedef void* spn_stream; /* cudaStream_t */

enum {
  SPN_OK = 0,
  SPN_E_INVALID = -1, /* bad argument / unsupported shape */
  SPN_E_CUDA = -2,    /* CUDA runtime error */
  SPN_E_STATE = -3,   /* weights missing, encoder not run, ... */
  SPN_E_NOMEM = -4
};

/* layer ids, in the order of the reference's state-dict prefixes
 * (models/model_utils/VGG_Backbone.py:44-58, models/model_utils/heads.py:11-13,54-56) */
enum {
  SPN_L_BLOCK1 = 0, SPN_L_BLOCK2, SPN_L_BLOCK3, SPN_L_BLOCK4, SPN_L_BLOCK5, SPN_L_BLOCK6, SPN_L_BLOCK7, SPN_L_BLOCK8,
  SPN_L_CONVPA = 8, SPN_L_CONVPB = 9, SPN_L_CONVDA = 10, SPN_L_CONVDB = 11, SPN_NUM_LAYERS = 12
};

/* numeric mode of the convolutions */
enum {
  SPN_MODE_FP32 = 0, /* strict: fp32 FFMA convolutions (1e-4 parity gate)                       */
  SPN_MODE_F16 = 1,  /* fast: tcgen05 implicit GEMM, fp16 operands, fp32 accumulate (5e-3 gate) */
  SPN_MODE_BF16 = 2, /* fast: tcgen05 implicit GEMM, bf16 operands, fp32 accumulate             */
  SPN_MODE_F16X3 = 3 /* strict on the tensor cores: activations and weights split into fp16 (hi, lo) pairs, three
                        tcgen05 MMAs per product (hi.hi + hi.lo + lo.hi), fp32 accumulate (1e-4 parity gate)  */
};

SPN_API const char* spn_last_error(void);
SPN_API int spn_version(void);

/* Context: device weights, workspace, TMA descriptors.  One per (process, GPU). */
SPN_API int spn_create(spn_ctx** out, int device);
SPN_API int spn_destroy(spn_ctx* ctx);

/* Options of the tensor-core path (read when a launch is planned, never from the environment): "fuse_front" (warp +
 * block_1 + block_2 in one kernel) and "fuse_head" (convPb + softmax + depth-to-space in one kernel), both default 1;
 * 0 selects the unfused kernels.  "ws_guard" (default 0): see spn_check_guards.  Any other name is SPN_E_INVALID. */
SPN_API int spn_set_option(spn_ctx* ctx, const char* name, int value);

/* BN fold + pack + upload of one VGG_Block (conv2d + BatchNorm2d eval, eps as given).
 * Replaces nn.Conv2d/nn.BatchNorm2d parameter storage (VGG_Backbone.py:11-14) as loaded by engine.py:108-117.
 * h_w [cout][cin][k][k], h_b/h_gamma/h_beta/h_mean/h_var [cout] are HOST fp32 arrays. */
SPN_API int spn_pack_weights(spn_ctx* ctx, int layer, const float* h_w, const float* h_b, const float* h_gamma,
                     const float* h_beta, const float* h_mean, const float* h_var, float eps, int cout, int cin,
                     int ksize, spn_stream stream);

/* One VGG_Block.forward (VGG_Backbone.py:23-36): conv + folded BN (+ ReLU) (+ 2x2 max-pool), NCHW fp32 in and out.
 * d_in [B][cin][H][W] -> d_out [B][cout][H or H/2][W or W/2].  In the tensor-core modes the activations are rounded
 * to fp16/bf16 on the way in (this entry point exists for layer-level parity tests and for callers that want a
 * single block; the fused forward keeps activations in the 16-bit C8 layout between layers). */
SPN_API int spn_conv_layer(spn_ctx* ctx, int layer, int mode, const float* d_in, int B, int H, int W, int relu, int pool,
                           float* d_out, spn_stream stream);

/* VGG_BACKBONE.forward (VGG_Backbone.py:60-71): d_images [B][H][W] fp32 in [0,1] -> feature map kept inside ctx
 * (H, W multiples of 8). */
SPN_API int spn_encoder_forward(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode, spn_stream stream);

/* Fused K.warp_perspective(image, H) (export.py:51) + VGG_BACKBONE.forward for the homography-adaptation slots
 * slot = i*(n_h+1) + j (j == 0: image i itself, j >= 1: image i warped by homography j-1) with
 * slot_begin <= slot < slot_begin + n_slots; tensor-core modes only.  The warped images are never written to memory:
 * the warp is evaluated inside the first convolution kernel.  d_images [n_images][H][W], d_hinv [n_images][n_h][9] =
 * the PIXEL-space inverses H_ij^-1 (export.py:49; kornia samples the source at H^-1 p).  The operands downstream are 16
 * bits wide, so this entry point does not need kornia's bit-exact normalised chain; the validity masks that go with
 * these forwards still come from spn_warp_batch.  Leaves the feature map of the n_slots forwards inside ctx. */
SPN_API int spn_encoder_forward_ha(spn_ctx* ctx, const float* d_images, int n_images, const float* d_hinv, int n_h,
                                   int slot_begin, int n_slots, int H, int W, int mode, spn_stream stream);

/* Detector_head.forward up to prob_heatmap (heads.py:17-28): convPa, convPb, softmax(65), drop dustbin,
 * pixel_shuffle(8).  d_mask (nullable) [B][H][W] u8 multiplies the heatmap (export.py:70).
 * d_logits (nullable) [B][65][H/8][W/8]; d_prob [B][H][W]. */
SPN_API int spn_detector_head_forward(spn_ctx* ctx, int B, int H, int W, int mode, const uint8_t* d_mask, float* d_logits,
                              float* d_prob, spn_stream stream);

/* Descriptor_head.forward up to desc_raw (heads.py:61-63): convDa, convDb.  d_desc_raw [B][256][H/8][W/8]. */
SPN_API int spn_descriptor_head_forward(spn_ctx* ctx, int B, int H, int W, int mode, float* d_desc_raw, spn_stream stream);

/* F.interpolate(bicubic, x grid, align_corners=False) + F.normalize(p=2, dim=1) (heads.py:65-66), dense.
 * d_desc_raw [B][C][Hc][Wc] -> d_desc [B][C][Hc*grid][Wc*grid]. */
SPN_API int spn_dense_descriptors(spn_ctx* ctx, const float* d_desc_raw, int B, int C, int Hc, int Wc, int grid, float* d_desc,
                          spn_stream stream);

/* The same value as dense desc[:, :, y, x] evaluated only at keypoints (what the consumers index:
 * evaluations/descriptor_evaluation.py:67-69).  d_kp [B][max_kp][2] int32 (row, col), d_kp_count [B];
 * d_out [B][max_kp][C].  interp: 0 = bicubic (reference parity), 1 = bilinear. */
SPN_API int spn_sample_descriptors(spn_ctx* ctx, const float* d_desc_raw, int B, int C, int Hc, int Wc, int grid,
                           const int32_t* d_kp, const int32_t* d_kp_count, int max_kp, int interp, float* d_out,
                           spn_stream stream);

/* SuperPoint.forward (models/SuperPoint.py:17-30) + the keypoint extraction every consumer performs on its output
 * (nonzero(prob_heatmap_nms), desc[:, y, x]: evaluations/descriptor_evaluation.py:55-69) in ONE call: encoder, detector
 * head, box_nms + top-k once, descriptor head, descriptors at the keypoints only (no dense 315 MB map).
 * d_images [B][H][W]; outputs: d_logits [B][65][H/8][W/8] (nullable), d_prob [B][H][W], d_nms [B][H][W] (nullable),
 * d_pred [B][H][W] int32 (nullable), d_kp [B][max_kp][2] int32 (row, col) row-major order, d_kp_count [B] (true count),
 * d_desc_raw [B][256][H/8][W/8] and d_desc_sparse [B][max_kp][256] (both or neither; rows >= count are zero).
 * interp: 0 = bicubic (the reference's dense desc evaluated at the keypoint), 1 = bilinear. */
SPN_API int spn_detect_describe(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode, float nms_size, float iou,
                                float det_thresh, int top_k, int interp, float* d_logits, float* d_prob, float* d_nms,
                                int32_t* d_pred, int32_t* d_kp, int32_t* d_kp_count, int max_kp, float* d_desc_raw,
                                float* d_desc_sparse, spn_stream stream);

/* box_nms (sp_utils.py:4-28) + threshold (heads.py:41 / export.py:123) + nonzero (export.py:125), batched.
 * d_prob [B][H][W]; outputs (each nullable): d_nms [B][H][W] fp32, d_pred [B][H][W] int32 (= nms >= det_thresh),
 * d_kp [B][max_kp][2] int32 (row, col) in row-major order, d_kp_count [B] (true count, may exceed max_kp).
 * 0 < size <= 8; box sizes up to 4 (the reference default) take the bit-plane kernel, larger ones the generic one;
 * the result is bit-identical to torchvision.ops.nms on the same heatmap either way. */
SPN_API int spn_box_nms_topk(spn_ctx* ctx, const float* d_prob, int B, int H, int W, float size, float iou, float min_prob,
                     int top_k, float det_thresh, float* d_nms, int32_t* d_pred, int32_t* d_kp, int32_t* d_kp_count,
                     int max_kp, spn_stream stream);

/* Statistics of the last spn_box_nms_topk call with the same (B,H,W): h_out[0] = global rounds (grid-wide
 * synchronisations), h_out[1] = tile-local iterations, h_out[2] = tile visits.  Synchronises the device. */
SPN_API int spn_nms_stats(spn_ctx* ctx, int B, int H, int W, int64_t* h_out);

/* Memory-safety probe (no reference counterpart; compute-sanitizer is not available on the target pool).  The
 * context's workspace and scratch buffer are allocated with a 64 KB band of 0xA5 before and after the usable range,
 * and the tensor-core workspace plan leaves 4 KB gaps between its regions which option "ws_guard" = 1 paints before
 * every encoder pass.  *h_bad = number of guard bytes that no longer hold the pattern (0 = no kernel wrote outside
 * its region).  Synchronises the device. */
SPN_API int spn_check_guards(spn_ctx* ctx, int64_t* h_bad);

/* ExportDetections.step warp part (export.py:51-66): for every image i < n_images and homography j < n_h
 *   slot = i*(n_h+1) + 1 + j : d_warped[slot] = warp_perspective(image_i, H_ij, bilinear, align_corners=True)
 *                              d_mask[slot]   = erosion(warp_perspective(ones, H_ij, nearest), ellipse(2*margin))
 *   slot = i*(n_h+1)         : the image itself, mask = 1 (identity forward, export.py:93)
 * d_ainv [n_images][n_h][9] fp32 are kornia's sampling matrices of H_ij in NORMALISED coordinates,
 *   Ainv = torch.inverse(normalize_homography(H_ij, (H,W), (H,W)))      (what K.warp_perspective builds internally),
 * the "fwd" output of spn_kornia_matrices.  The kernel follows kornia's fp32 coordinate chain operation for operation
 * (create_meshgrid -> bmm -> 1/(z+1e-8) -> grid_sample unnormalise / nearbyint / ATen bilinear weights), so masks and
 * warped pixels are BIT-IDENTICAL to the reference's CPU run when Ainv carries the reference's bits.
 * d_images [n_images][H][W]; d_warped [n_images*(n_h+1)][H][W] fp32; d_mask same shape u8.  d_warped may be NULL
 * (mask only: the fused encoder spn_encoder_forward_ha warps on the fly).
 * margin = 0 skips the erosion (Homographic_aug.compute_valid_mask with erosion = 0, homographic_augmentation.py:109-127).
 * Limits: 0 <= margin <= 8, n_images*(n_h+1) <= 65535 per call, W <= 8192, H, W >= 2. */
SPN_API int spn_warp_batch(spn_ctx* ctx, const float* d_images, int n_images, const float* d_ainv, int n_h, int H, int W,
                   int margin, float* d_warped, uint8_t* d_mask, spn_stream stream);

/* ExportDetections.step projection + homography_adaptation aggregation (export.py:72-77,106-114):
 * for every image: out(p) = [ prob_0(p) + sum_j count_j(p) * bilinear(prob_j, H_j p) ] / [ 1 + sum_j count_j(p) ]
 * with count_j = erosion(nearest warp of ones by H_j^-1)  (aggregation 0 = 'sum'), or the max over the same
 * terms (aggregation 1 = 'max').  d_probs [n_images][n_h+1][H][W] (already multiplied by the masks),
 * d_ainv_bwd [n_images][n_h][9] fp32 = kornia's sampling matrices of the INVERSE homographies,
 *   torch.inverse(normalize_homography(torch.inverse(H_ij)))            (export.py:49,55,72),
 * the "bwd" output of spn_kornia_matrices; same bit-exact coordinate chain as spn_warp_batch.  d_out [n_images][H][W].
 * Limits: 1 <= margin <= 8, n_h <= 255, (n_h+1)*H*W < 2^30. */
SPN_API int spn_ha_aggregate(spn_ctx* ctx, const float* d_probs, const float* d_ainv_bwd, int n_images, int n_h, int H, int W,
                     int margin, int aggregation, float* d_out, spn_stream stream);

/* Homographic_aug.sample_homography (data/data_utils/homographic_augmentation.py:21-106) on the device:
 * counter-based RNG keyed by (seed, first_index + i); truncated normals, scale/angle choice, translation,
 * 4-point DLT solve in fp64, fp32 inverse.  Writes d_h [count][9] (what the reference returns) and
 * d_hinv [count][9].  Statistically equivalent to, not bit-equal with, the numpy-RNG reference. */
typedef struct spn_homography_params {
  int translation, rotation, scaling, perspective;
  float scaling_amplitude, perspective_amplitude_x, perspective_amplitude_y, patch_ratio, max_angle,
      translation_overflow;
  int n_scales, n_angles, allow_artifacts;
} spn_homography_params;
SPN_API int spn_sample_homographies(spn_ctx* ctx, const spn_homography_params* params, uint64_t seed, uint64_t first_index,
                            int count, int H, int W, float* d_h, float* d_hinv, spn_stream stream);

/* kornia.geometry normalize_homography + torch.inverse for a batch of pixel-space homographies d_h [count][9]
 * (the matrices K.warp_perspective derives at export.py:51-55,72): d_ainv_fwd = inverse(N (H N^-1)) and d_ainv_bwd =
 * the same for H^-1, N = normal_transform_pixel(H, W).  Device arithmetic (adjugate inverse): equal to the reference's
 * LAPACK inverse to a few ulp, not bit for bit - callers that need bit-identical masks pass matrices computed with the
 * reference's own torch calls (the Python binding does so whenever the homographies come from the host). */
SPN_API int spn_kornia_matrices(spn_ctx* ctx, const float* d_h, int count, int H, int W, float* d_ainv_fwd, float* d_ainv_bwd,
                                spn_stream stream);

/* Loader pre-processing of one decoded grayscale image (data/COCO.py:66-76 ratio_preserving_resize + the /255 of
 * COCO.py:135; data/HPatches.py:64-72): bilinear resize to new_h x new_w (align_corners=False, as kornia.resize ->
 * F.interpolate), centre crop at (crop_top, crop_left) to H x W (zero padded when the resized image is smaller, as
 * torchvision center_crop does), divide by `divisor`.  d_src [H0][W0] uint8 (src_is_u8 != 0) or fp32; d_out [H][W]. */
SPN_API int spn_resize_crop(spn_ctx* ctx, const void* d_src, int src_is_u8, int H0, int W0, int new_h, int new_w,
                            int crop_top, int crop_left, int H, int W, float divisor, float* d_out, spn_stream stream);

/* 3x3 inverse, fp32, batched (export.py:49 torch.inverse). d_in/d_out [count][9]. */
SPN_API int spn_invert3x3(spn_ctx* ctx, const float* d_in, int count, float* d_out, spn_stream stream);

/* ---- on-GPU evaluation of the exports (evaluations/detector_evaluation.py, evaluations/descriptor_evaluation.py) ---- */

/* np.where(prob > 0) + warp_keypoints / keep_true_keypoints / filter_keypoints + select_k_best
 * (detector_evaluation.py:152-206, descriptor_evaluation.py:17-52), per map.  d_prob [B][H][W] (an NMS'd heatmap);
 * h_warp HOST double [B][9] (nullable): homography applied to (x = col, y = row, 1) in fp64 like numpy; a point is kept
 * iff its warped position satisfies 0 <= row' < bound_h and 0 <= col' < bound_w.  emit_warped = 0 writes the original
 * integer (row, col) (keep_true_keypoints), 1 writes the warped (row', col') (warp_keypoints + filter_keypoints).
 * Output: the keep_k most probable points in ASCENDING order of probability (select_k_best): d_pts [B][keep_k][2] double,
 * d_score [B][keep_k], d_count [2*B]: [b] = points written, [B + b] = candidates before the selection (at most 16384
 * candidates per map are held on chip; a larger count means the result is truncated and the caller must fall back). */
SPN_API int spn_select_keypoints(spn_ctx* ctx, const float* d_prob, int B, int H, int W, const double* h_warp, int bound_h,
                                 int bound_w, int emit_warped, int keep_k, double* d_pts, float* d_score, int32_t* d_count,
                                 spn_stream stream);

/* Repeatability counts (detector_evaluation.py:214-233): d_pts1 / d_pts2 [B][cap][2] double with d_n1 / d_n2 [B] valid
 * points; d_out [B][4] = {N1, N2, count1, count2}, count1 = points of set 1 whose nearest point of set 2 lies within
 * `thresh` (Euclidean, fp64), count2 the converse.  repeatability = (count1 + count2) / (N1 + N2). */
SPN_API int spn_repeatability_counts(spn_ctx* ctx, const double* d_pts1, const int32_t* d_n1, const double* d_pts2,
                                     const int32_t* d_n2, int B, int cap, double thresh, int32_t* d_out, spn_stream stream);

/* cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(desc1, desc2) (descriptor_evaluation.py:71-78), batched:
 * d_desc1 [B][cap1][C], d_desc2 [B][cap2][C] fp32 with d_n1 / d_n2 [B] valid rows, C a multiple of 64.  The distance
 * matrix is a tcgen05 GEMM on (hi, lo) fp16 splits of the descriptors (fp32-quality dot products), arg-min by 64-bit
 * atomicMin, ties to the lower index.  d_match [B][cap1] = train index of query i or -1, d_dist [B][cap1] = L2 distance. */
SPN_API int spn_mutual_nn_match(spn_ctx* ctx, const float* d_desc1, const int32_t* d_n1, const float* d_desc2,
                                const int32_t* d_n2, int B, int cap1, int cap2, int C, int32_t* d_match, float* d_dist,
                                spn_stream stream);

/* Detector-loss label building (utils/losses.py:13-27): d_kpts_heatmap [B][H][W] int32 (0/1), d_valid_mask [B][H][W] int32
 * (nullable = all valid), d_noise [B][65][H/8][W/8] fp32 (nullable: the U(0, 0.1) tie-break noise is drawn from a
 * counter-based generator keyed by `seed`).  d_labels [B][H/8][W/8] int64 = argmax over the 65 classes of
 * cat([2 * pixel_unshuffle(heatmap), 1]) + noise; d_valid_cells [B][H/8][W/8] fp32 = product of the mask over the cell. */
SPN_API int spn_detector_labels(spn_ctx* ctx, const int32_t* d_kpts_heatmap, const int32_t* d_valid_mask, const float* d_noise,
                                uint64_t seed, int B, int H, int W, int64_t* d_labels, float* d_valid_cells, spn_stream stream);

/* ExportNeRFDetections.step splat (engine_solvers/export.py:271-283): for every pair i in order, the 3x3 patch of
 * d_prob_src [H][W] around the source point d_src_pts[i] (int32 row, col) is copied onto the 3x3 patch of d_out [H][W]
 * around int(d_dst_pts[i]) (fp32 row, col) - a single pixel if either point is within one pixel of the border; later
 * pairs overwrite earlier ones, everything else is 0. */
SPN_API int spn_nerf_splat(spn_ctx* ctx, const float* d_prob_src, const float* d_dst_pts, const int32_t* d_src_pts, int n_pairs, int H,
                           int W, float* d_out, spn_stream stream);

/* Per-kernel CUDA-event timing for bench.py's roofline leg.  Slots 0..11 = the convolution of layer SPN_L_*,
 * then the bandwidth-bound kernels.  spn_profile_read synchronises, writes the accumulated milliseconds and launch
 * counts per slot into HOST arrays of SPN_PROF_SLOTS entries and resets the counters. */
enum {
  SPN_PROF_WARP = 12, SPN_PROF_AGGREGATE = 13, SPN_PROF_NMS = 14, SPN_PROF_SOFTMAX = 15, SPN_PROF_DESC = 16,
  SPN_PROF_PREP = 17, SPN_PROF_SAMPLER = 18, SPN_PROF_SLOTS = 24
};
SPN_API int spn_profile_enable(spn_ctx* ctx, int enable);
SPN_API int spn_profile_read(spn_ctx* ctx, float* h_ms, int64_t* h_count);

/* number of kernels launched through this context since creation (bench.py's gpu_launches) */
SPN_API int64_t spn_launch_count(spn_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* SPN_B200_H */
