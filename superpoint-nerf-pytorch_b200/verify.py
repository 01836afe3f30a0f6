"""Geometric verification of descriptor matches on the GPU: one fundamental matrix or homography per image pair by
RANSAC, and the matches that agree with it.  The rule is include/spn_verify.h's; oracle/verify_oracle.py restates it."""
from __future__ import annotations

import numpy as np
import torch

from ._native import Context, get_context


def verify_pairs(kp, offsets, matches, pairs, model="fundamental", threshold=3.0, confidence=0.999, max_iters=10000, seed=0):
    """RANSAC over the matches of every pair: kp (N,cap,2) int32 (row, col) CUDA keypoint pool
    (``matching.extract_features``), offsets (P+1,) int64 and matches (M,2) int32 CUDA tensors (``matching.match_pairs``),
    pairs (P,2) host (a, b) image indices.  -> (models (P,3,3) fp64, num_inliers (P,) int32, hypotheses (P,) int32,
    best (P,) int32, inliers (M,) bool), CUDA tensors.  A pair's result depends only on its own matches, (a, b) and the
    settings, so pair lists longer than Context.VERIFY_MAX_PAIRS are split over several calls with the same result."""
    ctx = get_context(kp.device)
    pr = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    P = len(pr)
    offsets = offsets.contiguous()
    if offsets.dim() != 1 or offsets.shape[0] != P + 1:
        raise ValueError(f"verify_pairs: {P} pairs need {P + 1} offsets, got shape {tuple(offsets.shape)}")
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or not 0 <= seed < 2 ** 64:
        raise ValueError(f"verify_pairs: seed must be an integer in [0, 2^64), got {seed!r}")
    step = Context.VERIFY_MAX_PAIRS
    parts = [ctx.verify_pairs(kp, offsets[s:s + step + 1], matches, pr[s:s + step], model, threshold, confidence, max_iters,
                              int(seed)) for s in range(0, P, step)]
    if not parts:
        parts = [ctx.verify_pairs(kp, offsets, matches, pr, model, threshold, confidence, max_iters, int(seed))]
    models, num, hyp, best = (torch.cat([p[k] for p in parts]) for k in range(4))
    inliers = parts[0][4]
    for p in parts[1:]:                      # each call writes only the rows of its own pairs; the others stay 0
        inliers = torch.maximum(inliers, p[4])
    return models, num, hyp, best, inliers.bool()
