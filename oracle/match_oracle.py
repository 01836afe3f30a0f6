"""fp64 numpy restatement of spn_match_pairs (include/spn_match.h): brute-force L2 distances between every row of a and
every row of b, the nearest and second-nearest row with ties to the lower index, and the mutual, ratio and distance
filters.

Besides the decisions it returns each query's decision margin: how far the fp64 values are from flipping a decision,
in SQUARED distance, where the GPU's error is bounded (~1e-6 for unit-norm descriptors: fp32 accumulation of the
tensor-core hi/lo products); the square root amplifies that error near 0 (d^2 = 1e-6 gives d = 1e-3).  Exact duplicates
of b's best row are not a margin (identical rows give identical distances on the GPU too, and the lower index wins on
both sides)."""
import math

import numpy as np


def distances(a, b):
    """(n_a, n_b) fp64 L2 distances."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    d2 = (a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * (a @ b.T)
    return np.sqrt(np.maximum(d2, 0.0))


def top2(a, b):
    """-> best_j, d1, d2 (second-nearest distance over j != best_j, inf with one row) and gap: d^2 to the nearest row
    of b that is not an exact copy of b[best_j], minus d1^2 (inf when there is none)."""
    d = distances(a, b)
    n_a, n_b = d.shape
    if n_a == 0 or n_b == 0:
        z = np.zeros(n_a)
        return np.zeros(n_a, np.int64), z + np.inf, z + np.inf, z + np.inf
    best = d.argmin(1)                                   # the first minimum: ties go to the lower index
    rows = np.arange(n_a)
    d1 = d[rows, best]
    others = d.copy()
    others[rows, best] = np.inf
    d2 = others.min(1)
    ids = np.unique(np.asarray(b), axis=0, return_inverse=True)[1].reshape(-1)
    copy = ids[None, :] == ids[best][:, None]             # (n_a, n_b): b_j identical to b[best_i]
    gap = np.where(copy, np.inf, d).min(1) ** 2 - d1 ** 2
    return best, d1, d2, gap


def match(a, b, mutual=True, ratio=0.0, max_dist=math.inf):
    """One pair -> dict with match (n_a,) int (index into b or -1), dist (n_a,) (d1 where kept, else 0), keep, best,
    d1, d2 and margin (n_a,): the smallest of the best/second gap (and the reverse gap of b's row with mutual),
    |d1^2 - ratio^2 d2^2| with a ratio and |d1^2 - max_dist^2| with a finite threshold, all in squared distance."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    n_a, n_b = len(a), len(b)
    best, d1, d2, gap = top2(a, b)
    keep = np.full(n_a, n_b > 0)
    margin = gap.copy()
    if mutual and n_a and n_b:
        back, _, _, gap_b = top2(b, a)
        keep &= back[best] == np.arange(n_a)
        margin = np.minimum(margin, gap_b[best])
    if ratio > 0 and n_b:
        keep &= d1 < ratio * d2
        margin = np.minimum(margin, np.abs(d1 ** 2 - ratio ** 2 * d2 ** 2))
    if n_b:
        keep &= d1 <= max_dist
        if math.isfinite(max_dist):
            margin = np.minimum(margin, np.abs(d1 ** 2 - max_dist ** 2))
    return {"match": np.where(keep, best, -1), "dist": np.where(keep, d1, 0.0), "keep": keep, "best": best, "d1": d1,
            "d2": d2, "margin": margin}


def match_pairs(desc, counts, pairs, mutual=True, ratio=0.0, max_dist=math.inf):
    """The pool form: desc (N,cap,C), counts (N,), pairs (P,2) -> match (P,cap) int64 (-1 past a's count), dist (P,cap)
    and margin (P,cap) (inf past a's count)."""
    desc = np.asarray(desc)
    N, cap, _ = desc.shape
    counts = np.clip(np.asarray(counts, np.int64), 0, cap)
    P = len(pairs)
    out = {"match": np.full((P, cap), -1, np.int64), "dist": np.zeros((P, cap)), "margin": np.full((P, cap), np.inf)}
    for q, (ia, ib) in enumerate(pairs):
        n_a = counts[ia]
        r = match(desc[ia, :n_a], desc[ib, :counts[ib]], mutual, ratio, max_dist)
        for k in out:
            out[k][q, :n_a] = r[k]
    return out
