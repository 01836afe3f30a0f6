"""numpy restatement of include/spn_retrieval.h and retrieval.py: the k nearest rows in fp64 with ties to the lower
index, the residual sums as the fp32 sequential loop of the header (bit-equal), VLAD normalisation and one k-means
step in fp64, and the pair list of neighbour lists.

``knn`` also returns each query's decision margin in squared distance, as oracle/match_oracle.py does for the matcher:
the smallest d^2 gap between adjacent ranks among the first k + 1 (so both the order of the k kept rows and the choice
of the k-th against the (k+1)-th count).  Adjacent ranks that hold exact copies of one train row are not a margin:
identical rows give identical bits on the GPU too, and the lower index wins on both sides."""
import numpy as np


def knn(q, t, k, exclude_self=False):
    """-> index (nq,k) int64 (-1 past the usable rows), d2 (nq,k) fp64 (+inf there), margin (nq,) fp64."""
    q, t = np.asarray(q, np.float64), np.asarray(t, np.float64)
    nq, nt = len(q), len(t)
    index = np.full((nq, k), -1, np.int64)
    d2 = np.full((nq, k), np.inf)
    margin = np.full(nq, np.inf)
    if nq == 0 or nt == 0:
        return index, d2, margin
    d = (q * q).sum(1)[:, None] + (t * t).sum(1)[None, :] - 2.0 * (q @ t.T)
    d = np.maximum(d, 0.0)
    if exclude_self:
        d[np.arange(nq), np.arange(nq)] = np.inf
    order = np.argsort(d, axis=1, kind="stable")                     # equal distances: ascending index
    usable = nt - 1 if exclude_self else nt
    m = min(k, usable)
    rows = np.arange(nq)[:, None]
    index[:, :m] = order[:, :m]
    d2[:, :m] = d[rows, order[:, :m]]
    ids = np.unique(t, axis=0, return_inverse=True)[1].reshape(-1)
    top = order[:, :min(k + 1, usable)]
    if top.shape[1] > 1:
        ds = d[rows, top]
        gaps = np.where(ids[top[:, 1:]] == ids[top[:, :-1]], np.inf, ds[:, 1:] - ds[:, :-1])
        margin = gaps.min(1)
    return index, d2, margin


def residual_sums(desc, counts, assign, words):
    """sums (N,K,C) fp32 and n (N,K) int64: the header's loop, every subtraction and addition rounded to fp32."""
    desc, words = np.asarray(desc, np.float32), np.asarray(words, np.float32)
    N, cap, C = desc.shape
    K = len(words)
    counts = np.clip(np.asarray(counts, np.int64), 0, cap)
    assign = np.asarray(assign, np.int64)
    sums = np.zeros((N, K, C), np.float32)
    n = np.zeros((N, K), np.int64)
    for img in range(N):
        for i in range(counts[img]):
            w = assign[img, i]
            if 0 <= w < K:
                sums[img, w] += desc[img, i] - words[w]              # two fp32 array operations, each rounded
                n[img, w] += 1
    return sums, n


def vlad(sums):
    """(N,K,C) residual sums -> (N,K*C) fp64 intra-normalised VLAD (empty blocks and empty images stay 0)."""
    s = np.asarray(sums, np.float64)
    norm = np.linalg.norm(s, axis=2, keepdims=True)
    v = np.divide(s, norm, out=np.zeros_like(s), where=norm > 0).reshape(len(s), -1)
    norm = np.linalg.norm(v, axis=1, keepdims=True)
    return np.divide(v, norm, out=np.zeros_like(v), where=norm > 0)


def kmeans_step(desc, counts, assign, words):
    """One Lloyd update in fp64 from given assignments: each word with members moves to the mean of its members."""
    desc, words = np.asarray(desc, np.float64), np.asarray(words, np.float64)
    cap = desc.shape[1]
    valid = np.arange(cap)[None] < np.clip(np.asarray(counts), 0, cap)[:, None]
    x, a = desc[valid], np.asarray(assign)[valid]
    out = words.copy()
    for w in range(len(words)):
        if (a == w).any():
            out[w] = x[a == w].mean(0)
    return out


def objective(desc, counts, assign, words):
    """Sum over the valid rows of d^2 to the assigned word, fp64."""
    desc, words = np.asarray(desc, np.float64), np.asarray(words, np.float64)
    cap = desc.shape[1]
    valid = np.arange(cap)[None] < np.clip(np.asarray(counts), 0, cap)[:, None]
    x, a = desc[valid], np.asarray(assign)[valid]
    return float(((x - words[a]) ** 2).sum())


def retrieval_pairs(index):
    """Neighbour lists (N,k), -1 = none -> sorted list of distinct (min(a, b), max(a, b)) with a != b."""
    pairs = set()
    for a, row in enumerate(np.asarray(index)):
        for b in row:
            if b >= 0 and b != a:
                pairs.add((min(a, int(b)), max(a, int(b))))
    return sorted(pairs)
