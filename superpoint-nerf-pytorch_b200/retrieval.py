"""Image retrieval over a SuperPoint descriptor pool on the GPU: a k-means vocabulary, VLAD vectors and the k nearest
images of every image, for selecting the pairs to match in a collection with no order.

Every function takes the pool as ``model(x, keypoints=True)`` returns it (``matching.extract_features``): desc
(N,cap,C) fp32 and counts (N,) int32 CUDA tensors, row i of image n valid for i < counts[n].  The rule:
  - words: ``kmeans`` draws K distinct valid descriptors, ``np.random.RandomState(0).choice(n_valid, K,
    replace=False)`` over the valid rows in (image, keypoint) order, then runs exactly ``iters`` Lloyd steps: every
    valid row goes to its nearest word (``spn_knn`` with k = 1, ties to the lower word), and every word with members
    moves to c_w + sum_n sums[n][w] / sum_n n[n][w] (``spn_residual_sums``, summed over images in torch); a word with
    no members keeps its centroid;
  - VLAD of an image: the residual sums of its rows against their nearest words, each word block normalised to unit L2
    norm (blocks with no members stay 0), then the whole (K*C,) vector normalised to unit L2 norm (intra-normalisation,
    Arandjelovic & Zisserman, "All about VLAD").  An image without keypoints gets the zero vector;
  - neighbours: the k nearest VLAD vectors of every image among the other images that have keypoints (``spn_knn`` with
    exclude_self, squared L2 distance, ascending, ties to the lower index), -1 / +inf past the last one and on every
    row of an image without keypoints;
  - pairs: every (min(a, b), max(a, b)) of an image and one of its neighbours, de-duplicated and sorted.  With k >= N - 1
    and keypoints in every image this is ``matching.pair_list(names, "exhaustive")``.
"""
from __future__ import annotations

import numpy as np
import torch

from ._native import get_context


def _valid(desc, counts):
    cap = desc.shape[1]
    return torch.arange(cap, device=desc.device)[None] < counts.clamp(0, cap)[:, None]


def assign_words(desc, counts, words):
    """Nearest word of every row of the pool -> (N, cap) int32, -1 at rows at or beyond counts[n]."""
    N, cap, C = desc.shape
    index, _ = get_context(desc.device).knn(desc.reshape(N * cap, C), words, 1)
    return torch.where(_valid(desc, counts), index.view(N, cap), -1)


def kmeans(desc, counts, K, iters):
    """A K-word vocabulary of the pool's valid descriptors -> (K, C) fp32 CUDA tensor (the rule of the module)."""
    flat = desc[_valid(desc, counts)]
    if len(flat) < K:
        raise ValueError(f"retrieval.vocab_size: {K} words need at least as many keypoints, the collection has {len(flat)}")
    pick = np.random.RandomState(0).choice(len(flat), K, replace=False)
    words = flat[torch.from_numpy(pick).to(desc.device)].contiguous()
    for _ in range(iters):
        words = lloyd_step(desc, counts, words)
    return words


def lloyd_step(desc, counts, words):
    """One k-means step: assign every valid row to its nearest word, move every word with members to c_w +
    sum_n sums[n][w] / sum_n n[n][w]; a word with no members keeps its centroid."""
    sums, n = get_context(desc.device).residual_sums(desc, counts, assign_words(desc, counts, words), words)
    total = n.sum(0)
    step = sums.sum(0) / total.clamp(min=1)[:, None].to(torch.float32)
    return torch.where(total[:, None] > 0, words + step, words).contiguous()


def vlad(desc, counts, words):
    """Intra-normalised VLAD vector of every image -> (N, K*C) fp32 CUDA tensor."""
    sums, _ = get_context(desc.device).residual_sums(desc, counts, assign_words(desc, counts, words), words)
    norm = sums.norm(dim=2, keepdim=True)
    v = torch.where(norm > 0, sums / norm.clamp(min=1e-30), 0.0).reshape(len(desc), -1)
    norm = v.norm(dim=1, keepdim=True)
    return torch.where(norm > 0, v / norm.clamp(min=1e-30), 0.0)


def neighbors(vectors, counts, k):
    """The k nearest images of every image by VLAD -> (index (N,k) int32, dist2 (N,k) fp32) CUDA tensors; -1 / +inf
    past the last neighbour and on the rows of images without keypoints."""
    N = len(vectors)
    has = torch.nonzero(counts > 0).view(-1)
    index = torch.full((N, k), -1, dtype=torch.int32, device=vectors.device)
    dist2 = torch.full((N, k), float("inf"), dtype=torch.float32, device=vectors.device)
    if len(has):
        idx, d2 = get_context(vectors.device).knn(vectors[has], vectors[has], k, exclude_self=True)
        index[has] = torch.where(idx >= 0, has.to(torch.int32)[idx.clamp(min=0).long()], -1)
        dist2[has] = d2
    return index, dist2


def retrieval_pairs(index):
    """Neighbour lists (N, k) (host or CUDA, -1 = none) -> sorted, de-duplicated list of (min(a, b), max(a, b))."""
    idx = index.cpu().numpy() if torch.is_tensor(index) else np.asarray(index)
    a = np.repeat(np.arange(len(idx)), idx.shape[1] if idx.ndim == 2 else 0)
    b = idx.reshape(-1)
    keep = (b >= 0) & (b != a)
    pairs = np.unique(np.stack([np.minimum(a, b)[keep], np.maximum(a, b)[keep]], 1).astype(np.int64).reshape(-1, 2), axis=0)
    return [(int(x), int(y)) for x, y in pairs]
