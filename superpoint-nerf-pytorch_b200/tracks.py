"""Multi-view feature tracks on the GPU: the connected components of the graph of kept matches over every keypoint of
a collection, as a track table.  The rule is include/spn_tracks.h's; oracle/tracks_oracle.py restates it."""
from __future__ import annotations

import numpy as np
import torch

from ._native import Context, get_context


def image_offsets(counts):
    """counts (N,) keypoints per image -> (N+1,) int64 offsets on the same device: image n's keypoints are the rows
    offsets[n]:offsets[n+1] of the collection's keypoint table (features.npz's ``offsets``)."""
    off = torch.zeros(counts.shape[0] + 1, dtype=torch.int64, device=counts.device)
    torch.cumsum(counts.to(torch.int64), 0, out=off[1:])
    return off


def match_edges(counts, pairs, offsets, matches, keep=None):
    """The edges of the match graph: kept match (i, j) of pair (a, b) -> (img_off[a] + i, img_off[b] + j).
    counts (N,) int32, offsets (P+1,) int64, matches (M,2) int32 and keep (M,) bool or None are CUDA tensors, pairs
    (P,2) host (a, b).  -> (edges (E,2) int32, img_off (N+1,) int64).  ValueError for inputs that do not fit together,
    including a keypoint index outside [0, count of its image)."""
    dev = counts.device
    if counts.dim() != 1 or counts.shape[0] < 1:
        raise ValueError(f"build_tracks: counts must be (N,) with N >= 1, got shape {tuple(counts.shape)}")
    N = counts.shape[0]
    pr = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    P, M = len(pr), int(matches.shape[0])
    if pr.size and (pr.min() < 0 or pr.max() >= N):
        raise ValueError(f"build_tracks: a pair holds an image index outside [0, {N})")
    if offsets.dim() != 1 or offsets.shape[0] != P + 1:
        raise ValueError(f"build_tracks: {P} pairs need {P + 1} offsets, got shape {tuple(offsets.shape)}")
    if matches.dim() != 2 or matches.shape[1] != 2:
        raise ValueError(f"build_tracks: matches must be (M, 2), got shape {tuple(matches.shape)}")
    if keep is not None and tuple(keep.shape) != (M,):
        raise ValueError(f"build_tracks: keep must be ({M},), got shape {tuple(keep.shape)}")
    offsets = offsets.to(dev, torch.int64)
    counts64 = counts.to(torch.int64)
    steps = offsets.diff()
    bad_counts, bad_offsets = (counts64 < 0).any(), (offsets[0] != 0) | (offsets[-1] != M) | (steps < 0).any()
    if bool(bad_counts | bad_offsets):
        raise ValueError("build_tracks: counts must be >= 0 and offsets must rise from 0 to len(matches)")
    img_off = image_offsets(counts)
    pr_d = torch.from_numpy(pr).to(dev)
    pair_of = torch.repeat_interleave(torch.arange(P, device=dev), steps, output_size=M)
    a, b = pr_d[pair_of, 0], pr_d[pair_of, 1]
    i, j = matches[:, 0].to(torch.int64), matches[:, 1].to(torch.int64)
    outside = (i < 0) | (i >= counts64[a]) | (j < 0) | (j >= counts64[b])
    if bool(outside.any()):
        m = int(torch.nonzero(outside)[0, 0])
        p = int(pair_of[m])
        raise ValueError(f"build_tracks: match {m} ({int(i[m])}, {int(j[m])}) of pair {p} = ({pr[p, 0]}, {pr[p, 1]}) has a "
                         f"keypoint index outside [0, count) (counts {int(counts64[pr[p, 0]])}, {int(counts64[pr[p, 1]])})")
    edges = torch.stack([img_off[a] + i, img_off[b] + j], 1)
    if keep is not None:
        edges = edges[keep.to(dev, torch.bool)]
    return edges.to(torch.int32), img_off


def build_tracks(counts, pairs, offsets, matches, keep=None, min_length=2):
    """Tracks of a collection's matches: counts (N,) int32 (``matching.extract_features``), offsets (P+1,) int64 and
    matches (M,2) int32 (``matching.match_pairs``), keep (M,) bool (e.g. the inliers of verified pairs; None keeps
    every match), all CUDA, and pairs (P,2) host (a, b).  -> (track_offsets (T+1,) int64, observations (O,2) int32
    (image, keypoint), consistent (T,) bool, track_of (K,) int32, -1 for keypoints in no track), CUDA tensors.
    Tracks are the components of at least min_length keypoints, ordered by their smallest row of the keypoint table;
    a track's observations are in row order, which is image order; a track is consistent iff it has at most one
    keypoint per image."""
    if isinstance(min_length, bool) or not isinstance(min_length, (int, np.integer)) or min_length < 2:
        raise ValueError(f"build_tracks: min_length must be an integer >= 2, got {min_length!r}")
    edges, img_off = match_edges(counts, pairs, offsets, matches, keep)
    dev = counts.device
    K = int(img_off[-1])
    if K > Context.TRACKS_MAX_ROWS:
        raise ValueError(f"build_tracks: {K} keypoints exceed {Context.TRACKS_MAX_ROWS} rows")
    if K == 0:                               # no keypoints: no nodes, so no tracks
        return (torch.zeros(1, dtype=torch.int64, device=dev), torch.zeros((0, 2), dtype=torch.int32, device=dev),
                torch.zeros(0, dtype=torch.bool, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    ctx = get_context(dev)
    labels, bad_edges = ctx.track_labels(edges, K)
    track_off, obs, consistent, track_of, totals, bad_labels = ctx.track_table(labels, img_off, int(min_length))
    n_bad_edges, n_bad_labels, T, O = torch.cat([bad_edges, bad_labels, totals]).tolist()
    if n_bad_edges or n_bad_labels:
        raise RuntimeError(f"build_tracks: {n_bad_edges} edges outside [0, {K}) and {n_bad_labels} bad labels or offsets "
                           "reached the track kernels")
    return track_off[:T + 1], obs[:O], consistent[:T].bool(), track_of
