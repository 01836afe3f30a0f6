"""Host oracle for include/spn_tracks.h / tracks.py: the track rule restated with numpy and scipy.

Nodes are the rows of a collection's keypoint table (image n's keypoint i is row img_offsets[n] + i); a kept match
(i, j) of the pair (a, b) is the edge (img_offsets[a] + i, img_offsets[b] + j).  A row's label is the smallest row of
its connected component.  Tracks are the components of at least min_length rows, ordered by label; a track's
observations are its rows in ascending order as (image, keypoint); a track is consistent iff no two of its
observations lie in one image.  Test infrastructure only.
"""
from __future__ import annotations

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components


def labels(edges, K):
    """edges (E,2) rows in [0, K) -> (K,) int32: the smallest row of every row's component."""
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    graph = coo_matrix((np.ones(len(edges), np.int8), (edges[:, 0], edges[:, 1])), shape=(K, K)).tocsr()
    _, comp = connected_components(graph, directed=False)
    _, first = np.unique(comp, return_index=True)        # rows ascend, so a component's first row is its smallest
    smallest = np.empty(len(first), np.int64)
    smallest[comp[first]] = first
    return smallest[comp].astype(np.int32)


def tracks(label, img_offsets, min_length=2):
    """label (K,) from labels(), img_offsets (N+1,) -> (track_offsets (T+1,) int64, observations (O,2) int32 (image,
    keypoint), consistent (T,) bool, track_of (K,) int32, -1 for rows in no track)."""
    label = np.asarray(label, dtype=np.int64)
    img_offsets = np.asarray(img_offsets, dtype=np.int64)
    K = len(label)
    size = np.bincount(label, minlength=K)
    rows = np.nonzero(size[label] >= min_length)[0]
    rows = rows[np.argsort(label[rows], kind="stable")]   # by track, rows ascending inside a track
    keys = label[rows]
    roots, starts = np.unique(keys, return_index=True)
    T = len(roots)
    track_offsets = np.r_[starts, len(rows)].astype(np.int64)
    image = np.searchsorted(img_offsets, rows, side="right") - 1
    observations = np.stack([image, rows - img_offsets[image]], 1).astype(np.int32).reshape(-1, 2)
    index = np.full(K, -1, np.int64)
    index[roots] = np.arange(T)
    track_of = index[label].astype(np.int32)
    consistent = np.ones(T, bool)
    clash = (keys[1:] == keys[:-1]) & (image[1:] == image[:-1])
    consistent[index[keys[1:][clash]]] = False
    return track_offsets, observations, consistent, track_of


def match_edges(counts, pairs, offsets, matches, keep=None):
    """The edges of kept matches: counts (N,), pairs (P,2), offsets (P+1,), matches (M,2), keep (M,) bool or None ->
    (edges (E,2) int64, img_offsets (N+1,) int64)."""
    counts = np.asarray(counts, dtype=np.int64)
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    matches = np.asarray(matches, dtype=np.int64).reshape(-1, 2)
    img_offsets = np.r_[0, np.cumsum(counts)].astype(np.int64)
    pair_of = np.repeat(np.arange(len(pairs)), np.diff(np.asarray(offsets, dtype=np.int64)))
    a, b = pairs[pair_of, 0], pairs[pair_of, 1]
    assert ((matches[:, 0] >= 0) & (matches[:, 0] < counts[a]) & (matches[:, 1] >= 0) & (matches[:, 1] < counts[b])).all()
    edges = np.stack([img_offsets[a] + matches[:, 0], img_offsets[b] + matches[:, 1]], 1).reshape(-1, 2)
    if keep is not None:
        edges = edges[np.asarray(keep, bool)]
    return edges, img_offsets


def build_tracks(counts, pairs, offsets, matches, keep=None, min_length=2):
    """tracks.build_tracks restated -> (track_offsets, observations, consistent, track_of, label)."""
    edges, img_offsets = match_edges(counts, pairs, offsets, matches, keep)
    label = labels(edges, int(img_offsets[-1]))
    return (*tracks(label, img_offsets, min_length), label)
