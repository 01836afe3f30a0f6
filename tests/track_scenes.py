"""Planted multi-view scenes for the track tests and tools/bench_tracks.py: landmarks seen in several views, each
view's keypoints its visible landmarks plus distractors, matches every true pair plus chance outliers.  numpy
RandomState only."""
import numpy as np


def planted(rng, n_images=16, n_land=400, visible=0.35, distractors=60, outliers=0, clashes=0):
    """Landmarks seen in several views.  Each image's keypoints are its visible landmarks and some distractors, shuffled;
    matches are every true pair plus ``outliers`` chance matches between distractors per pair.  ``clashes`` extra
    outliers each join two distractors of one image through a distractor of another.  -> (counts, pairs, offsets,
    matches, landmark of every row (-1: distractor))."""
    seen = rng.rand(n_images, n_land) < visible
    land_of, index = [], []
    for n in range(n_images):
        ids = np.r_[np.nonzero(seen[n])[0], -np.ones(distractors, np.int64)]
        ids = ids[rng.permutation(len(ids))]
        land_of.append(ids)
        index.append({int(lm): i for i, lm in enumerate(ids) if lm >= 0})
    pairs, rows = [], []
    for a in range(n_images):
        for b in range(a + 1, n_images):
            common = np.nonzero(seen[a] & seen[b])[0]
            m = [(index[a][lm], index[b][lm]) for lm in common]
            da, db = np.nonzero(land_of[a] < 0)[0], np.nonzero(land_of[b] < 0)[0]
            m += list(zip(rng.choice(da, outliers), rng.choice(db, outliers)))
            pairs.append((a, b))
            rows.append(np.array(m, np.int64).reshape(-1, 2)[rng.permutation(len(m))])
    for _ in range(clashes):
        p = rng.randint(len(pairs))
        a, b = pairs[p]
        d1, d2 = rng.choice(np.nonzero(land_of[a] < 0)[0], 2, replace=False)
        d3 = rng.choice(np.nonzero(land_of[b] < 0)[0])
        rows[p] = np.r_[rows[p], [[d1, d3], [d2, d3]]]
    counts = np.array([len(x) for x in land_of], np.int32)
    offsets = np.r_[0, np.cumsum([len(x) for x in rows])].astype(np.int64)
    return counts, np.array(pairs, np.int32), offsets, np.concatenate(rows).astype(np.int32), np.concatenate(land_of)
