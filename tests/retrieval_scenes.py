"""Descriptor sets for the retrieval and matching tests: random unit rows and planted multi-view scenes.  numpy
RandomState only."""
import math

import numpy as np


def unit(shape, rng):
    x = rng.randn(*shape).astype(np.float32)
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def planted_scenes(seed, S=8, V=4, L=400, keep=300, distractors=50, C=256, sigma=0.1):
    """S scenes of L random unit landmarks; each of V views holds `keep` of its scene's landmarks with noise and
    `distractors` random unit rows.  sigma is the noise's scale relative to the unit-norm descriptor (per-component
    standard deviation sigma / sqrt(C), so the noise vector has norm ~sigma) before re-normalisation."""
    rng = np.random.RandomState(seed)
    desc = np.zeros((S * V, keep + distractors, C), np.float32)
    for s in range(S):
        landmarks = unit((L, C), rng)
        for v in range(V):
            x = landmarks[rng.choice(L, keep, replace=False)] + sigma / math.sqrt(C) * rng.randn(keep, C).astype(np.float32)
            rows = np.concatenate([x / np.linalg.norm(x, axis=1, keepdims=True), unit((distractors, C), rng)])
            desc[s * V + v] = rows[rng.permutation(len(rows))]
    return desc
