"""SuperPoint feature matching across an image collection on the GPU.

    python -m superpoint_nerf_pytorch_b200.matching --config_path configs/superpoint_match.yaml [--random_init True]

The images are the ``data/ImageFolder.py`` listing of ``<DATA_PATH>/<data.name>/``.  Per run, in one process:
  1. one ``model(x, keypoints=True)`` per group of at most ``data.batch_size`` images of the same network input size;
     keypoints, counts and sparse descriptors are copied into one pool on the device ([N][top_k][256]);
  2. with ``pairs: retrieval`` only: the pair list from image retrieval (``retrieval.py``): a k-means vocabulary of the
     pool (or the ``words`` of an earlier run's ``retrieval.npz``), VLAD vectors and each image's nearest images;
  3. ``spn_match_pairs`` calls over the pool (include/spn_match.h), at most ``Context.MATCH_MAX_PAIRS`` pairs each:
     nearest neighbour of every keypoint of a among the keypoints of b, filtered by the ``matching`` block's mutual
     check, ratio test and distance threshold;
  4. the kept matches compacted in (pair, keypoint of a) order on the device and one copy to the host;
  5. with a ``verification`` block only: RANSAC per pair over those matches (``verify.verify_pairs``);
  6. with a ``tracks`` block only: the tracks of the inlier matches of the verified pairs (``tracks.build_tracks``).

``matching`` keys: ``pairs`` (``exhaustive``: every i < j; ``sequential``: 0 < j - i <= ``window``; ``file``: the
``pairs_file``, one ``name_a name_b`` per line, blank lines and lines starting with ``#`` skipped; ``retrieval``: each
image with its ``retrieval.num_neighbors`` nearest images by VLAD), ``mutual`` (bool),
``ratio`` (0 = off, else in (0, 1]: keep iff d1 < ratio d2) and ``max_dist`` (keep iff d1 <= max_dist; ``.inf`` = off).

``retrieval`` keys (a top-level block, read only with ``pairs: retrieval``): ``num_neighbors`` (1..128, default 20),
``vocab_size`` (1..256 words, default 64), ``kmeans_iters`` (>= 1, default 20) and ``vocabulary`` (the path of an
earlier run's ``retrieval.npz``, whose words are reused instead of running k-means; exclusive with the two k-means
keys).

``verification`` keys (an optional top-level block; without it nothing is verified and geometry.npz is not written):
``model`` (required: ``fundamental``, 7-point RANSAC with the Sampson error, or ``homography``, 4-point RANSAC with the
forward transfer error), ``threshold`` (pixels > 0, default 3.0), ``confidence`` (in (0, 1), default 0.999),
``max_iters`` (1..16777216, default 10000), ``min_inliers`` (>= 0, default 15: a pair is verified iff its model has at
least this many inliers) and ``seed`` (integer >= 0, default 0).  With the block, step 5 runs ``verify.verify_pairs``
(include/spn_verify.h) on the matches of step 4; features.npz, matches.npz and retrieval.npz are the same bytes as
without it.

``tracks`` keys (an optional top-level block that needs a ``verification`` block; without it tracks.npz is not
written): ``min_length`` (integer >= 2, default 2: a track has at least this many keypoints).  With the block, step 6
runs ``tracks.build_tracks`` (include/spn_tracks.h) on the inliers of the verified pairs: a track is a connected
component of the graph of those matches over all keypoints.  The other outputs are the same bytes as without it.

Outputs, under ``<EXPER_PATH>/matches/<data.experiment_name>/``; the same inputs give byte-identical files:
  features.npz   names (N,), shapes (N,2) decoded (H, W), resize_geometry (N,4) (new_h, new_w, crop_top, crop_left;
                 with ``data.preprocessing.resize`` only), offsets (N+1,) int64 and keypoints (K,2) int32 (row, col) at
                 the network's input size: image n's keypoints are keypoints[offsets[n]:offsets[n+1]]
  matches.npz    pairs (P,2) int32 image indices, offsets (P+1,) int64, matches (M,2) int32 (keypoint of a, keypoint
                 of b), distances (M,) fp32 and the settings mutual, ratio, max_dist
  retrieval.npz  (``pairs: retrieval`` only) words (K,256) fp32, neighbors (N,k) int32 (-1: none), dist2 (N,k) fp32
                 squared VLAD distances, num_neighbors and kmeans_iters (-1 when the vocabulary was loaded)
  geometry.npz   (with a ``verification`` block only) pairs (P,2) int32, models (P,3,3) fp64 (F: x_b^T F x_a = 0,
                 ||F|| = 1; H: x_b ~ H x_a, H[2][2] = 1; x = (col, row, 1); zeros without a model), num_inliers,
                 hypotheses and best (P,) int32, inliers (M,) bool row-aligned with matches.npz, verified (P,) bool
                 (num_inliers >= min_inliers) and the settings model, threshold, confidence, max_iters, min_inliers,
                 seed
  tracks.npz     (with a ``tracks`` block only) offsets (T+1,) int64: track t's observations are
                 observations[offsets[t]:offsets[t+1]], (image, keypoint) int32 pairs in image order, tracks ordered by
                 their smallest row of features.npz's keypoints; consistent (T,) bool (no two observations in one
                 image; inconsistent tracks are kept and flagged); track_of (K,) int32 row-aligned with features.npz's
                 keypoints (-1: in no track); and the setting min_length
"""
from __future__ import annotations

import json
import math
import os
from pathlib import Path

import numpy as np
import torch

from . import retrieval, settings, tracks, verify
from ._native import Context
from .utils.npz import write_npz

PAIR_MODES = ("exhaustive", "sequential", "file", "retrieval")
MATCH_DEFAULTS = {"pairs": "exhaustive", "window": None, "pairs_file": None, "mutual": True, "ratio": 0.0, "max_dist": math.inf}
RETRIEVAL_DEFAULTS = {"num_neighbors": 20, "vocab_size": 64, "kmeans_iters": 20, "vocabulary": None}
VERIFY_MODELS = ("fundamental", "homography")
VERIFY_DEFAULTS = {"model": None, "threshold": 3.0, "confidence": 0.999, "max_iters": 10000, "min_inliers": 15, "seed": 0}
TRACKS_DEFAULTS = {"min_length": 2}


def match_config(config) -> dict:
    """The ``matching`` block with defaults filled in, after checking the model and data blocks the matcher relies on.
    Unknown or out-of-range keys raise ValueError naming the key."""
    block = config.get("matching") or {}
    if not isinstance(block, dict):
        raise ValueError(f"matching: expected a mapping, got {block!r}")
    for k in block:
        if k not in MATCH_DEFAULTS:
            raise ValueError(f"matching.{k}: unknown key (known: {', '.join(MATCH_DEFAULTS)})")
    m = dict(MATCH_DEFAULTS, **block)
    if m["pairs"] not in PAIR_MODES:
        raise ValueError(f"matching.pairs: must be one of {', '.join(PAIR_MODES)}, got {m['pairs']!r}")
    if m["window"] is not None and (isinstance(m["window"], bool) or not isinstance(m["window"], int) or m["window"] < 1):
        raise ValueError(f"matching.window: must be an integer >= 1, got {m['window']!r}")
    if m["pairs"] == "sequential" and m["window"] is None:
        raise ValueError("matching.window: required with pairs: sequential")
    if m["pairs_file"] is not None and not isinstance(m["pairs_file"], str):
        raise ValueError(f"matching.pairs_file: must be a path, got {m['pairs_file']!r}")
    if m["pairs"] == "file" and not m["pairs_file"]:
        raise ValueError("matching.pairs_file: required with pairs: file")
    if not isinstance(m["mutual"], bool):
        raise ValueError(f"matching.mutual: must be true or false, got {m['mutual']!r}")

    def number(k, ok, what):
        v = m[k]
        if isinstance(v, bool) or not isinstance(v, (int, float)) or math.isnan(v) or not ok(v):
            raise ValueError(f"matching.{k}: must be {what}, got {v!r}")
        return float(v)

    m["ratio"] = number("ratio", lambda v: 0 <= v <= 1, "a number in [0, 1] (0: no ratio test)")
    m["max_dist"] = number("max_dist", lambda v: v >= 0, "a number >= 0 (.inf: no threshold)")
    model = config.get("model") or {}
    if "descriptor_head" not in model or model.get("model_name") == "magicpoint":
        raise ValueError("model: a MagicPoint config has no descriptors to match; use a SuperPoint config")
    dh = model.get("detector_head") or {}
    if not isinstance(dh.get("top_k"), int) or dh["top_k"] <= 0:
        raise ValueError(f"model.detector_head.top_k: must be an integer > 0 (it bounds the keypoints per image), "
                         f"got {dh.get('top_k')!r}")
    if not dh.get("nms"):
        raise ValueError("model.detector_head.nms: must be > 0 (the matcher takes the post-NMS keypoint lists)")
    data = config.get("data") or {}
    bs = data.get("batch_size", 1)
    if isinstance(bs, bool) or not isinstance(bs, int) or bs < 1:
        raise ValueError(f"data.batch_size: must be an integer >= 1, got {bs!r}")
    return m


def retrieval_config(config) -> dict:
    """The top-level ``retrieval`` block with defaults filled in (consulted with ``matching.pairs: retrieval`` only).
    Unknown or out-of-range keys raise ValueError naming the key; the vocabulary file is checked by load_vocabulary."""
    block = config.get("retrieval") or {}
    if not isinstance(block, dict):
        raise ValueError(f"retrieval: expected a mapping, got {block!r}")
    for k in block:
        if k not in RETRIEVAL_DEFAULTS:
            raise ValueError(f"retrieval.{k}: unknown key (known: {', '.join(RETRIEVAL_DEFAULTS)})")
    r = dict(RETRIEVAL_DEFAULTS, **block)
    for k, lo, hi in (("num_neighbors", 1, 128), ("vocab_size", 1, 256), ("kmeans_iters", 1, None)):
        v = r[k]
        if isinstance(v, bool) or not isinstance(v, int) or v < lo or (hi is not None and v > hi):
            what = f"in [{lo}, {hi}]" if hi is not None else f">= {lo}"
            raise ValueError(f"retrieval.{k}: must be an integer {what}, got {v!r}")
    if r["vocabulary"] is not None:
        if not isinstance(r["vocabulary"], str) or not r["vocabulary"]:
            raise ValueError(f"retrieval.vocabulary: must be the path of a retrieval.npz, got {r['vocabulary']!r}")
        both = [k for k in ("vocab_size", "kmeans_iters") if block.get(k) is not None]
        if both:
            raise ValueError(f"retrieval.vocabulary: a loaded vocabulary takes no retrieval.{both[0]} (it would be ignored)")
    return r


def verify_config(config):
    """The top-level ``verification`` block with defaults filled in, or None when the config has none.  Unknown,
    missing or out-of-range keys raise ValueError naming the key."""
    block = config.get("verification")
    if block is None:
        return None
    if not isinstance(block, dict):
        raise ValueError(f"verification: expected a mapping, got {block!r}")
    for k in block:
        if k not in VERIFY_DEFAULTS:
            raise ValueError(f"verification.{k}: unknown key (known: {', '.join(VERIFY_DEFAULTS)})")
    v = dict(VERIFY_DEFAULTS, **block)
    if v["model"] not in VERIFY_MODELS:
        raise ValueError(f"verification.model: required, one of {', '.join(VERIFY_MODELS)}, got {v['model']!r}")

    def number(k, ok, what):
        x = v[k]
        if isinstance(x, bool) or not isinstance(x, (int, float)) or math.isnan(x) or not ok(x):
            raise ValueError(f"verification.{k}: must be {what}, got {x!r}")
        return float(x)

    v["threshold"] = number("threshold", lambda x: 0 < x < math.inf, "a number of pixels > 0")
    v["confidence"] = number("confidence", lambda x: 0 < x < 1, "a number in (0, 1)")
    for k, lo, hi in (("max_iters", 1, 1 << 24), ("min_inliers", 0, None), ("seed", 0, 2 ** 64 - 1)):
        x = v[k]
        if isinstance(x, bool) or not isinstance(x, int) or x < lo or (hi is not None and x > hi):
            what = f"in [{lo}, {hi}]" if hi is not None else f">= {lo}"
            raise ValueError(f"verification.{k}: must be an integer {what}, got {x!r}")
    return v


def tracks_config(config):
    """The top-level ``tracks`` block with defaults filled in, or None when the config has none.  Unknown or
    out-of-range keys, and a block without a ``verification`` block, raise ValueError naming the key."""
    block = config.get("tracks")
    if block is None:
        return None
    if not isinstance(block, dict):
        raise ValueError(f"tracks: expected a mapping, got {block!r}")
    for k in block:
        if k not in TRACKS_DEFAULTS:
            raise ValueError(f"tracks.{k}: unknown key (known: {', '.join(TRACKS_DEFAULTS)})")
    t = dict(TRACKS_DEFAULTS, **block)
    x = t["min_length"]
    if isinstance(x, bool) or not isinstance(x, int) or x < 2:
        raise ValueError(f"tracks.min_length: must be an integer >= 2, got {x!r}")
    if config.get("verification") is None:
        raise ValueError("tracks: needs a verification block (tracks are built from the inliers of verified pairs)")
    return t


def load_vocabulary(path):
    """The ``words`` of a retrieval.npz -> (K, 256) fp32 numpy array; ValueError naming ``retrieval.vocabulary`` and
    the file unless it holds a finite (K, 256) fp32 array with 1 <= K <= 256."""
    where = f"retrieval.vocabulary: {path}"
    try:
        with np.load(path, allow_pickle=False) as z:
            members = {k: z[k] for k in z.files}
    except Exception as e:
        raise ValueError(f"{where}: cannot be read as an .npz file ({e})") from None
    if "words" not in members:
        raise ValueError(f"{where}: no 'words' array (members: {', '.join(members)})")
    words = members["words"]
    if words.dtype != np.float32 or words.ndim != 2 or words.shape[1] != 256 or not 1 <= words.shape[0] <= 256:
        raise ValueError(f"{where}: words must be a (K, 256) float32 array with 1 <= K <= 256, got {words.dtype} "
                         f"{words.shape}")
    if not np.isfinite(words).all():
        raise ValueError(f"{where}: words hold non-finite values")
    return words


def pair_list(names, mode, window=None, pairs_file=None):
    """Image index pairs (a, b) of ``names``: ``exhaustive`` every a < b in order, ``sequential`` 0 < b - a <= window,
    ``file`` the ``name_a name_b`` lines of pairs_file in file order."""
    n = len(names)
    if mode == "exhaustive":
        return [(a, b) for a in range(n) for b in range(a + 1, n)]
    if mode == "sequential":
        if isinstance(window, bool) or not isinstance(window, int) or window < 1:
            raise ValueError(f"sequential pairs need an integer window >= 1, got {window!r}")
        return [(a, b) for a in range(n) for b in range(a + 1, min(n, a + window + 1))]
    if mode == "retrieval":
        raise ValueError("pair mode retrieval needs the descriptors: use retrieval.neighbors and retrieval.retrieval_pairs")
    if mode != "file":
        raise ValueError(f"pair mode must be one of {', '.join(PAIR_MODES)}, got {mode!r}")
    index = {name: i for i, name in enumerate(names)}
    pairs, seen = [], {}
    for ln, line in enumerate(Path(pairs_file).read_text().splitlines(), 1):
        line = line.strip()
        if not line or line.startswith("#"):
            continue
        where = f"{pairs_file}:{ln}"
        fields = line.split()
        if len(fields) != 2:
            raise ValueError(f"{where}: expected 'name_a name_b', got {line!r}")
        for name in fields:
            if name not in index:
                raise ValueError(f"{where}: unknown image name {name!r}")
        a, b = index[fields[0]], index[fields[1]]
        if a == b:
            raise ValueError(f"{where}: pairs an image with itself ({fields[0]!r})")
        key = (min(a, b), max(a, b))
        if key in seen:
            raise ValueError(f"{where}: duplicate of the pair on line {seen[key]}")
        seen[key] = ln
        pairs.append((a, b))
    return pairs


def match_pairs(desc, counts, pairs, mutual=True, ratio=0.0, max_dist=math.inf):
    """Matches of every pair (a, b) of a descriptor pool: desc (N,cap,C) fp32 and counts (N,) int32 CUDA tensors (the
    ``desc_sparse`` / ``keypoint_count`` layout of ``model(x, keypoints=True)``), pairs (P,2) host indices.
    -> (offsets (P+1,) int64, matches (M,2) int32 (keypoint of a, keypoint of b), distances (M,) fp32), CUDA tensors;
    pair p's matches are rows offsets[p]:offsets[p+1], in keypoint order of a.  The rule is include/spn_match.h's;
    pair lists longer than Context.MATCH_MAX_PAIRS are split over several calls with the same result."""
    from ._native import get_context
    ctx = get_context(desc.device)
    pr = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    step = Context.MATCH_MAX_PAIRS
    parts = [ctx.match_pairs(desc, counts, pr[s:s + step], mutual, ratio, max_dist) for s in range(0, len(pr), step)]
    cap = desc.shape[1]
    match = torch.cat([p[0] for p in parts]) if parts else torch.empty((0, cap), dtype=torch.int32, device=desc.device)
    dist = torch.cat([p[1] for p in parts]) if parts else torch.empty((0, cap), dtype=torch.float32, device=desc.device)
    kept = match >= 0
    offsets = torch.zeros(len(pr) + 1, dtype=torch.int64, device=desc.device)
    torch.cumsum(kept.sum(1), 0, out=offsets[1:])
    q, i = torch.nonzero(kept, as_tuple=True)
    matches = torch.stack([i.to(torch.int32), match[q, i]], 1)
    return offsets, matches, dist[q, i]


@torch.no_grad()
def extract_features(model, dataset, batch_size):
    """Keypoints and descriptors of every image of ``dataset`` (data.ImageFolder) -> (items, kp (N,cap,2) int32,
    counts (N,) int32, desc (N,cap,256) fp32), the last three on the model's device.  One forward per group of at most
    ``batch_size`` images of the same input size, groups in order of first appearance."""
    dev = next(model.parameters()).device
    items = [dataset[i] for i in range(len(dataset))]
    shapes = [dataset.resize or it["shape"] for it in items]
    groups = {}
    for i, s in enumerate(shapes):
        groups.setdefault(tuple(s), []).append(i)
    cap = int(model.detector_head.config["top_k"])
    N = len(items)
    kp = torch.zeros((N, cap, 2), dtype=torch.int32, device=dev)
    counts = torch.zeros((N,), dtype=torch.int32, device=dev)
    desc = torch.zeros((N, cap, 256), dtype=torch.float32, device=dev)
    for idx in groups.values():
        for s in range(0, len(idx), batch_size):
            chunk = idx[s:s + batch_size]
            x = torch.stack([dataset.network_input(items[i]) for i in chunk])[:, None]
            out = model(x, keypoints=True)
            sel = torch.tensor(chunk, dtype=torch.int64, device=dev)
            kp[sel] = out["detector_output"]["keypoints"]
            counts[sel] = out["detector_output"]["keypoint_count"]
            desc[sel] = out["descriptor_output"]["desc_sparse"]
    return items, kp, counts, desc


def match_folder(config, model, dataset):
    """Extract and match every image of ``dataset`` (data.ImageFolder) with the ``matching`` block of ``config`` ->
    summary dictionary; writes ``<EXPER_PATH>/matches/<data.experiment_name>/features.npz`` and ``matches.npz`` (and
    ``retrieval.npz`` with ``pairs: retrieval``)."""
    m = match_config(config)
    r = retrieval_config(config) if m["pairs"] == "retrieval" else None
    v = verify_config(config)
    tr = tracks_config(config)
    vocabulary = load_vocabulary(r["vocabulary"]) if r and r["vocabulary"] else None
    model = model.eval()
    items, kp, counts, desc = extract_features(model, dataset, int(config["data"].get("batch_size", 1)))
    names = [it["name"] for it in items]
    if r:
        if vocabulary is not None:
            words = torch.from_numpy(vocabulary).to(desc.device)
        else:
            words = retrieval.kmeans(desc, counts, r["vocab_size"], r["kmeans_iters"])
        index, dist2 = retrieval.neighbors(retrieval.vlad(desc, counts, words), counts, r["num_neighbors"])
        pairs = retrieval.retrieval_pairs(index)
        found = {"words": words.cpu().numpy(), "neighbors": index.cpu().numpy(), "dist2": dist2.cpu().numpy(),
                 "num_neighbors": np.array(r["num_neighbors"]),
                 "kmeans_iters": np.array(-1 if vocabulary is not None else r["kmeans_iters"])}
    else:
        pairs = pair_list(names, m["pairs"], m["window"], m["pairs_file"])
    offsets, matches, distances = match_pairs(desc, counts, pairs, m["mutual"], m["ratio"], m["max_dist"])
    cap, N, P, M = kp.shape[1], len(items), len(pairs), len(matches)
    valid = torch.arange(cap, device=kp.device)[None] < counts[:, None].clamp(0, cap)
    kp_flat = kp[valid]
    # the one device-to-host copy: counts, keypoints, match offsets, matches and distance bits as int32 words
    flat = torch.cat([counts, kp_flat.reshape(-1), offsets.to(torch.int32), matches.reshape(-1), distances.view(torch.int32)]).cpu().numpy()
    parts = np.split(flat, np.cumsum([N, kp_flat.numel(), P + 1, 2 * M])[:])
    cnt = parts[0]
    if cnt.max(initial=0) > cap:
        raise RuntimeError("keypoint list overflow: the model returned more keypoints than model.detector_head.top_k")
    features = {"names": np.array(names, dtype=str), "shapes": np.array([it["shape"] for it in items], np.int32).reshape(N, 2),
                "offsets": np.r_[0, np.cumsum(cnt.astype(np.int64))], "keypoints": parts[1].reshape(-1, 2)}
    if dataset.resize is not None:
        features["resize_geometry"] = np.array([it["geometry"] for it in items], np.int32).reshape(N, 4)
    result = {"pairs": np.array(pairs, np.int32).reshape(P, 2), "offsets": parts[2].astype(np.int64),
              "matches": parts[3].reshape(M, 2), "distances": parts[4].view(np.float32),
              "mutual": np.array(m["mutual"]), "ratio": np.array(m["ratio"]), "max_dist": np.array(m["max_dist"])}
    out_dir = Path(settings.EXPER_PATH, "matches", config["data"]["experiment_name"])
    out_dir.mkdir(parents=True, exist_ok=True)
    write_npz(out_dir / "features.npz", features)
    write_npz(out_dir / "matches.npz", result)
    summary = {"n_images": N, "n_keypoints": int(cnt.sum()), "n_pairs": P, "n_matches": M, "output": str(out_dir),
               **{k: m[k] for k in ("pairs", "mutual", "ratio", "max_dist")}}
    if r:
        write_npz(out_dir / "retrieval.npz", found)
        summary["n_retrieval_pairs"] = P
    if v:
        models, num, hyp, best, inliers = verify.verify_pairs(kp, offsets, matches, pairs, v["model"], v["threshold"],
                                                              v["confidence"], v["max_iters"], v["seed"])
        inliers_d = inliers
        num, inliers = num.cpu().numpy(), inliers.cpu().numpy()
        geometry = {"pairs": result["pairs"], "models": models.cpu().numpy(), "num_inliers": num,
                    "hypotheses": hyp.cpu().numpy(), "best": best.cpu().numpy(), "inliers": inliers,
                    "verified": num >= v["min_inliers"], **{k: np.array(v[k]) for k in VERIFY_DEFAULTS}}
        geometry["seed"] = np.array(v["seed"], np.uint64)
        write_npz(out_dir / "geometry.npz", geometry)
        summary["n_verified_pairs"] = int(geometry["verified"].sum())
        summary["n_inlier_matches"] = int(inliers[np.repeat(geometry["verified"], np.diff(result["offsets"]))].sum())
    if tr:
        verified = torch.from_numpy(geometry["verified"]).to(inliers_d.device)
        keep = inliers_d & torch.repeat_interleave(verified, offsets.diff(), output_size=M)
        t_off, obs, consistent, track_of = (x.cpu().numpy() for x in tracks.build_tracks(
            counts, pairs, offsets, matches, keep, tr["min_length"]))
        write_npz(out_dir / "tracks.npz", {"offsets": t_off, "observations": obs, "consistent": consistent,
                                            "track_of": track_of, "min_length": np.array(tr["min_length"])})
        lengths = np.diff(t_off)
        summary["n_tracks"] = len(consistent)
        summary["n_consistent_tracks"] = int(consistent.sum())
        summary["n_track_observations"] = len(obs)
        summary["mean_track_length"] = float(lengths[consistent].mean()) if consistent.any() else 0.0
    return summary


def main(config_path: str, random_init: bool = False) -> None:
    """Match the SuperPoint features of an image folder.

    Args:
        config_path: Path to configuration.
        random_init: skip loading `pretrained` (random-init weights, torch.manual_seed(0)).
    """
    import yaml
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        raise SystemExit("matching runs as a single process: run it without torchrun (WORLD_SIZE > 1)")
    with open(config_path, "r") as f:
        config = yaml.safe_load(f)
    if match_config(config)["pairs"] == "retrieval":
        retrieval_config(config)
    verify_config(config)
    tracks_config(config)
    if not torch.cuda.is_available():
        raise SystemExit("CUDA is not available: this implementation has no CPU fallback")
    from .data.ImageFolder import ImageFolder
    from .engine import load_pretrained
    from .utils.get_model import get_model
    device = f"cuda:{torch.cuda.current_device()}"
    if random_init:
        torch.manual_seed(0)
    model = get_model(config["model"], device=device)
    if not random_init:
        assert config["pretrained"], "Use a pretrained model to match."
        load_pretrained(model, config, device)
    dataset = ImageFolder(config["data"], device=device)
    print(json.dumps(match_folder(config, model, dataset), indent=2, sort_keys=True))


if __name__ == "__main__":
    import tyro
    tyro.cli(tyro.conf.configure(tyro.conf.FlagConversionOff)(main), use_underscores=True)
