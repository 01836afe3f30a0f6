#!/usr/bin/env python
"""Feature tracks (include/spn_tracks.h, tracks.py): kernel times against the host oracle, and one end-to-end row after
retrieval matching and verification.

Kernels (CUDA events around --reps calls after one warm-up call of the same shape; the GPU's name, power limit and
clocks are read in the same run): spn_track_labels and spn_track_table, each through its Context method, on
  - random graphs: K rows in 1000-keypoint images, E edges with uniform endpoints (duplicates and self-loops included);
  - planted multi-view scenes (tests/track_scenes.py): landmarks seen by ~30 % of the views plus distractors, every
    true match plus chance outliers between distractors over the exhaustive pairs;
  - the adversarial chain: K = 10^6, edges (r, r + 1) fed in descending r, the deepest union-find forest.
Union-find is bound by the latency of dependent loads and of atomicCAS, not by bandwidth, so the bytes are reported
as a count (edges read once, two label reads per edge, the labels written twice; the table's inputs and outputs), not
as a share of peak.  The labels of K = 10^7 rows (40 MB) fit in the 126 MB L2; nothing is flushed between calls.
Host baseline: oracle/tracks_oracle.py (scipy connected_components, a stable argsort by label) on the same graphs on
this machine's host, one run each.
End to end (synthetic collection of tools/bench_retrieval.py, random-init seeded weights; not a statement about trained
models): 1000 images, one extraction, retrieval pairs, matching with the mutual check and ratio 0.8, verify.verify_pairs
with a fundamental matrix, then tracks.build_tracks on the inliers of the verified pairs; wall times of the three steps
(host clock around device-synchronised steps), and the tracks found.

    python tools/bench_tracks.py [--reps 5] [--images 1000] [--out profiles/r9_tracks.json]
"""
import argparse
import copy
import json
import math
import os
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))

from bench_nerf_export import gpu_info  # noqa: E402
from oracle import tracks_oracle as T  # noqa: E402
from track_scenes import planted  # noqa: E402

RANDOM = ((10 ** 6, 2 * 10 ** 5), (10 ** 6, 2 * 10 ** 6), (10 ** 6, 15 * 10 ** 6), (10 ** 7, 2 * 10 ** 6), (10 ** 7, 15 * 10 ** 6))


def graphs():
    rng = np.random.RandomState(0)
    for K, E in RANDOM:
        yield {"graph": "random", "K": K, "E": E}, rng.randint(0, K, (E, 2)), np.r_[np.arange(0, K, 1000), K]
    for n_images, n_land in ((48, 30000), (200, 4000)):
        counts, pairs, offsets, matches, _ = planted(rng, n_images=n_images, n_land=n_land, visible=0.3, distractors=500,
                                                     outliers=20)
        edges, img_off = T.match_edges(counts, pairs, offsets, matches)
        yield ({"graph": "planted", "images": n_images, "landmarks": n_land, "pairs": len(pairs), "K": int(img_off[-1]),
                "E": len(edges)}, edges, img_off)
    K = 10 ** 6
    r = np.arange(K - 2, -1, -1)
    yield {"graph": "descending chain", "K": K, "E": K - 1}, np.c_[r, r + 1], np.arange(K + 1)


def timed_events(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def kernels(ctx, reps, rec):
    for info, edges, img_off in graphs():
        K, E = info["K"], info["E"]
        d_edges = torch.from_numpy(edges.astype(np.int32)).cuda()
        d_off = torch.from_numpy(img_off.astype(np.int64)).cuda()
        ms_l, (labels, bad) = timed_events(lambda: ctx.track_labels(d_edges, K), reps)
        ms_t, out = timed_events(lambda: ctx.track_table(labels, d_off, 2), reps)
        n_t, n_o = out[4].tolist()
        assert bad.item() == 0 and out[5].item() == 0
        t = time.perf_counter()
        lab = T.labels(edges, K)
        t_lab = time.perf_counter() - t
        want = T.tracks(lab, img_off, 2)
        t_host = time.perf_counter() - t
        same = (np.array_equal(labels.cpu().numpy(), lab) and np.array_equal(out[0][:n_t + 1].cpu().numpy(), want[0])
                and np.array_equal(out[1][:n_o].cpu().numpy(), want[1]))
        N = len(img_off) - 1
        bytes_labels = 8 * E + 8 * E + 8 * K
        bytes_table = 4 * K + 8 * (N + 1) + 8 * (n_t + 1) + 8 * n_o + n_t + 4 * K
        run = dict(info, what="spn_track_labels + spn_track_table", reps=reps, labels_ms=ms_l, table_ms=ms_t,
                   edges_per_s=E / (ms_l * 1e-3), labels_bytes_counted=bytes_labels, table_bytes_counted=bytes_table,
                   labels_GBps_counted=bytes_labels / (ms_l * 1e-3) / 1e9, tracks=n_t, observations=n_o,
                   consistent_tracks=int(out[2][:n_t].sum().item()), equals_oracle=bool(same),
                   host_oracle={"labels_s": t_lab, "labels_and_table_s": t_host, "threads": "scipy / numpy, one process",
                                "cpus": os.cpu_count()},
                   host_over_gpu=t_host / ((ms_l + ms_t) * 1e-3))
        rec["runs"].append(run)
        print(json.dumps(run), flush=True)
        del d_edges, d_off, labels, out


def end_to_end(n_images, rec):
    import cv2
    import yaml
    from bench_retrieval import scene_images
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import retrieval, settings, tracks, verify
    from superpoint_nerf_pytorch_b200.data.ImageFolder import ImageFolder
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    cfg = yaml.safe_load(open(ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match_retrieval.yaml"))
    views = 10
    with tempfile.TemporaryDirectory() as tmp:
        root = Path(tmp) / "scenes"
        root.mkdir()
        for i, img in enumerate(scene_images(n_images, views)):
            cv2.imwrite(str(root / f"{i:05d}.png"), img)
        settings.DATA_PATH = tmp
        cfg["data"].update(name="scenes", preprocessing=None)
        torch.manual_seed(0)
        model = get_model(copy.deepcopy(cfg["model"]), device="cuda:0").eval()
        ds = ImageFolder(cfg["data"], device="cuda:0")
        items, kp, counts, desc = M.extract_features(model, ds, int(cfg["data"]["batch_size"]))
    r = M.retrieval_config(cfg)

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t

    words = retrieval.kmeans(desc, counts, r["vocab_size"], r["kmeans_iters"])
    index, _ = retrieval.neighbors(retrieval.vlad(desc, counts, words), counts, r["num_neighbors"])
    pairs = retrieval.retrieval_pairs(index)
    (offsets, matches, _), t_match = timed(lambda: M.match_pairs(desc, counts, pairs, True, 0.8, math.inf))
    verify.verify_pairs(kp, offsets[:65], matches, pairs[:64], "fundamental")               # warm-up
    (_, num, _, _, inl), t_ver = timed(lambda: verify.verify_pairs(kp, offsets, matches, pairs, "fundamental"))
    keep = inl & torch.repeat_interleave(num >= 15, offsets.diff(), output_size=len(matches))
    tracks.build_tracks(counts, pairs[:64], offsets[:65], matches[:int(offsets[64])], keep[:int(offsets[64])])  # warm-up
    (t_off, obs, cons, _), t_trk = timed(lambda: tracks.build_tracks(counts, pairs, offsets, matches, keep))
    lengths = t_off.diff().cpu().numpy()
    cons = cons.cpu().numpy()
    run = {"what": "end_to_end", "images": len(items), "size": [480, 640], "weights": "random-init, torch.manual_seed(0)",
           "keypoints": int(counts.sum().item()), "pairs": len(pairs), "matches": int(len(matches)),
           "verified_pairs": int((num >= 15).sum().item()), "kept_matches": int(keep.sum().item()), "match_s": t_match,
           "verify_s": t_ver, "tracks_s": t_trk, "tracks_over_match": t_trk / t_match, "tracks_over_verify": t_trk / t_ver,
           "tracks": len(cons), "consistent_tracks": int(cons.sum()), "observations": int(len(obs)),
           "mean_consistent_track_length": float(lengths[cons].mean()) if cons.any() else None,
           "note": "synthetic collection, random-init weights: not a statement about trained models"}
    rec["runs"].append(run)
    print(json.dumps(run), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--images", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tracks needs a GPU")
    from superpoint_nerf_pytorch_b200 import _native
    ctx = _native.get_context(0)
    rec = {"gpu": gpu_info(), "reps": args.reps, "runs": []}
    kernels(ctx, args.reps, rec)
    end_to_end(args.images, rec)
    rec["gpu_after"] = gpu_info()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rec, indent=2) + "\n")
    print(json.dumps({"gpu": rec["gpu"]}))


if __name__ == "__main__":
    main()
