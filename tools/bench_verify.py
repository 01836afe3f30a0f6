#!/usr/bin/env python
"""Geometric verification (include/spn_verify.h, verify.py): kernel times against a host cv2 baseline, and one
end-to-end row after retrieval matching.

Kernel (CUDA events after a warm-up call on 64 pairs; one timed call for F at 0.25, --reps for the others; the GPU's name, power limit and clocks are read in the same run):
spn_verify_pairs on P = 8128 pairs (the exhaustive pairs of 128 images) of 1000 integer-rounded planted matches each
(tests/verify_scenes.py: random 3-D points seen by two cameras for F, a plane for H, uniform outliers), both models at
inlier ratios 0.25 / 0.5 / 0.9, threshold 3 px, confidence 0.999, max_iters 10 000.  64 distinct scenes are tiled over
the pairs; every pair has its own (a, b) and so its own samples.  Reports the time per call, the hypotheses drawn per
pair and the inliers found.
Host baseline: cv2.findFundamentalMat(FM_RANSAC) / cv2.findHomography(RANSAC) with the same threshold, confidence and
iterations on a 128-pair SAMPLE on 15 threads, extrapolated linearly to all pairs (labelled as extrapolated).
End to end (synthetic collection of tools/bench_retrieval.py, random-init seeded weights; not a statement about trained
models): 1000 images, one extraction, retrieval pairs, matching with the mutual check and ratio 0.8, then
verify.verify_pairs with both models; wall times of matching and verification (host clock around device-synchronised
steps) and the verified pairs.

    python tools/bench_verify.py [--reps 3] [--images 1000] [--out profiles/r8_verify.json]
"""
import argparse
import copy
import json
import math
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))

from bench_nerf_export import gpu_info  # noqa: E402
from verify_scenes import scene  # noqa: E402

P, N_MATCH, DISTINCT = 8128, 1000, 64
THRESH, CONF, ITERS = 3.0, 0.999, 10000


def planted(kind, ratio):
    rng = np.random.RandomState(int(ratio * 100) + (0 if kind == "fundamental" else 1000))
    scenes = [scene(rng, N_MATCH, ratio, kind)[:2] for _ in range(DISTINCT)]
    kp = np.zeros((2 * P, N_MATCH, 2), np.int32)
    for p in range(P):
        xa, xb = scenes[p % DISTINCT]
        kp[2 * p], kp[2 * p + 1] = xa[:, ::-1], xb[:, ::-1]
    pairs = np.arange(2 * P).reshape(P, 2)
    offsets = np.arange(P + 1, dtype=np.int64) * N_MATCH
    matches = np.tile(np.c_[np.arange(N_MATCH), np.arange(N_MATCH)], (P, 1)).astype(np.int32)
    return scenes, kp, pairs, offsets, matches


def host_sample(scenes, kind, n=128, threads=15):
    import cv2

    def one(i):
        xa, xb = (x.astype(np.float64) for x in scenes[i % len(scenes)])
        if kind == "fundamental":
            _, mask = cv2.findFundamentalMat(xa, xb, cv2.FM_RANSAC, THRESH, CONF, ITERS)
        else:
            _, mask = cv2.findHomography(xa, xb, cv2.RANSAC, THRESH, maxIters=ITERS, confidence=CONF)
        return 0 if mask is None else int(mask.sum())

    cv2.setNumThreads(1)
    t = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        counts = list(ex.map(one, range(n)))
    return time.perf_counter() - t, counts


def kernels(ctx, reps, rec):
    for kind in ("fundamental", "homography"):
        for ratio in (0.25, 0.5, 0.9):
            scenes, kp, pairs, offsets, matches = planted(kind, ratio)
            d_kp, d_off, d_m = (torch.from_numpy(x).cuda() for x in (kp, offsets, matches))
            call = lambda: ctx.verify_pairs(d_kp, d_off, d_m, pairs, kind, THRESH, CONF, ITERS, 0)   # noqa: E731
            ctx.verify_pairs(d_kp, d_off[:65], d_m, pairs[:64], kind, THRESH, CONF, ITERS, 0)           # warm-up
            torch.cuda.synchronize()
            n_reps = 1 if kind == "fundamental" and ratio == 0.25 else reps   # ~10 240 hypotheses per pair: one call
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n_reps):
                out = call()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / n_reps
            num, hyp = out[1].cpu().numpy(), out[2].cpu().numpy()
            host_s, host_counts = host_sample(scenes, kind)
            run = {"what": "spn_verify_pairs", "model": kind, "inlier_ratio": ratio, "pairs": P, "matches_per_pair": N_MATCH,
                   "threshold": THRESH, "confidence": CONF, "max_iters": ITERS, "reps": n_reps, "ms_per_call": ms,
                   "us_per_pair": 1e3 * ms / P, "hypotheses_per_pair": {"mean": float(hyp.mean()), "min": int(hyp.min()),
                                                                        "max": int(hyp.max())},
                   "mean_inliers": float(num.mean()),
                   "host_cv2": {"sample_pairs": len(host_counts), "threads": 15, "sample_s": host_s,
                                "extrapolated_all_pairs_s": host_s * P / len(host_counts),
                                "mean_inliers": float(np.mean(host_counts)),
                                "note": "extrapolated linearly from the sample, not measured on all pairs"}}
            rec["runs"].append(run)
            print(json.dumps(run), flush=True)
            del d_kp, d_off, d_m, out


def end_to_end(n_images, rec):
    import cv2
    import yaml
    from bench_retrieval import scene_images
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import retrieval, settings, verify
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
    scene_id = np.arange(len(items)) // views
    same = np.array([scene_id[a] == scene_id[b] for a, b in pairs])
    run = {"what": "end_to_end", "images": len(items), "size": [480, 640], "weights": "random-init, torch.manual_seed(0)",
           "pairs": len(pairs), "matches": int(len(matches)), "match_s": t_match, "verify": {},
           "note": "synthetic collection, random-init weights: not a statement about trained models"}
    for kind in ("fundamental", "homography"):
        verify.verify_pairs(kp, offsets[:65], matches, pairs[:64], kind)             # warm-up
        (models, num, hyp, best, inl), t_ver = timed(lambda: verify.verify_pairs(kp, offsets, matches, pairs, kind))
        num, hyp = num.cpu().numpy(), hyp.cpu().numpy()
        ok = num >= 15
        run["verify"][kind] = {"verify_s": t_ver, "verify_over_match": t_ver / t_match, "verified_pairs": int(ok.sum()),
                               "verified_same_scene_fraction": float(same[ok].mean()) if ok.any() else None,
                               "inlier_matches": int(inl.sum().item()), "mean_hypotheses": float(hyp.mean())}
    rec["runs"].append(run)
    print(json.dumps(run), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--images", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_verify needs a GPU")
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
