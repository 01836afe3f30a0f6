#!/usr/bin/env python
"""Retrieval (include/spn_retrieval.h, retrieval.py): kernel times, a host baseline and one end-to-end comparison of
retrieval against exhaustive pair selection.

Kernels (CUDA events over --reps calls after warm-up; the GPU's name, power limit and clocks are read in the same run):
  * spn_knn as word assignment (k = 1) of a pool of N x 1000 rows of C = 256 at N x cap = 1e6 and 1e7 rows, K = 64 and
    256 words; spn_residual_sums on the same pool; one k-means step (retrieval.lloyd_step: assignment, residual sums,
    the sum over images and the update).  The 1e7-row pool is 10 GB: every pass streams it from HBM;
  * spn_knn as retrieval (exclude_self, k = 20) over N = 1000, 4000 and 10 000 random unit VLAD-sized vectors of
    D = K x C = 16 384 and 65 536.  Useful FLOP = 2 N^2 D, executed = x3 (hi.hi + hi.lo + lo.hi).  The grid has
    ceil(N / 128) CTAs, fewer than the 148 SMs at every N here; the time is reported as it is.
Host baseline: numpy (BLAS) assignment and VLAD residual sums on a 1e5-row SAMPLE, extrapolated linearly (labelled).
End to end (synthetic collection, random-init seeded weights; not a statement about trained models): N images at
480 x 640, S = N / 10 scenes of drawn rectangles, ellipses, lines and checkerboards at seeded positions and scales, 10
views per scene by mild random homographies.  One feature extraction, then exhaustive pairs and retrieval pairs (k =
20, 64 words, 20 k-means steps), both matched with the mutual check and ratio 0.8.  Reports the wall time of pair
selection and of matching (host clock around device-synchronised steps), the pair counts and the pair recall: the
fraction of exhaustive pairs with >= 30 kept matches that retrieval also selects.

    python tools/bench_retrieval.py [--reps 5] [--images 1000] [--out profiles/r7_retrieval.json]
"""
import argparse
import copy
import json
import math
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_match import event_ms  # noqa: E402
from bench_nerf_export import gpu_info  # noqa: E402

CAP, DIM = 1000, 256


def unit_rows(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g)
    return x / x.norm(dim=-1, keepdim=True)


def kernels(ctx, retrieval, reps, rec):
    for rows in (10 ** 6, 10 ** 7):
        N = rows // CAP
        desc = unit_rows((N, CAP, DIM), rows)
        counts = torch.full((N,), CAP, dtype=torch.int32, device="cuda")
        for K in (64, 256):
            words = unit_rows((K, DIM), K)
            flat = desc.view(rows, DIM)
            knn_ms = event_ms(lambda: ctx.knn(flat, words, 1), reps)
            assign = retrieval.assign_words(desc, counts, words)
            res_ms = event_ms(lambda: ctx.residual_sums(desc, counts, assign, words), reps)
            step_ms = event_ms(lambda: retrieval.lloyd_step(desc, counts, words), reps)
            useful = 2.0 * rows * K * DIM
            run = {"what": "assignment", "rows": rows, "K": K, "C": DIM, "knn_ms": knn_ms,
                   "knn_useful_tflops": useful / knn_ms / 1e9, "knn_executed_tflops": 3 * useful / knn_ms / 1e9,
                   "residual_sums_ms": res_ms, "residual_sums_input_GBps": rows * DIM * 4 / res_ms / 1e6,
                   "kmeans_step_ms": step_ms}
            rec["runs"].append(run)
            print(json.dumps(run), flush=True)
            del assign
        del desc
        torch.cuda.empty_cache()
    for N in (1000, 4000, 10000):
        for D in (16384, 65536):
            v = unit_rows((N, D), N + D)
            ms = event_ms(lambda: ctx.knn(v, v, 20, True), max(1, reps // 2), warmup=1)
            useful = 2.0 * N * N * D
            run = {"what": "retrieval_knn", "N": N, "D": D, "k": 20, "ctas": math.ceil(N / 128), "ms": ms,
                   "useful_tflops": useful / ms / 1e9, "executed_tflops": 3 * useful / ms / 1e9}
            rec["runs"].append(run)
            print(json.dumps(run), flush=True)
            del v
            torch.cuda.empty_cache()


def host_baseline(rec):
    rng = np.random.RandomState(0)
    x = rng.randn(10 ** 5, DIM).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    for K in (64, 256):
        w = x[rng.choice(len(x), K, replace=False)]
        t0 = time.perf_counter()
        a = (-2.0 * (x @ w.T) + (w * w).sum(1)).argmin(1)
        t1 = time.perf_counter()
        sums = np.zeros((K, DIM), np.float32)
        np.add.at(sums, a, x - w[a])
        t2 = time.perf_counter()
        run = {"what": "host_numpy_sample", "rows": len(x), "K": K, "assign_ms": (t1 - t0) * 1e3, "vlad_sums_ms": (t2 - t1) * 1e3,
               "assign_ms_extrapolated_1e7": (t1 - t0) * 1e3 * 100, "vlad_sums_ms_extrapolated_1e7": (t2 - t1) * 1e3 * 100,
               "note": "numpy on a 1e5-row sample; the 1e7 figures are linear extrapolations, not measurements"}
        rec["runs"].append(run)
        print(json.dumps(run), flush=True)


def scene_images(n_images, views, H=480, W=640, seed=0):
    """Scenes of drawn shapes, lines and checkerboards; views by mild random homographies."""
    import cv2
    rng = np.random.RandomState(seed)
    out = []
    for s in range(n_images // views):
        base = np.full((H, W), rng.randint(60, 190), np.uint8)
        for _ in range(rng.randint(12, 24)):
            kind, c = rng.randint(4), int(rng.randint(0, 256))
            x0, y0 = int(rng.randint(0, W)), int(rng.randint(0, H))
            sz = int(rng.randint(15, 160))
            if kind == 0:
                cv2.rectangle(base, (x0, y0), (x0 + sz, y0 + int(sz * rng.uniform(0.3, 1.5))), c, -1)
            elif kind == 1:
                cv2.ellipse(base, (x0, y0), (sz // 2, int(sz * rng.uniform(0.2, 0.6))), float(rng.uniform(0, 180)), 0, 360, c, -1)
            elif kind == 2:
                cv2.line(base, (x0, y0), (int(rng.randint(0, W)), int(rng.randint(0, H))), c, int(rng.randint(2, 8)))
            else:
                cell = max(4, sz // int(rng.randint(3, 8)))
                yy, xx = np.mgrid[0:sz, 0:sz]
                board = np.where(((yy // cell) + (xx // cell)) % 2 == 0, c, 255 - c).astype(np.uint8)
                h, w = min(sz, H - y0), min(sz, W - x0)
                base[y0:y0 + h, x0:x0 + w] = board[:h, :w]
        for v in range(views):
            src = np.float32([[0, 0], [W, 0], [W, H], [0, H]])
            dst = src + rng.uniform(-0.06, 0.06, (4, 2)).astype(np.float32) * np.float32([W, H])
            hmat = cv2.getPerspectiveTransform(src, dst)
            out.append(cv2.warpPerspective(base, hmat, (W, H), borderMode=cv2.BORDER_REFLECT))
    return out


def end_to_end(n_images, rec):
    import cv2
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import retrieval, settings
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
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        items, kp, counts, desc = M.extract_features(model, ds, int(cfg["data"]["batch_size"]))
        torch.cuda.synchronize()
        t_extract = time.perf_counter() - t0
    N = len(items)
    r = M.retrieval_config(cfg)

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t

    def select():
        words = retrieval.kmeans(desc, counts, r["vocab_size"], r["kmeans_iters"])
        index, _ = retrieval.neighbors(retrieval.vlad(desc, counts, words), counts, r["num_neighbors"])
        return retrieval.retrieval_pairs(index)

    exh_pairs, t_exh_sel = timed(lambda: M.pair_list([it["name"] for it in items], "exhaustive"))
    (offsets, _, _), t_exh_match = timed(lambda: M.match_pairs(desc, counts, exh_pairs, True, 0.8, math.inf))
    kept = np.diff(offsets.cpu().numpy())
    strong = {p for p, n in zip(exh_pairs, kept) if n >= 30}
    ret_pairs, t_ret_sel = timed(select)
    _, t_ret_match = timed(lambda: M.match_pairs(desc, counts, ret_pairs, True, 0.8, math.inf))
    scene = np.arange(N) // views
    run = {"what": "end_to_end", "images": N, "size": [480, 640], "scenes": N // views, "views_per_scene": views,
           "weights": "random-init, torch.manual_seed(0)", "top_k": int(cfg["model"]["detector_head"]["top_k"]),
           "mean_keypoints": float(counts.float().mean()), "extract_s": t_extract,
           "exhaustive": {"pairs": len(exh_pairs), "select_s": t_exh_sel, "match_s": t_exh_match,
                          "pairs_with_30_matches": len(strong)},
           "retrieval": {"pairs": len(ret_pairs), "num_neighbors": r["num_neighbors"], "vocab_size": r["vocab_size"],
                         "kmeans_iters": r["kmeans_iters"], "select_s": t_ret_sel, "match_s": t_ret_match,
                         "pair_recall": len(strong & set(ret_pairs)) / max(1, len(strong)),
                         "same_scene_fraction": float(np.mean([scene[a] == scene[b] for a, b in ret_pairs]))},
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
        raise SystemExit("bench_retrieval needs a GPU")
    from superpoint_nerf_pytorch_b200 import _native, retrieval
    ctx = _native.get_context(0)
    rec = {"gpu": gpu_info(), "reps": args.reps, "runs": []}
    kernels(ctx, retrieval, args.reps, rec)
    host_baseline(rec)
    end_to_end(args.images, rec)
    rec["gpu_after"] = gpu_info()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rec, indent=2) + "\n")
    print(json.dumps({"gpu": rec["gpu"]}))


if __name__ == "__main__":
    main()
