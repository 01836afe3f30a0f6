#!/usr/bin/env python
"""Posed-view evaluation (evaluations/posed_evaluation.py): time per chunk of the GPU path, of the host pose step and of
a per-pair host composition.

Synthetic posed scenes from a seed (tools/bench_nerf_export.posed_batch: the tests/conftest.make_nerf_batch geometry at
full size) at 480x640 with V = 8, 16 and 32 views and every pair of the chunk (28, 120 and 496 pairs), a SuperPoint (f16,
random init, seeded logit gain so that heatmaps are peaky) keeping its top 1000 keypoints.  Reports, with the GPU's
name, power limit and clocks read in the same run:
  * ms per chunk of evaluate_chunk without pose: forward, spn_posed_reproject, repeatability counts, matching, match
    correctness and the one host copy;
  * ms per chunk of the pose step: evaluate_chunk with pose minus evaluate_chunk without it (medians); the essential
    matrices run on the host on a thread pool;
  * ms per chunk of a per-pair host composition: the same forward and one host copy, then per pair the oracle
    reprojection (oracle/posed_oracle.py), brute-force counting, cv2.BFMatcher(NORM_L2, crossCheck=True) and match
    correctness;
  * CUDA-event ms of spn_posed_reproject alone on the chunk's keypoints.

    python tools/bench_posed_eval.py [--reps 3] [--out profiles/r5_posed_eval.json]
"""
import argparse
import copy
import json
import os
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_nerf_export import gpu_info, posed_batch  # noqa: E402

MODEL = {"script": "SuperPoint", "class_name": "SuperPoint", "model_name": "superpoint", "precision": "f16",
         "vgg_cn": [64, 64, 64, 64, 128, 128, 128, 128],
         "detector_head": {"detector_dim": [128, 256], "grid_size": 8, "nms": 4, "det_thresh": 0.015, "top_k": 1000},
         "descriptor_head": {"descriptor_dim": [128, 256], "grid_size": 8}}
EV = {"distance_thresh": 3.0, "depth_tol": 0.05, "max_gap": 0, "pose": True, "pose_thresh_px": 1.0}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


@torch.no_grad()
def per_pair_host(model, data, ev):
    """The evaluation as a user would compose it without the batched GPU path: one forward and one host copy, then one
    numpy reprojection, brute-force count and cv2 cross-checked match per pair."""
    import cv2

    from oracle import posed_oracle as O
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import pair_list
    out = model(data["raw"]["image"].cuda(), keypoints=True)
    kp = out["detector_output"]["keypoints"].cpu().numpy()
    cnt = out["detector_output"]["keypoint_count"].cpu().numpy()
    desc = out["descriptor_output"]["desc_sparse"].cpu().numpy()
    raw = data["raw"]
    depth, K = raw["input_depth"].numpy(), data["camera_intrinsic_matrix"].numpy()
    R, t = raw["input_rotation"].numpy(), raw["input_translation"].numpy()
    bf = cv2.BFMatcher(cv2.NORM_L2, crossCheck=True)
    res = []
    for a, b in pair_list(len(data["name"])):
        pa, va = O.reproject_points(kp[a, :cnt[a]], depth[a], depth[b], K[a], R[a], t[a], K[b], R[b], t[b], ev["depth_tol"])
        _, vb = O.reproject_points(kp[b, :cnt[b]], depth[b], depth[a], K[b], R[b], t[b], K[a], R[a], t[a], ev["depth_tol"])
        s1, s2 = pa[va][None], kp[b, :cnt[b]][vb].astype(np.float64)[None]
        counts = O.repeatability_counts(s1, [s1.shape[1]], s2, [s2.shape[1]], ev["distance_thresh"])[0]
        match = np.full(cnt[a], -1)
        for m in bf.match(desc[a, :cnt[a]], desc[b, :cnt[b]]):
            match[m.queryIdx] = m.trainIdx
        res.append((counts, O.match_correct(pa, va, kp[b], match, ev["distance_thresh"])))
    return res


def run_case(model, H, W, V, reps):
    import concurrent.futures as cf

    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import evaluate_chunk, pair_list, pose_auc
    res = {"H": H, "W": W, "V": V, "pairs": len(pair_list(V))}
    chunks = [posed_batch(V * 1000 + H + r, V, H, W, f"r{r}") for r in range(reps + 1)]
    ev_np = dict(EV, pose=False)
    with cf.ThreadPoolExecutor(max_workers=max(1, min(32, (os.cpu_count() or 2) - 1))) as pool:
        t = {"gpu_no_pose": [], "with_pose": [], "per_pair_host": []}
        for r, data in enumerate(chunks):
            ms_gpu, _ = timed(lambda: evaluate_chunk(model, data, ev_np, pool))
            ms_pose, out_pose = timed(lambda: evaluate_chunk(model, data, EV, pool))
            if r:                                               # chunk 0 warms up
                t["gpu_no_pose"].append(ms_gpu)
                t["with_pose"].append(ms_pose)
        for r, data in enumerate(chunks[:2]):                    # the host composition is slow: one warm-up, one timed
            ms, _ = timed(lambda: per_pair_host(model, data, EV))
            if r:
                t["per_pair_host"].append(ms)
    med = {k: float(np.median(v)) for k, v in t.items()}
    res["ms_per_chunk"] = {k: {"median": med[k], "runs": [round(x, 3) for x in v]} for k, v in t.items()}
    res["pose_step_ms"] = med["with_pose"] - med["gpu_no_pose"]
    res["per_pair_host_over_gpu_no_pose"] = med["per_pair_host"] / med["gpu_no_pose"]
    res["matches_per_pair_mean"] = float(np.mean(out_pose["n_matches"]))
    res["pose_auc_5_10_20"] = pose_auc(out_pose["pose_error"])

    # spn_posed_reproject alone on the last chunk's keypoints
    data = chunks[-1]
    dev = torch.device("cuda", 0)
    det = model(data["raw"]["image"].to(dev), keypoints=True)["detector_output"]
    raw = data["raw"]
    args = (det["keypoints"], det["keypoint_count"], raw["input_depth"].to(dev), data["camera_intrinsic_matrix"].to(dev),
            raw["input_rotation"].to(dev), raw["input_translation"].to(dev), pair_list(V), EV["depth_tol"])
    ctx = model.native()
    for _ in range(3):
        ctx.posed_reproject(*args)
    n_calls = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_calls):
        ctx.posed_reproject(*args)
    e1.record()
    torch.cuda.synchronize()
    res["posed_reproject_ms"] = e0.elapsed_time(e1) / n_calls
    res["keypoints_per_view_mean"] = float(det["keypoint_count"].float().mean())
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3, help="timed chunks per GPU measurement (after one warm-up chunk)")
    ap.add_argument("--views", default="8,16,32")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r5_posed_eval.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("CUDA is not available: this measurement needs the GPU")
    from oracle import spn_oracle as O
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    torch.cuda.set_device(0)
    model = get_model(copy.deepcopy(MODEL), "cuda:0").eval()
    model.load_state_dict(O.make_state_dict("superpoint", seed=13, logit_gain=12.0))
    res = {"tool": "tools/bench_posed_eval.py", "gpu_before": gpu_info(), "host_cpus": os.cpu_count(),
           "model": "superpoint f16, random init, logit gain 12 (seed 13), top_k 1000", "evaluation": EV, "reps": args.reps,
           "cases": []}
    for V in (int(v) for v in args.views.split(",")):
        case = run_case(model, 480, 640, V, args.reps)
        print(json.dumps(case), flush=True)
        res["cases"].append(case)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
