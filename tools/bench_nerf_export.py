#!/usr/bin/env python
"""ExportNeRFDetections: the fused multi-view label pass (spn_nerf_fuse) against the per-pair path it replaced.

Synthetic posed batches in the style of tests/conftest.make_nerf_batch (smooth images, ray depth with an edge, small
relative poses; focal length scaled with the width) at 240x320 and 480x640 with V = 8, 16 and 32 views, a random-init
MagicPoint (f16) whose logits carry a seeded gain so that heatmaps are sparse, as in the goldens.  Reports, with the
GPU's name, power limit and clocks read in the same run:
  * ms per batch of export_NeRF (forward, draws, fusion, NMS, host copy, .npy writes): fused, and the per-pair path
    (one ExportNeRFDetections.reproject per (target, source) pair, one box_nms per target);
  * CUDA-event ms of spn_nerf_fuse alone on the same batch (heatmaps and keypoint lists already on the device);
  * keypoints per view, pairs per batch and the worst keypoint agreement (within 1 px, both directions) between the
    two paths' files, drawn with the same python seed.

    python tools/bench_nerf_export.py [--reps 5] [--out profiles/r4_nerf_fuse.json]
"""
import argparse
import copy
import json
import random
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

MODEL = {"script": "SuperPoint", "class_name": "SuperPoint", "model_name": "magicpoint", "precision": "f16",
         "vgg_cn": [64, 64, 64, 64, 128, 128, 128, 128],
         "detector_head": {"detector_dim": [128, 256], "grid_size": 8, "nms": 4, "det_thresh": 0.015, "top_k": 0}}


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def posed_batch(seed, V, H, W, tag):
    rng = np.random.RandomState(seed)
    coarse = torch.from_numpy(rng.rand(V, 1, H // 8 + 1, W // 8 + 1).astype(np.float32))
    imgs = torch.nn.functional.interpolate(coarse, size=(H, W), mode="bicubic", align_corners=False).clamp(0, 1)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    depth = np.stack([2.5 + 0.3 * np.sin(xx / (17.0 * W / 96)) + 0.2 * np.cos(yy / (11.0 * H / 64)) + 0.5 * (xx > W * (0.45 + 0.05 * (i % 8)))
                      for i in range(V)]).astype(np.float32)
    f = 85.0 * W / 96.0
    K = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]], np.float32)

    def rot(ax, ay, az):
        cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
        return (np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
                @ np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]))
    R = np.stack([rot(*rng.uniform(-0.03, 0.03, 3)) for _ in range(V)]).astype(np.float32)
    t = rng.uniform(-0.08, 0.08, (V, 3, 1)).astype(np.float32)
    return {"raw": {"image": imgs, "input_depth": torch.from_numpy(depth), "input_rotation": torch.from_numpy(R),
                    "input_translation": torch.from_numpy(t)},
            "camera_intrinsic_matrix": torch.from_numpy(np.stack([K] * V)), "name": [f"{tag}_{i:02d}" for i in range(V)]}


def exporter(model, out_dir, batches=()):
    from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportNeRFDetections
    ex = object.__new__(ExportNeRFDetections)
    ex.config, ex.model, ex.dataloader, ex.split, ex.device = {"model": copy.deepcopy(MODEL)}, model, list(batches), "bench", "cuda"
    ex.output_dir = Path(out_dir)
    ex.output_dir.mkdir(parents=True, exist_ok=True)
    return ex


@torch.no_grad()
def export_per_pair(ex, data):
    """The export loop as it ran before spn_nerf_fuse: per target, one reproject per drawn source view, stack / sum /
    divide, one box_nms, one host copy."""
    from superpoint_nerf_pytorch_b200.utils.train_utils import move_to_device
    dh = ex.config["model"]["detector_head"]
    data = move_to_device(data, ex.device)
    names = data["name"]
    out = ex.model(data["raw"]["image"], keypoints=True)["detector_output"]
    prob, kp, cnt = out["prob_heatmap"], out["keypoints"], out["keypoint_count"].cpu().numpy()
    ctx = ex.model.native()
    for j in range(len(names)):
        others = [k for k in range(len(names)) if k != j]
        others = random.choices(others, k=int(0.75 * len(others)))
        mean = ex.fuse_per_pair(prob, kp, cnt, data, [j], [0, len(others)], others)
        cap = min(mean.numel(), 16384)
        r = ctx.box_nms(mean, float(dh["nms"]), 0.1, float(dh["det_thresh"]), int(dh["top_k"]), det_thresh=float(dh["det_thresh"]),
                        want_map=False, max_kp=cap)
        n = int(r["kp_count"][0])
        np.save(Path(ex.output_dir, f"{names[j]}.npy"), r["kp"][0, :min(n, cap)].cpu().numpy().astype(np.int64))


def agreement(dir_a, dir_b, names):
    """Worst fraction, over files and both directions, of keypoints with a keypoint of the other file within 1 px."""
    from scipy.spatial import cKDTree
    worst = 1.0
    for nm in names:
        a, b = np.load(Path(dir_a, f"{nm}.npy")).astype(np.float64), np.load(Path(dir_b, f"{nm}.npy")).astype(np.float64)
        if len(a) == 0 and len(b) == 0:
            continue
        if len(a) == 0 or len(b) == 0:
            return 0.0
        da, _ = cKDTree(b).query(a, p=np.inf)
        db, _ = cKDTree(a).query(b, p=np.inf)
        worst = min(worst, float((da <= 1).mean()), float((db <= 1).mean()))
    return worst


def run_case(model, H, W, V, reps, tmp):
    dev = torch.device("cuda", 0)
    res = {"H": H, "W": W, "V": V}
    # spn_nerf_fuse alone on one batch
    data = posed_batch(V * 1000 + H, V, H, W, "k")
    data = {"raw": {k: v.to(dev) for k, v in data["raw"].items()}, "camera_intrinsic_matrix": data["camera_intrinsic_matrix"].to(dev)}
    out = model(data["raw"]["image"], keypoints=True)["detector_output"]
    rng = random.Random(V)
    targets, offsets, sources = list(range(V)), [0], []
    for j in range(V):
        sources += rng.choices([k for k in range(V) if k != j], k=int(0.75 * (V - 1)))
        offsets.append(len(sources))
    ctx = model.native()
    raw = data["raw"]
    args = (out["prob_heatmap"], out["keypoints"], out["keypoint_count"], raw["input_depth"], data["camera_intrinsic_matrix"],
            raw["input_rotation"], raw["input_translation"], targets, offsets, sources)
    for _ in range(3):
        ctx.nerf_fuse(*args)
    n_calls = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_calls):
        ctx.nerf_fuse(*args)
    e1.record()
    torch.cuda.synchronize()
    res["fuse_kernel_ms"] = e0.elapsed_time(e1) / n_calls
    res["pairs_per_batch"] = len(sources)
    res["keypoints_per_view_mean"] = float(out["keypoint_count"].float().mean())
    res["keypoints_per_view_max"] = int(out["keypoint_count"].max())

    # whole export_NeRF per batch: fused and per-pair, same batches, same python seed
    batches = [posed_batch(V * 1000 + H + r, V, H, W, f"r{r}") for r in range(reps + 1)]
    timings = {}
    for path in ("fused", "per_pair"):
        out_dir = Path(tmp, f"{path}_{H}x{W}_V{V}")
        ex = exporter(model, out_dir)
        random.seed(1234)
        times = []
        for r, bt in enumerate(batches):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if path == "fused":
                ex.dataloader = [bt]
                ex.export_NeRF()
            else:
                export_per_pair(ex, bt)
            torch.cuda.synchronize()
            if r:                                            # batch 0 warms up
                times.append((time.perf_counter() - t0) * 1e3)
        timings[path] = times
    res["export_ms_per_batch"] = {p: {"median": float(np.median(t)), "min": float(np.min(t)), "runs": [round(x, 3) for x in t]}
                                  for p, t in timings.items()}
    res["speedup_median"] = res["export_ms_per_batch"]["per_pair"]["median"] / res["export_ms_per_batch"]["fused"]["median"]
    res["keypoint_agreement_worst"] = agreement(Path(tmp, f"fused_{H}x{W}_V{V}"), Path(tmp, f"per_pair_{H}x{W}_V{V}"),
                                                [nm for bt in batches for nm in bt["name"]])
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5, help="timed batches per path and case (after one warm-up batch)")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_nerf_fuse.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("CUDA is not available: this measurement needs the GPU")
    from oracle import spn_oracle as O
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    torch.cuda.set_device(0)
    model = get_model(copy.deepcopy(MODEL), "cuda:0").eval()
    model.load_state_dict(O.make_state_dict("magicpoint", seed=13, logit_gain=12.0))
    res = {"tool": "tools/bench_nerf_export.py", "gpu_before": gpu_info(), "model": "magicpoint f16, random init, logit gain 12 (seed 13)",
           "reps": args.reps, "cases": []}
    with tempfile.TemporaryDirectory() as tmp:
        for H, W in ((240, 320), (480, 640)):
            for V in (8, 16, 32):
                case = run_case(model, H, W, V, args.reps, tmp)
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
