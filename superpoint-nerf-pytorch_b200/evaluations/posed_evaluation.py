"""Detector and descriptor evaluation on posed multi-view scenes (data/PosedViews.py): depth-reprojected repeatability,
match precision and matching score, and relative-pose AUC.

    python -m superpoint_nerf_pytorch_b200.evaluations.posed_evaluation --config_path configs/superpoint_posed_eval.yaml \
        [--split training] [--random_init True]

The unit of work is one chunk of views as the ``export_NeRF_labels`` loader yields it (up to ``data.batch_size``
consecutive frames of one scene).  Pairs are taken inside a chunk only and never span chunks: set ``data.batch_size`` to
the scene length to evaluate every pair of a scene.  ``pair_list`` gives the pairs (a, b), a < b, optionally limited to
b - a <= ``evaluation.max_gap``.

Per chunk, up to one device-to-host copy, everything runs on the GPU:
  1. one ``model(images, keypoints=True)`` call: the keypoints of the model config's NMS, ``det_thresh`` and ``top_k``;
  2. one ``spn_posed_reproject`` call: every keypoint of a mapped into b through a's ray depth and both poses, with the
     visibility and occlusion test of include/spn_posed.h (``evaluation.depth_tol``);
  3. one ``spn_repeatability_counts`` call over all pairs: {N1, N2, count1, count2} within ``distance_thresh`` and
     repeatability = (count1 + count2) / (N1 + N2), as in detector_evaluation;
  4. SuperPoint only: ``spn_mutual_nn_match`` on the sparse descriptors of a and b (gathered in groups of at most 64
     pairs).  A match (i, j) is correct when keypoint i of a is visible in b and its reprojection lies within
     ``distance_thresh`` of keypoint j of b (fp64).  Precision = correct / matches, matching score = correct / N1.
  5. SuperPoint with ``evaluation.pose``: the relative pose of each pair from its matches, on the host on a thread pool
     (as compute_homography keeps cv2.findHomography on the host).  This protocol is this package's own definition; it
     is not a port of the reference's pose_evaluation.py, whose source this package does not have.  The matched points
     are normalised with K_a and K_b; cv2.findEssentialMat(identity K, RANSAC, prob 0.99999, threshold
     ``pose_thresh_px`` / mean(fx_a, fy_a, fx_b, fy_b)); cv2.recoverPose on each 3x3 candidate, keeping the one with the
     most inliers.  Ground truth: R_ab = R_b^-1 R_a, t_ab = R_b^-1 (t_a - t_b).  The pose error is the larger of the
     rotation angle of R_est^T R_ab and the angle between the translation directions (min(e, 180 - e)); it is inf with
     fewer than 5 matches or when no pose is found.  The AUC at 5, 10 and 20 degrees integrates the cumulative error
     curve with np.trapezoid.

MagicPoint models have no descriptors: they get repeatability only, and the summary says so.

``evaluate_posed_views`` writes ``<EXPER_PATH>/posed_eval/<experiment_name>/<split>/pairs.npz`` (per-pair arrays with
the frame names) and ``summary.json``; the same inputs give byte-identical files.
"""
from __future__ import annotations

import concurrent.futures as cf
import io
import json
import math
import os
import zipfile
from pathlib import Path
from typing import Literal

import numpy as np
import torch

from .. import settings

AUC_THRESHOLDS = (5.0, 10.0, 20.0)
MATCH_GROUP = 64          # pairs per mutual_nn_match call: bounds the gathered descriptors to 2 x 64 x max_kp x 256 fp32
MAX_PAIRS = 65535         # pairs per chunk (one spn_posed_reproject call)
EVAL_DEFAULTS = {"distance_thresh": 3.0, "depth_tol": 0.05, "max_gap": 0, "pose": True, "pose_thresh_px": 1.0}


def eval_config(config) -> dict:
    """The ``evaluation`` block with defaults filled in.  Unknown or out-of-range keys raise ValueError naming the key."""
    block = config.get("evaluation") or {}
    if not isinstance(block, dict):
        raise ValueError(f"evaluation: expected a mapping, got {block!r}")
    for k in block:
        if k not in EVAL_DEFAULTS:
            raise ValueError(f"evaluation.{k}: unknown key (known: {', '.join(EVAL_DEFAULTS)})")
    ev = dict(EVAL_DEFAULTS, **block)

    def number(k, ok, what):
        v = ev[k]
        if isinstance(v, bool) or not isinstance(v, (int, float)) or not math.isfinite(v) or not ok(v):
            raise ValueError(f"evaluation.{k}: must be {what}, got {v!r}")
        return float(v)

    ev["distance_thresh"] = number("distance_thresh", lambda v: v > 0, "a finite number > 0")
    ev["depth_tol"] = number("depth_tol", lambda v: v >= 0, "a finite number >= 0")
    ev["pose_thresh_px"] = number("pose_thresh_px", lambda v: v > 0, "a finite number > 0")
    if isinstance(ev["max_gap"], bool) or not isinstance(ev["max_gap"], int) or ev["max_gap"] < 0:
        raise ValueError(f"evaluation.max_gap: must be an integer >= 0 (0: every pair of a chunk), got {ev['max_gap']!r}")
    if not isinstance(ev["pose"], bool):
        raise ValueError(f"evaluation.pose: must be true or false, got {ev['pose']!r}")
    return ev


def pair_list(V, max_gap=0):
    """All (a, b) with a < b < V, and b - a <= max_gap when max_gap > 0."""
    return [(a, b) for a in range(V) for b in range(a + 1, V) if max_gap <= 0 or b - a <= max_gap]


def pose_auc(errors, thresholds=AUC_THRESHOLDS):
    """Area under the cumulative pose-error curve up to each threshold, divided by the threshold."""
    e = np.sort(np.asarray(errors, np.float64))
    recall = np.arange(1, len(e) + 1) / max(len(e), 1)
    e, recall = np.r_[0.0, e], np.r_[0.0, recall]
    out = []
    for th in thresholds:
        last = int(np.searchsorted(e, th))
        out.append(float(np.trapezoid(np.r_[recall[:last], recall[last - 1]], x=np.r_[e[:last], th]) / th))
    return out


def relative_pose(R_a, t_a, R_b, t_b):
    """Motion from camera a to camera b of camera-to-world poses: X_b = R_ab X_a + t_ab."""
    Rb_inv = np.linalg.inv(np.asarray(R_b, np.float64).reshape(3, 3))
    return (Rb_inv @ np.asarray(R_a, np.float64).reshape(3, 3),
            Rb_inv @ (np.asarray(t_a, np.float64).reshape(3) - np.asarray(t_b, np.float64).reshape(3)))


def angle_errors(R_est, t_est, R_gt, t_gt):
    """(rotation error, translation-direction error) in degrees; the sign of the translation is not observable."""
    cos_r = (np.trace(np.asarray(R_est, np.float64).T @ R_gt) - 1.0) / 2.0
    err_r = math.degrees(math.acos(min(1.0, max(-1.0, cos_r))))
    t_est, t_gt = np.asarray(t_est, np.float64).reshape(3), np.asarray(t_gt, np.float64).reshape(3)
    den = np.linalg.norm(t_est) * np.linalg.norm(t_gt)
    if not den > 0:
        return err_r, math.inf
    err_t = math.degrees(math.acos(min(1.0, max(-1.0, float(t_est @ t_gt) / den))))
    return err_r, min(err_t, 180.0 - err_t)


def estimate_pose(pts_a, pts_b, K_a, K_b, thresh_px):
    """(R, t) from (n,2) (row, col) correspondences of two calibrated views, or None (fewer than 5 points, no model)."""
    import cv2
    if len(pts_a) < 5:
        return None

    def normalise(pts, K):
        Ki = np.linalg.inv(np.asarray(K, np.float64).reshape(3, 3))
        h = np.stack([pts[:, 1], pts[:, 0], np.ones(len(pts))]).astype(np.float64)   # (x = col, y = row, 1)
        x = Ki @ h
        return np.ascontiguousarray((x[:2] / x[2]).T)

    K_a, K_b = np.asarray(K_a, np.float64).reshape(3, 3), np.asarray(K_b, np.float64).reshape(3, 3)
    xa, xb = normalise(pts_a, K_a), normalise(pts_b, K_b)
    thresh = thresh_px / np.mean([K_a[0, 0], K_a[1, 1], K_b[0, 0], K_b[1, 1]])
    E, mask = cv2.findEssentialMat(xa, xb, np.eye(3), method=cv2.RANSAC, prob=0.99999, threshold=float(thresh))
    if E is None or E.shape[0] < 3:
        return None
    best = None
    for Ei in np.split(E, E.shape[0] // 3):
        n, R, t, _ = cv2.recoverPose(Ei, xa, xb, np.eye(3), mask=mask.copy())
        if best is None or n > best[0]:
            best = (n, R, t)
    return best[1], best[2].reshape(3)


def _pose_job(pts_a, pts_b, K_a, K_b, gt, thresh_px):
    est = estimate_pose(pts_a, pts_b, K_a, K_b, thresh_px)
    if est is None:
        return math.inf, math.inf
    return angle_errors(est[0], est[1], *gt)


def _check_model(model):
    dh = model.config["detector_head"]
    if not dh.get("nms"):
        raise ValueError("model.detector_head.nms must be > 0: the evaluation takes the model's post-NMS keypoint lists")
    return hasattr(model, "descriptor_head")


@torch.no_grad()
def evaluate_chunk(model, data, ev, pool=None):
    """One chunk (the loader's item dictionary) -> dict of per-pair numpy arrays (a, b, N1, N2, count1, count2,
    repeatability and, for SuperPoint, n_matches, n_correct, precision, matching_score and with ``ev["pose"]`` err_R,
    err_t, pose_error).  ``ev`` is eval_config's result."""
    sp = _check_model(model)
    dev = next(model.parameters()).device
    raw = data["raw"]
    V = len(data["name"])
    pairs = pair_list(V, ev["max_gap"])
    P = len(pairs)
    if P > MAX_PAIRS:
        raise ValueError(f"{P} pairs in one chunk (at most {MAX_PAIRS}): lower data.batch_size or set evaluation.max_gap")
    res = {"a": np.array([p[0] for p in pairs], np.int32).reshape(P), "b": np.array([p[1] for p in pairs], np.int32).reshape(P)}
    if P == 0:
        return res
    f32 = lambda x: x.to(dev, torch.float32)  # noqa: E731
    out = model(f32(raw["image"]), keypoints=True)
    det = out["detector_output"]
    kp, cnt = det["keypoints"], det["keypoint_count"]
    max_kp = kp.shape[1]
    ctx = model.native()
    K = data["camera_intrinsic_matrix"]
    r = ctx.posed_reproject(kp, cnt, f32(raw["input_depth"]), f32(K), f32(raw["input_rotation"]), f32(raw["input_translation"]),
                            pairs, ev["depth_tol"])
    counts = ctx.repeatability_counts(r["set1"], r["set_count"][:, 0].contiguous(), r["set2"], r["set_count"][:, 1].contiguous(),
                                      ev["distance_thresh"])
    host = [counts.reshape(-1), cnt]
    pose = sp and ev["pose"]
    if sp:
        ia = torch.tensor(res["a"], dtype=torch.int64, device=dev)
        ib = torch.tensor(res["b"], dtype=torch.int64, device=dev)
        desc = out["descriptor_output"]["desc_sparse"]
        n = cnt.clamp(0, max_kp)
        match = torch.empty((P, max_kp), dtype=torch.int32, device=dev)
        for g in range(0, P, MATCH_GROUP):
            sa, sb = ia[g:g + MATCH_GROUP], ib[g:g + MATCH_GROUP]
            match[g:g + MATCH_GROUP] = ctx.mutual_nn_match(desc.index_select(0, sa), n.index_select(0, sa),
                                                           desc.index_select(0, sb), n.index_select(0, sb))[0]
        matched = match >= 0
        j = match.clamp(min=0).to(torch.int64)
        kp_b = torch.gather(kp.index_select(0, ib), 1, j[..., None].expand(-1, -1, 2)).to(torch.float64)
        dy = r["proj"][..., 0] - kp_b[..., 0]
        dx = r["proj"][..., 1] - kp_b[..., 1]
        correct = matched & (r["vis"][:, 0] != 0) & (torch.sqrt(dy * dy + dx * dx) <= ev["distance_thresh"])
        host += [matched.sum(1, dtype=torch.int32), correct.sum(1, dtype=torch.int32)]
        if pose:
            host += [match.reshape(-1), kp.reshape(-1)]
    flat = torch.cat(host).cpu().numpy()          # the one device-to-host copy
    sizes = [4 * P, V] + ([P, P] if sp else []) + ([P * max_kp, V * max_kp * 2] if pose else [])
    parts = np.split(flat, np.cumsum(sizes)[:-1])
    counts, cnt = parts[0].reshape(P, 4), parts[1]
    if cnt.max(initial=0) > max_kp:
        raise RuntimeError("keypoint list overflow: set model.detector_head.top_k")
    res.update(N1=counts[:, 0], N2=counts[:, 1], count1=counts[:, 2], count2=counts[:, 3])
    n12 = counts[:, 0] + counts[:, 1]
    with np.errstate(invalid="ignore", divide="ignore"):
        res["repeatability"] = np.where(n12 > 0, (counts[:, 2] + counts[:, 3]) / np.maximum(n12, 1), np.nan)
        if sp:
            nm, nc = parts[2], parts[3]
            res.update(n_matches=nm, n_correct=nc, precision=np.where(nm > 0, nc / np.maximum(nm, 1), np.nan),
                       matching_score=np.where(counts[:, 0] > 0, nc / np.maximum(counts[:, 0], 1), np.nan))
    if pose:
        match, kp_h = parts[4].reshape(P, max_kp), parts[5].reshape(V, max_kp, 2)
        Kh = K.cpu().numpy().reshape(V, 3, 3)
        Rh, th = raw["input_rotation"].cpu().numpy().reshape(V, 3, 3), raw["input_translation"].cpu().numpy().reshape(V, 3)
        jobs = []
        for q, (a, b) in enumerate(pairs):
            i = np.nonzero(match[q] >= 0)[0]
            jobs.append((kp_h[a, i], kp_h[b, match[q, i]], Kh[a], Kh[b], relative_pose(Rh[a], th[a], Rh[b], th[b]),
                         ev["pose_thresh_px"]))
        errs = list(pool.map(lambda j: _pose_job(*j), jobs)) if pool is not None else [_pose_job(*j) for j in jobs]
        res["err_R"] = np.array([e[0] for e in errs], np.float64)
        res["err_t"] = np.array([e[1] for e in errs], np.float64)
        res["pose_error"] = np.maximum(res["err_R"], res["err_t"])
    return res


def _mean(x):
    x = np.asarray(x, np.float64)
    x = x[~np.isnan(x)]
    return float(x.mean()) if len(x) else None


def summarize(per_pair, sp, pose, ev, model_name):
    """Summary of the concatenated per-pair arrays."""
    s = {"model": model_name, "n_pairs": int(len(per_pair["a"])), "distance_thresh": ev["distance_thresh"],
         "depth_tol": ev["depth_tol"], "max_gap": ev["max_gap"], "repeatability": _mean(per_pair.get("repeatability", []))}
    if not sp:
        s["note"] = "repeatability only: the model has no descriptor head, so there are no matches and no poses"
        return s
    s["precision"] = _mean(per_pair["precision"])
    s["matching_score"] = _mean(per_pair["matching_score"])
    if pose:
        aucs = pose_auc(per_pair["pose_error"]) if len(per_pair["pose_error"]) else [None] * len(AUC_THRESHOLDS)
        s.update({f"pose_auc@{int(t)}": v for t, v in zip(AUC_THRESHOLDS, aucs)})
        s["pose_thresh_px"] = ev["pose_thresh_px"]
    else:
        s["note"] = "pose not evaluated (evaluation.pose: false)"
    return s


def _write_npz(path, arrays):
    """np.savez without the zip members' wall-clock timestamps, so that equal arrays give equal bytes."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_STORED) as z:
        for k in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[k]), allow_pickle=False)
            z.writestr(zipfile.ZipInfo(f"{k}.npy", date_time=(1980, 1, 1, 0, 0, 0)), buf.getvalue())


def evaluate_posed_views(config, model, loader, split="training", workers=None):
    """Evaluate every chunk of ``loader`` (the ``export_NeRF_labels`` loader's items) -> the summary dictionary; writes
    ``<EXPER_PATH>/posed_eval/<data.experiment_name>/<split>/pairs.npz`` and ``summary.json``."""
    ev = eval_config(config)
    model = model.eval()
    sp = _check_model(model)
    pose = sp and ev["pose"]
    keys = ["chunk", "a", "b", "name_a", "name_b", "N1", "N2", "count1", "count2", "repeatability"]
    keys += ["n_matches", "n_correct", "precision", "matching_score"] if sp else []
    keys += ["err_R", "err_t", "pose_error"] if pose else []
    acc = {k: [] for k in keys}
    with cf.ThreadPoolExecutor(max_workers=workers or max(1, min(32, (os.cpu_count() or 2) - 1))) as pool:
        for c, data in enumerate(loader):
            res = evaluate_chunk(model, data, ev, pool)
            names = list(data["name"])
            res.update(chunk=np.full(len(res["a"]), c, np.int32), name_a=np.array([names[a] for a in res["a"]], dtype=str),
                       name_b=np.array([names[b] for b in res["b"]], dtype=str))
            if len(res["a"]) == 0:
                continue
            for k in keys:
                acc[k].append(res[k])
    dtypes = {"chunk": np.int32, "a": np.int32, "b": np.int32, "name_a": str, "name_b": str}
    per_pair = {k: np.concatenate(v) if v else np.zeros(0, dtypes.get(k, np.float64)) for k, v in acc.items()}
    summary = summarize(per_pair, sp, pose, ev, config["model"].get("model_name", ""))
    summary["split"] = split
    out_dir = Path(settings.EXPER_PATH, "posed_eval", config["data"]["experiment_name"], split)
    out_dir.mkdir(parents=True, exist_ok=True)
    _write_npz(out_dir / "pairs.npz", per_pair)
    (out_dir / "summary.json").write_text(json.dumps(summary, indent=2, sort_keys=True) + "\n")
    return summary


def main(config_path: str, split: Literal["training", "validation", "test"] = "training", random_init: bool = False) -> None:
    """Evaluate a model on the posed views of one split.

    Args:
        config_path: Path to configuration.
        split: The split of the PosedViews dataset to evaluate.
        random_init: skip loading `pretrained` (random-init weights, torch.manual_seed(0)).
    """
    import yaml
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        raise SystemExit("posed_evaluation runs as a single process: run it without torchrun (WORLD_SIZE > 1)")
    with open(config_path, "r") as f:
        config = yaml.safe_load(f)
    eval_config(config)
    if not torch.cuda.is_available():
        raise SystemExit("CUDA is not available: this implementation has no CPU fallback")
    from ..engine import load_pretrained
    from ..utils.data_loaders import get_loader
    from ..utils.get_model import get_model
    device = f"cuda:{torch.cuda.current_device()}"
    if random_init:
        torch.manual_seed(0)
    model = get_model(config["model"], device=device)
    if not random_init:
        assert config["pretrained"], "Use a pretrained model to evaluate."
        load_pretrained(model, config, device)
    loader = get_loader(config, "export_NeRF_labels", device=device, export_split=split)
    print(json.dumps(evaluate_posed_views(config, model, loader, split), indent=2, sort_keys=True))


if __name__ == "__main__":
    import tyro
    tyro.cli(tyro.conf.configure(tyro.conf.FlagConversionOff)(main), use_underscores=True)
