"""Posed-view evaluation without a GPU: the fp64 reprojection oracle against closed forms, pose estimation and AUC, the
pair list, config validation, the output writer and the C ABI of include/spn_posed.h."""
import json
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_nerf_batch
from oracle import posed_oracle as O


def _plane_views(H=64, W=96, f=64.0, Z=4.0, tx=0.5):
    """Two views of a fronto-parallel plane at depth Z: view 0 at the origin, view 1 moved by tx along x (no rotation).
    With f = 64, Z = 4 and tx = 0.5 a point shifts by f tx / Z = 8 pixels exactly."""
    K = np.array([[f, 0, W / 2], [0, f, H / 2], [0, 0, 1]], np.float32)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    ray = np.sqrt(((xx - W / 2) / f) ** 2 + ((yy - H / 2) / f) ** 2 + 1.0)
    depth = np.stack([Z * ray, Z * ray]).astype(np.float32)     # distance along each pixel's ray
    R = np.stack([np.eye(3), np.eye(3)]).astype(np.float32)
    t = np.array([[0, 0, 0], [tx, 0, 0]], np.float32)
    return depth, np.stack([K, K]), R, t


def _grid_kp(H, W, step=5):
    rc = np.stack(np.meshgrid(np.arange(0, H, step), np.arange(0, W, step), indexing="ij"), -1).reshape(-1, 2)
    return rc.astype(np.int32)


def test_same_view_pair_maps_every_keypoint_onto_itself():
    bt = make_nerf_batch(3, n_views=3, h=64, w=96)
    depth = bt["raw"]["input_depth"].numpy()
    K, R, t = bt["camera_intrinsic_matrix"].numpy(), bt["raw"]["input_rotation"].numpy(), bt["raw"]["input_translation"].numpy()
    kp = _grid_kp(64, 96, 3)
    # the chain is not exact, so a keypoint on the image border may land a few ulps outside it: interior keypoints only
    kp = kp[(kp[:, 0] > 0) & (kp[:, 0] < 63) & (kp[:, 1] > 0) & (kp[:, 1] < 95)]
    for v in range(3):
        proj, vis = O.reproject_points(kp, depth[v], depth[v], K[v], R[v], t[v], K[v], R[v], t[v], 0.05)
        assert vis.all()
        assert np.allclose(proj, kp, rtol=0, atol=1e-9), np.abs(proj - kp).max()


def test_fronto_parallel_plane_shifts_by_f_tx_over_z():
    H, W = 64, 96
    depth, K, R, t = _plane_views(H, W)
    kp = _grid_kp(H, W)
    proj, vis = O.reproject_points(kp, depth[0], depth[1], K[0], R[0], t[0], K[1], R[1], t[1], 1e-3)
    want = kp.astype(np.float64) - [0.0, 8.0]
    assert np.abs(proj - want).max() < 1e-5
    assert np.array_equal(vis, want[:, 1] >= 0)                   # everything lands in b except what leaves on the left
    centre, cvis = O.reproject_points(np.array([[32, 48]]), depth[0], depth[1], K[0], R[0], t[0], K[1], R[1], t[1], 1e-3)
    assert centre.tolist() == [[32.0, 40.0]] and cvis.tolist() == [True]     # the principal ray: exact in binary
    # and back: b's keypoints move 8 pixels to the right in a
    proj_ba, vis_ba = O.reproject_points(kp, depth[1], depth[0], K[1], R[1], t[1], K[0], R[0], t[0], 1e-3)
    assert np.abs(proj_ba - (kp + [0.0, 8.0])).max() < 1e-5 and np.array_equal(vis_ba, kp[:, 1] + 8 <= W - 1)


def test_depth_step_hides_points_behind_an_occluder():
    H, W = 64, 96
    depth, K, R, t = _plane_views(H, W)
    depth[1][:, 60:] *= np.float32(0.5)                            # a nearer surface covers b's columns 60..95
    kp = _grid_kp(H, W)
    proj, vis = O.reproject_points(kp, depth[0], depth[1], K[0], R[0], t[0], K[1], R[1], t[1], 0.05)
    nearest = np.floor(proj[:, 1] + 0.5)
    assert np.array_equal(vis, (proj[:, 1] >= 0) & (nearest < 60))
    assert vis.sum() > 0 and (~vis & (nearest >= 60)).sum() > 0


def test_invalid_depths_and_outside_keypoints_are_never_visible():
    H, W = 64, 96
    depth, K, R, t = _plane_views(H, W)
    kp = np.array([[10, 20], [11, 21], [12, 22], [13, 23], [14, 24], [-1, 5], [5, W], [H, 0], [30, 40]], np.int32)
    for (r, c), v in zip(kp[:5], (0.0, np.nan, -4.0, np.inf, -np.inf)):
        depth[0][r, c] = v                                         # zero, NaN, behind the camera, infinite
    proj, vis = O.reproject_points(kp, depth[0], depth[1], K[0], R[0], t[0], K[1], R[1], t[1], 0.05)
    assert vis.tolist() == [False] * 8 + [True]
    assert np.isnan(proj[1]).all() and np.isnan(proj[5:8]).all()   # NaN depth and keypoints outside the image
    assert np.isfinite(proj[8]).all()


def test_oracle_layout_sets_and_counts():
    """posed_reproject's compacted sets are the visible points in keypoint order; a count above max_kp is clamped."""
    H, W = 64, 96
    depth, K, R, t = _plane_views(H, W)
    kp = np.zeros((2, 40, 2), np.int32)
    kp[0, :30] = _grid_kp(H, W, 12)[:30]
    kp[1, :40] = _grid_kp(H, W, 11)[:40]
    out = O.posed_reproject(kp, np.array([30, 99]), depth, K, R, t, [(0, 1), (1, 1)], 1e-3)
    v = out["vis"][0, 0, :30].astype(bool)
    assert out["set_count"][0, 0] == v.sum() and np.array_equal(out["set1"][0, :v.sum()], out["proj"][0, :30][v])
    v2 = out["vis"][0, 1, :40].astype(bool)
    assert out["set_count"][0, 1] == v2.sum() and np.array_equal(out["set2"][0, :v2.sum()], kp[1, :40][v2].astype(np.float64))
    assert out["set_count"][1].tolist() == [40, 40]                # (b, b): count 99 clamped to max_kp = 40
    assert np.isnan(out["set1"][0, v.sum():]).all() and np.isnan(out["proj"][0, 30:]).all()


def _camera_pair(seed):
    rng = np.random.RandomState(seed)

    def rot(ax, ay, az):
        cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
        return (np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
                @ np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]))
    R = [rot(*rng.uniform(-0.2, 0.2, 3)) for _ in range(2)]
    t = [rng.uniform(-0.5, 0.5, 3) for _ in range(2)]
    K = [np.array([[500.0, 0, 320], [0, 510, 240], [0, 0, 1]]), np.array([[450.0, 0, 300], [0, 440, 250], [0, 0, 1]])]
    Xc = np.stack([rng.uniform(-2, 2, 200), rng.uniform(-1.5, 1.5, 200), rng.uniform(4, 8, 200)], 1)   # in camera a
    Xw = Xc @ R[0].T + t[0]

    def project(v):
        Xv = (Xw - t[v]) @ R[v]                                    # R^-1 = R^T for a rotation
        p = Xv @ K[v].T
        return np.stack([p[:, 1] / p[:, 2], p[:, 0] / p[:, 2]], 1)  # (row, col)
    return project(0), project(1), K, R, t


def test_pose_from_exact_correspondences():
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import angle_errors, estimate_pose, relative_pose
    for seed in range(3):
        pa, pb, K, R, t = _camera_pair(seed)
        R_gt, t_gt = relative_pose(R[0], t[0], R[1], t[1])
        R_o, t_o = O.relative_pose(R[0], t[0], R[1], t[1])
        assert np.allclose(R_gt, R_o) and np.allclose(t_gt, t_o)
        R_est, t_est = estimate_pose(pa, pb, K[0], K[1], 1.0)
        err_r, err_t = angle_errors(R_est, t_est, R_gt, t_gt)
        assert err_r < 1e-3 and err_t < 1e-3, (seed, err_r, err_t)
        assert np.allclose((err_r, err_t), O.pose_error(R_est, t_est, R_gt, t_gt), atol=1e-9)
        # a flipped translation has the same direction error; an unrelated rotation does not pass
        assert angle_errors(R_est, -t_est, R_gt, t_gt)[1] < 1e-3
        assert angle_errors(R_est @ O.relative_pose(np.eye(3), [0, 0, 0], R[1], [0, 0, 0])[0], t_est, R_gt, t_gt)[0] > 1.0
    assert estimate_pose(pa[:4], pb[:4], K[0], K[1], 1.0) is None


def test_pose_auc_hand_computed():
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import pose_auc
    # errors 1, 2, inf, inf: the curve goes (0, 0) -> (1, 1/4) -> (2, 1/2), then stays at 1/2
    #   at 5:  (1 * 1/8 + 1 * 3/8 + 3 * 1/2) / 5 = 0.4      at 10: (0.5 + 8 * 1/2) / 10 = 0.45     at 20: (0.5 + 9) / 20
    want = [0.4, 0.45, 9.5 / 20]
    assert np.allclose(pose_auc([2.0, np.inf, 1.0, np.inf]), want, rtol=0, atol=1e-15)
    assert np.allclose(O.pose_auc([2.0, np.inf, 1.0, np.inf], (5, 10, 20)), want, rtol=0, atol=1e-15)
    assert pose_auc([0.0, 0.0]) == [1.0, 1.0, 1.0] and pose_auc([np.inf]) == [0.0, 0.0, 0.0]
    rng = np.random.RandomState(0)
    e = np.where(rng.rand(300) < 0.2, np.inf, rng.exponential(8.0, 300))
    assert np.allclose(pose_auc(e), O.pose_auc(e, (5, 10, 20)), rtol=1e-12, atol=0)


def test_pair_list():
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import pair_list
    assert pair_list(4) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    assert pair_list(4, 1) == [(0, 1), (1, 2), (2, 3)]
    assert pair_list(5, 2) == [(0, 1), (0, 2), (1, 2), (1, 3), (2, 3), (2, 4), (3, 4)]
    assert pair_list(1) == [] and pair_list(0) == []
    assert len(pair_list(32)) == 496


def test_config_validation_names_the_key():
    import yaml
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import EVAL_DEFAULTS, eval_config
    cfg = yaml.safe_load((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_posed_eval.yaml").read_text())
    assert eval_config(cfg) == {"distance_thresh": 3.0, "depth_tol": 0.05, "max_gap": 0, "pose": True, "pose_thresh_px": 1.0}
    assert eval_config({}) == EVAL_DEFAULTS
    bad = [("distance_tresh", 3), ("distance_thresh", 0), ("distance_thresh", "3"), ("depth_tol", -0.1),
           ("depth_tol", float("inf")), ("max_gap", -1), ("max_gap", 1.5), ("max_gap", True), ("pose", "yes"),
           ("pose_thresh_px", 0.0), ("pose_thresh_px", float("nan"))]
    for key, value in bad:
        with pytest.raises(ValueError, match=f"evaluation.{key}"):
            eval_config({"evaluation": {key: value}})


def test_summary_and_files(tmp_path):
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import _write_npz, summarize
    ev = {"distance_thresh": 3.0, "depth_tol": 0.05, "max_gap": 0, "pose": True, "pose_thresh_px": 1.0}
    per_pair = {"a": np.array([0, 0]), "repeatability": np.array([0.5, np.nan]), "precision": np.array([1.0, np.nan]),
                "matching_score": np.array([0.25, 0.75]), "pose_error": np.array([1.0, np.inf])}
    s = summarize(per_pair, True, True, ev, "superpoint")
    assert s["n_pairs"] == 2 and s["repeatability"] == 0.5 and s["precision"] == 1.0 and s["matching_score"] == 0.5
    assert s["pose_auc@5"] == pytest.approx(0.5 * 4 / 5 + 0.25 / 5)
    m = summarize({"a": per_pair["a"], "repeatability": per_pair["repeatability"]}, False, False, ev, "magicpoint")
    assert "repeatability only" in m["note"] and "precision" not in m and "pose_auc@5" not in m
    arrays = {"name_a": np.array(["s_f000", "s_f001"]), "x": np.arange(3.0)}
    _write_npz(tmp_path / "one.npz", arrays)
    _write_npz(tmp_path / "two.npz", arrays)
    assert (tmp_path / "one.npz").read_bytes() == (tmp_path / "two.npz").read_bytes()
    z = np.load(tmp_path / "one.npz")
    assert z["name_a"].tolist() == ["s_f000", "s_f001"] and np.array_equal(z["x"], arrays["x"])
    json.dumps(s)


@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_cabi_exports_the_posed_reproject_symbol(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_posed.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.POSED_PROTOTYPES) == ["spn_posed_reproject"]
    assert not set(N.POSED_PROTOTYPES) & (set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES) | set(N.NERF_PROTOTYPES))
    assert hasattr(ctypes.CDLL(str(built_lib)), "spn_posed_reproject")


def test_posed_reproject_rejects_null_arguments(built_lib):
    """NULL context and zero arguments -> -1 and a message, no CUDA call (child process)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
for name, (res, args) in N.POSED_PROTOTYPES.items():
    rc = getattr(lib, name)(*[None if a in (C.c_void_p, C.c_char_p) else a(0) for a in args])
    msg = lib.spn_last_error().decode()
    assert rc == -1 and "null pointer" in msg, (name, rc, msg)
print("checked", len(N.POSED_PROTOTYPES))
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 1" in out.stdout, out.stderr[-2000:]


def test_cli_is_single_process(tmp_path, monkeypatch):
    from superpoint_nerf_pytorch_b200.evaluations import posed_evaluation as PE
    cfg = tmp_path / "eval.yaml"
    cfg.write_text((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_posed_eval.yaml").read_text())
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit, match="single process"):
        PE.main(config_path=str(cfg))
    monkeypatch.setenv("WORLD_SIZE", "1")
    bad = tmp_path / "bad.yaml"
    bad.write_text(cfg.read_text().replace("depth_tol: 0.05", "depth_tol: -1"))
    with pytest.raises(ValueError, match="evaluation.depth_tol"):
        PE.main(config_path=str(bad))
    if not torch.cuda.is_available():
        with pytest.raises(SystemExit, match="CUDA is not available"):
            PE.main(config_path=str(cfg), random_init=True)
