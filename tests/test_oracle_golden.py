"""CPU: the oracle restatement (oracle/spn_oracle.py, oracle/nms_ref.c) against the golden vectors produced by the
unmodified reference (tests/golden/make_golden.py).  These pin the oracle; the GPU tests then use the oracle."""
import numpy as np
import pytest
import torch

from conftest import HA_CFG, MP_MODEL, SP_MODEL, rel_err
from oracle import kornia_shim as K
from oracle import spn_oracle as O

# The oracle's convolutions run on torch's CPU backend (oneDNN), whose float32 accumulation order depends on the host's
# instruction set and thread count.  On a host like the one that generated the goldens the oracle reproduces them bit
# for bit; on others every convolution output moves in its last bits (up to 5e-6 of the largest value was seen with one
# thread and AVX2).  So values computed through a convolution are compared to CONV_RTOL of the golden's largest magnitude
# with the same zero pattern, and everything discrete (NMS support, point maps, keypoint lists) or computed without a
# convolution stays bit-exact.
CONV_RTOL = 3e-5


def assert_conv_close(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, what
    assert np.array_equal(got != 0, want != 0), f"{what}: zero pattern differs"
    err = rel_err(got, want)
    assert err <= CONV_RTOL, f"{what}: {err:.2e} relative"


def test_nms_python_and_c_match_reference(golden):
    g = golden("nms_cases.npz")
    for i in range(int(g["n"])):
        p, par, want = g[f"c{i}_prob"], g[f"c{i}_par"], g[f"c{i}_out"]
        got_tv = O.box_nms(torch.from_numpy(p), par[0], par[1], par[2], int(par[3])).numpy()
        got_c = O.box_nms_c(p, par[0], par[1], par[2], int(par[3])).numpy()
        assert np.array_equal(got_tv, want), f"case {i}: torchvision restatement differs"
        assert np.array_equal(got_c, want), f"case {i}: C greedy restatement differs"


def test_nms_known_answers():
    """SURVEY.md section 4 items 1-2: footprint of size 4 / iou 0.1 and the tie-break."""
    for dy in range(-4, 5):
        for dx in range(-4, 5):
            if dy == 0 and dx == 0:
                continue
            p = np.zeros((16, 16), np.float32)
            p[8, 8] = 0.9
            p[8 + dy, 8 + dx] = 0.5
            out = O.box_nms_c(p, 4, 0.1, 0.1).numpy()
            inter = max(0, 4 - abs(dx)) * max(0, 4 - abs(dy))
            suppressed = 11 * inter > 32
            assert (out[8 + dy, 8 + dx] == 0) == suppressed, (dy, dx)
            assert np.array_equal(out, O.box_nms(torch.from_numpy(p), 4, 0.1, 0.1).numpy())
    p = np.zeros((12, 12), np.float32)
    p[5, 5] = p[5, 6] = p[6, 5] = 0.5
    out = O.box_nms_c(p, 4, 0.1, 0.1).numpy()
    assert out[5, 5] == 0.5 and out[5, 6] == 0 and out[6, 5] == 0


@pytest.mark.parametrize("tag,cfg", [("magicpoint", MP_MODEL), ("superpoint", SP_MODEL)])
def test_forward_matches_reference(golden, tag, cfg):
    g = golden(f"forward_{tag}.npz")
    sd = O.make_state_dict(cfg["model_name"], seed=int(g["seed"]), logit_gain=float(g["gain"]))
    out = O.model_forward(sd, torch.from_numpy(g["x"]), cfg)
    for k in ("logits", "prob_heatmap", "prob_heatmap_nms"):
        assert_conv_close(out["detector_output"][k].numpy(), g[k], k)
    assert np.array_equal(out["detector_output"]["pred_pts"].numpy(), g["pred_pts"])
    if tag == "superpoint":
        assert_conv_close(out["descriptor_output"]["desc_raw"].numpy(), g["desc_raw"], "desc_raw")
        d = out["descriptor_output"]["desc"][0].numpy()
        pts = g["desc_pts"]
        assert_conv_close(d[:, pts[:, 0], pts[:, 1]].T, g["desc_at_pts"], "desc_at_pts")
        sparse = O.sparse_descriptors(torch.from_numpy(g["desc_raw"][0]), pts).numpy()
        assert np.abs(sparse - g["desc_at_pts"]).max() < 1e-6


def test_sampler_bit_equal(golden):
    g = golden("homographies.npz")
    for s in range(6):
        np.random.seed(s)
        got = torch.cat([O.sample_homography((240, 320), **HA_CFG["params"]) for _ in range(3)]).numpy()
        assert np.array_equal(got, g[f"s{s}"])
    np.random.seed(100)
    p2 = dict(HA_CFG["params"], allow_artifacts=False, patch_ratio=0.5, n_scales=5, n_angles=25, translation_overflow=0.0)
    got = torch.cat([O.sample_homography((120, 160), **p2) for _ in range(3)]).numpy()
    assert np.array_equal(got, g["noartifact"])


def test_ha_step_matches_reference(golden):
    g = golden("ha_step.npz")
    img = torch.from_numpy(g["image"])
    for i in range(3):
        H = torch.from_numpy(g["H"][i:i + 1])
        proj, count, warped, mask = O.ha_step(lambda x: 0.25 + 0.5 * x[:, 0], img, H, 3)
        assert np.array_equal(warped[0, 0].numpy(), g[f"warped{i}"])
        assert np.array_equal(mask[0].numpy(), g[f"mask{i}"])
        assert np.array_equal(count[0].numpy(), g[f"count{i}"])
        assert np.array_equal(proj[0].numpy(), g[f"proj{i}"])


def test_shim_agrees_with_pixel_space_and_cv2(golden):
    """kornia is restated, not pinned: cross-check the restatement against an independent pixel-space formulation
    and against cv2.warpPerspective (SURVEY.md section 4 item 5)."""
    import cv2
    g = golden("ha_step.npz")
    img = torch.from_numpy(g["image"])
    for i in range(3):
        H = torch.from_numpy(g["H"][i:i + 1])
        a = K.warp_perspective(img, H, (120, 160))[0, 0].numpy()
        b = O.warp_pixelspace(img, H)[0, 0].numpy()
        assert np.abs(a - b).max() < 2e-4
        c = cv2.warpPerspective(g["image"][0, 0], g["H"][i].astype(np.float64), (160, 120), flags=cv2.INTER_LINEAR)
        assert np.abs(a - c).max() < 2e-2 and np.abs(a - c).mean() < 2e-3
        ones = torch.ones_like(img)
        mn = K.warp_perspective(ones, H, (120, 160), mode="nearest")[0, 0].numpy()
        mp = O.warp_pixelspace(ones, H, mode="nearest")[0, 0].numpy()
        assert (mn != mp).sum() <= 2


def test_erosion_kernel_known_answer():
    k = O.erosion_kernel(3).numpy().astype(int)
    rows = ["".join(map(str, r)) for r in k]
    assert rows == ["000100", "011111", "111111", "111111", "111111", "011111"]
    k2 = O.erosion_kernel(2).numpy().astype(int)
    assert ["".join(map(str, r)) for r in k2] == ["0010", "1111", "1111", "1111"]


def test_ha_export_matches_reference(golden):
    g = golden("ha_export.npz")
    sd = O.make_state_dict("magicpoint", seed=int(g["seed"]), logit_gain=float(g["gain"]))
    cfg = {"homography_adaptation": HA_CFG, "model": MP_MODEL}
    r = O.homography_adaptation(sd, torch.from_numpy(g["image"]), cfg, homographies=torch.from_numpy(g["H"]))
    assert_conv_close(r["mean_prob"].numpy(), g["agg"], "agg")
    assert_conv_close(r["nms_prob"].numpy(), g["nms"], "nms")
    assert r["keypoints"].dtype == np.int64 and np.array_equal(r["keypoints"], g["keypoints"])
    # drawing the homographies from numpy's global RNG in the reference's order reproduces them too
    np.random.seed(int(g["np_seed"]))
    r2 = O.homography_adaptation(sd, torch.from_numpy(g["image"]), cfg, nms_fn=O.box_nms_c)
    assert np.array_equal(r2["homographies"].numpy(), g["H"])
    assert np.array_equal(r2["keypoints"], g["keypoints"])
    # label file layout (SURVEY.md section 4 item 7): (N,2) int64, (row, col), row-major sorted
    kp = g["keypoints"]
    lin = kp[:, 0] * 160 + kp[:, 1]
    assert kp.ndim == 2 and kp.shape[1] == 2 and np.all(np.diff(lin) > 0)


def test_preprocessing_matches_reference(golden):
    """SURVEY section 8f-1: COCO.ratio_preserving_resize (+ /255) and HPatches.adapt_homography_to_resize."""
    g = golden("preprocess.npz")
    for k in range(int(g["n"])):
        img = torch.from_numpy(g[f"img{k}"]).to(torch.float32)
        out = O.ratio_preserving_resize(img, tuple(g[f"tgt{k}"]))
        assert np.array_equal(out.numpy(), g[f"out{k}"]), k
    h = O.adapt_homography_to_resize(g["h_in"], [480.0, 640.0], [427.0, 600.0], (240, 320))
    assert np.array_equal(h.numpy(), g["h_out"])


def test_detector_labels_restatement_matches_reference_loss(golden):
    """oracle.detector_labels / detector_loss (losses.py:6-38 restated) reproduce the reference's loss on the same torch
    seed, and the committed labels are what the restatement yields for the committed noise."""
    g = golden("train_reuse.npz")
    kmap, valid, logits = (torch.from_numpy(g[k]) for k in ("lab_kmap", "lab_valid", "lab_logits"))
    torch.manual_seed(77)
    assert torch.equal(O.detector_loss(logits, kmap, valid, include_mask=True), torch.as_tensor(g["loss_ref_masked"]))
    labels, cells, _ = O.detector_labels(kmap, valid, include_mask=True, noise=torch.from_numpy(g["lab_noise"]))
    assert np.array_equal(labels.numpy(), g["lab_labels"]) and np.array_equal(cells.numpy(), g["lab_cells"])


def test_eval_oracle_matches_reference(golden):
    """oracle/eval_oracle.py (repeatability, keep_shared_points, cross-checked matching) against the values the unmodified
    reference produced on the same synthetic pairs: rationals and point lists bit-equal, cv2 distances within 1e-6."""
    from conftest import make_eval_pair
    from oracle import eval_oracle as E
    g = golden("eval_cases.npz")
    reps = []
    for k, seed in enumerate(g["seeds"]):
        d = make_eval_pair(int(seed))
        for kk, thr in ((300, 3), (50, 1)):
            rep = E.repeatability_pair(d["prob"], d["warped_prob"], d["homography"], kk, thr)[0]
            assert rep == float(g[f"rep{k}_k{kk}_t{thr}"]), (k, kk, thr)
        reps.append(E.repeatability_pair(d["prob"], d["warped_prob"], d["homography"], 300, 3)[0])
        for kk in (1000, 60):
            kp1 = E.keep_shared_points(d["prob"], d["homography"], kk)
            kp2 = E.keep_shared_points(d["warped_prob"], np.linalg.inv(d["homography"]), kk)
            assert np.array_equal(kp1, g[f"hom{k}_k{kk}_kp1"]) and np.array_equal(kp2, g[f"hom{k}_k{kk}_kp2"])
            pairs, dist = E.order_matches(*E.mutual_nn(d["desc"][kp1[:, 0], kp1[:, 1]], d["warped_desc"][kp2[:, 0], kp2[:, 1]]))
            assert np.array_equal(pairs, g[f"hom{k}_k{kk}_matches"]), (k, kk)
            assert np.abs(dist - g[f"hom{k}_k{kk}_dist"]).max() < 1e-6
            assert len(pairs) / len(kp1) == float(g[f"hom{k}_k{kk}_score"])
    assert abs(np.mean(reps) - float(g["rep_all_k300_t3"])) < 1e-12
    # degenerate inputs the reference handles: no detections on one / both sides
    z = np.zeros((32, 40), np.float32)
    one = z.copy()
    one[5, 7] = 0.5
    assert np.isnan(E.repeatability_pair(z, z, np.eye(3))[0])
    assert E.repeatability_pair(one, z, np.eye(3))[:3] == (0.0, 1, 0)
    assert E.repeatability_pair(one, one, np.eye(3)) == (1.0, 1, 1, 1, 1)
    assert E.mutual_nn(np.zeros((0, 256), np.float32), np.ones((3, 256), np.float32))[0].shape == (0, 2)


def test_nerf_step_oracle_matches_reference(golden):
    """oracle/eval_oracle.nerf_step (NMS -> nonzero -> depth-aware re-projection -> border filter -> ordered 3x3 splat)
    against ExportNeRFDetections.step of the unmodified reference run with a stub model: bit-equal maps."""
    from conftest import make_nerf_batch
    from oracle import eval_oracle as E
    g = golden("nerf_step.npz")
    for c in range(int(g["n"])):
        bseed, nv, j, k = (int(v) for v in g[f"case{c}"])
        bt = make_nerf_batch(bseed, n_views=nv)
        raw = bt["raw"]
        got, pts = E.nerf_step(torch.from_numpy(g[f"heat{c}"]), raw["input_depth"][k], bt["camera_intrinsic_matrix"][j],
                               raw["input_rotation"][k], raw["input_translation"][k], raw["input_rotation"][j],
                               raw["input_translation"][j], int(g["nms"]), float(g["det_thresh"]), int(g["top_k"]), O.box_nms)
        assert len(pts) > 50
        assert np.array_equal(got, g[f"splat{c}"]), f"case {c}"


def test_ha_export_variants_match_reference(golden):
    """The two ExportDetections variants the GPU tests check against the oracle - aggregation 'max' (export.py:107-110)
    and enable_HA False (one plain forward, export.py:93-95) - pinned to the unmodified reference: aggregated map (the
    input of the final box_nms) and keypoint file bit-equal."""
    g = golden("ha_export_variants.npz")
    sd = O.make_state_dict("magicpoint", seed=int(g["seed"]), logit_gain=float(g["gain"]))
    img = torch.from_numpy(g["image"])
    r = O.homography_adaptation(sd, img, {"homography_adaptation": dict(HA_CFG, aggregation="max"), "model": MP_MODEL},
                                homographies=torch.from_numpy(g["max_H"]))
    assert_conv_close(r["mean_prob"].numpy(), g["max_agg"][0] if g["max_agg"].ndim == 3 else g["max_agg"], "max_agg")
    assert np.array_equal(r["keypoints"], g["max_keypoints"])
    np.random.seed(int(g["np_seed"]))           # the same homographies from numpy's global RNG in the reference's order
    r2 = O.homography_adaptation(sd, img, {"homography_adaptation": dict(HA_CFG, aggregation="max"), "model": MP_MODEL})
    assert np.array_equal(r2["homographies"].numpy(), g["max_H"]) and np.array_equal(r2["keypoints"], g["max_keypoints"])
    r3 = O.homography_adaptation(sd, img, {"homography_adaptation": dict(HA_CFG, num=1), "model": MP_MODEL})
    assert g["noha_H"].shape[0] == 0
    assert_conv_close(r3["mean_prob"].numpy(), g["noha_agg"][0] if g["noha_agg"].ndim == 3 else g["noha_agg"], "noha_agg")
    assert np.array_equal(r3["keypoints"], g["noha_keypoints"])
    assert len(g["max_keypoints"]) != len(g["noha_keypoints"])


def test_ha_masks_oracle_matches_reference(golden):
    """O.ha_masks (nearest warps of ones by H and H^-1 + elliptical erosion, export.py:49-66) against the 46 masks and 46
    counts ExportDetections.step of the unmodified reference produced at five image sizes and four margins."""
    g = golden("ha_masks.npz")
    total = 0
    for ci in range(int(g["n"])):
        h, w, margin, n = (int(v) for v in g[f"c{ci}_par"])
        want_m = np.unpackbits(g[f"c{ci}_mask"], axis=-1)[..., :w]
        want_c = np.unpackbits(g[f"c{ci}_count"], axis=-1)[..., :w]
        Hs = torch.from_numpy(g[f"c{ci}_H"])
        for i in range(n):
            m, c, _ = O.ha_masks(Hs[i:i + 1], (h, w), margin)
            assert np.array_equal(m[0].numpy(), want_m[i]) and np.array_equal(c[0].numpy(), want_c[i]), (ci, i)
            total += 1
    assert total == 46


def test_hpatches_export_values_match_reference(golden):
    """The oracle forward on the HPatches-style pair = the values Export_Hpatches_Repeatability / _Descriptors of the
    unmodified reference wrote (prob_heatmap_nms of both images, (H,W,256) descriptors at sampled points)."""
    g = golden("hpatches_export.npz")
    sd = O.make_state_dict("superpoint", seed=4, logit_gain=12.0)
    pts = g["des_pts"]
    for img_key, prob_key, desc_key in (("image", "rep_prob", "des_desc_at_pts"), ("warped_image", "rep_warped_prob", "des_warped_desc_at_pts")):
        out = O.model_forward(sd, torch.from_numpy(g[img_key]), SP_MODEL)
        assert_conv_close(out["detector_output"]["prob_heatmap_nms"][0].numpy(), g[prob_key], prob_key)
        desc = out["descriptor_output"]["desc"][0].numpy().transpose(1, 2, 0)
        assert_conv_close(desc[pts[:, 0], pts[:, 1]], g[desc_key], desc_key)
