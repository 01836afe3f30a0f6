"""spn_verify_pairs (include/spn_verify.h) and verify.py on the GPU: decisions and models against the fp64 oracle
(oracle/verify_oracle.py) on planted scenes with ragged match counts, quality against the planted truth and cv2,
determinism and independence of the pair list, degenerate inputs, argument errors, guard bands and the matching CLI
end to end."""
import copy

import numpy as np
import pytest
import torch

from conftest import smooth_image
from oracle import verify_oracle as V
from verify_scenes import pool, scene

pytestmark = pytest.mark.gpu

KINDS = ("fundamental", "homography")
RATIOS = (0.25, 0.5, 0.9)
CAP = 2048


def _run(kp, pairs, offsets, matches, kind, **kw):
    from superpoint_nerf_pytorch_b200 import verify
    out = verify.verify_pairs(torch.from_numpy(kp).cuda(), torch.from_numpy(offsets).cuda(), torch.from_numpy(matches).cuda(),
                              pairs, kind, **kw)
    return [x.cpu().numpy() for x in out]


def _scenes(kind, seed):
    """Ragged match counts at every inlier ratio, plus a spread of mid-size pairs."""
    rng = np.random.RandomState(seed)
    sets = []
    for n in (0, 3, 7, 8, 127, 1000, CAP - 8):
        for ratio in RATIOS:
            xa, xb, _, _ = scene(rng, n, ratio, kind) if n >= 8 else (rng.randint(0, 640, (n, 2)), rng.randint(0, 480, (n, 2)), 0, 0)
            sets.append((xa, xb))
    for _ in range(40):
        xa, xb, _, _ = scene(rng, int(rng.randint(20, 400)), float(rng.choice([0.5, 0.7, 0.9])), kind)
        sets.append((xa, xb))
    return sets


def test_against_the_oracle():
    flagged = total = 0
    for kind in KINDS:
        sets = _scenes(kind, 11 if kind == "fundamental" else 12)
        kp, pairs, offsets, matches = pool(sets, CAP)
        models, num, hyp, best, inl = _run(kp, pairs, offsets, matches, kind)
        for p, (xa, xb) in enumerate(sets):
            a, b = pairs[p]
            want = V.ransac(xa, xb, a, b, kind)
            total += 1
            if want["margin"]:
                flagged += 1
                continue
            label = (kind, p, len(xa))
            assert (best[p], hyp[p], num[p]) == (want["best"], want["hypotheses"], want["num_inliers"]), \
                (label, best[p], hyp[p], num[p], want["best"], want["hypotheses"], want["num_inliers"])
            got_in = inl[offsets[p]:offsets[p + 1]]
            diff = got_in != want["inliers"]
            if diff.any():
                err = V.errors(want["model"], xa, xb, kind)
                assert (np.abs(err[diff] - 3.0) <= 1e-6).all(), label
            scale = max(np.abs(want["model"]).max(), 1e-300)
            assert np.abs(models[p] - want["model"]).max() <= 1e-8 * scale, (label, models[p], want["model"])
    print(f"margin rule: {flagged} of {total} pairs not compared")
    assert flagged < 0.01 * total


def test_quality_against_the_planted_truth_and_cv2():
    import cv2
    rng = np.random.RandomState(21)
    for kind in KINDS:
        for ratio in RATIOS:
            sets, truth = [], []
            for _ in range(4):
                # H: 0.3 px noise before rounding.  At 0.5 px the corner error of some 250-inlier planes exceeds 1 px
                # for the least-squares fit on all true matches too, which RANSAC's refit reproduces
                xa, xb, true, model = scene(rng, 1000, ratio, kind, noise=0.5 if kind == "fundamental" else 0.3)
                sets.append((xa, xb))
                truth.append((true, model))
            kp, pairs, offsets, matches = pool(sets, 1024)
            models, num, _, _, inl = _run(kp, pairs, offsets, matches, kind)
            rec, prec, ratio_cv = [], [], []
            for p, ((xa, xb), (true, model)) in enumerate(zip(sets, truth)):
                got = inl[offsets[p]:offsets[p + 1]]
                good = true & (V.errors(model, xa, xb, kind) < 1.5)
                rec.append((got & good).sum() / good.sum())
                prec.append((got & true).sum() / max(got.sum(), 1))
                fa, fb = xa.astype(np.float64), xb.astype(np.float64)
                if kind == "fundamental":
                    _, mask = cv2.findFundamentalMat(fa, fb, cv2.FM_RANSAC, 3.0, 0.999, 10000)
                else:
                    _, mask = cv2.findHomography(fa, fb, cv2.RANSAC, 3.0, maxIters=10000, confidence=0.999)
                ratio_cv.append(num[p] / max(int(mask.sum()) if mask is not None else 0, 1))
                if kind == "homography":
                    corners = np.array([[0, 0, 1], [639, 0, 1], [639, 479, 1], [0, 479, 1]], np.float64).T
                    pg, pt = models[p] @ corners, model @ corners
                    err = np.linalg.norm(pg[:2] / pg[2] - pt[:2] / pt[2], axis=0).max()
                    assert err < 1.0, (ratio, p, err)
            print(f"{kind} {ratio}: recall {min(rec):.4f} precision {min(prec):.4f} inliers / cv2 {min(ratio_cv):.3f}")
            assert min(ratio_cv) >= 0.95, (kind, ratio, ratio_cv)
            if kind == "fundamental" and ratio == 0.25:
                continue    # 10 000 7-point hypotheses are too few at w = 0.25 (w^7 = 6e-5): reported, not asserted
            assert min(rec) >= 0.99 and min(prec) >= 0.95, (kind, ratio, rec, prec)


def test_determinism_and_independence_of_the_pair_list():
    from superpoint_nerf_pytorch_b200 import _native
    rng = np.random.RandomState(31)
    for kind in KINDS:
        sets = [scene(rng, int(n), r, kind)[:2] for n, r in zip(rng.randint(8, 600, 12), rng.choice(RATIOS[1:], 12))]
        kp, pairs, offsets, matches = pool(sets, 1024)
        first = _run(kp, pairs, offsets, matches, kind)
        second = _run(kp, pairs, offsets, matches, kind)
        for x, y in zip(first, second):
            assert np.array_equal(x, y)
        for p in (0, 5, 11):                                     # alone
            sub_off = np.array([0, offsets[p + 1] - offsets[p]], np.int64)
            alone = _run(kp, pairs[p:p + 1], sub_off, matches[offsets[p]:offsets[p + 1]].copy(), kind)
            for k in range(4):
                assert np.array_equal(alone[k][0], first[k][p]), (kind, p, k)
            assert np.array_equal(alone[4], first[4][offsets[p]:offsets[p + 1]])
        rev = sets[::-1]                                         # reversed: same (a, b) per pair, other positions
        _, _, off_r, m_r = pool(rev, 1024)
        back = _run(kp, pairs[::-1].copy(), off_r, m_r, kind)
        for i in range(len(rev)):
            p = len(rev) - 1 - i
            for k in range(4):
                assert np.array_equal(back[k][i], first[k][p]), (kind, i, k)
            assert np.array_equal(back[4][off_r[i]:off_r[i + 1]], first[4][offsets[p]:offsets[p + 1]])
    # a list longer than VERIFY_MAX_PAIRS equals the calls split by hand
    n_pairs = _native.Context.VERIFY_MAX_PAIRS + 300
    sets = [(np.c_[rng.randint(0, 640, 10), rng.randint(0, 480, 10)], np.c_[rng.randint(0, 640, 10), rng.randint(0, 480, 10)])
            for _ in range(64)]
    kp, _, _, _ = pool(sets, 16)
    pairs = np.stack([np.arange(n_pairs) % 128, (np.arange(n_pairs) // 128 + np.arange(n_pairs) + 1) % 128], 1)
    offsets = np.arange(n_pairs + 1, dtype=np.int64) * 10
    matches = np.tile(np.c_[np.arange(10), np.arange(10)[::-1]], (n_pairs, 1)).astype(np.int32)
    whole = _run(kp, pairs, offsets, matches, "homography", max_iters=256)
    ctx = _native.get_context(0)
    step = _native.Context.VERIFY_MAX_PAIRS
    d = lambda x: torch.from_numpy(x).cuda()                     # noqa: E731
    for s in (0, step):
        part = ctx.verify_pairs(d(kp), d(offsets[s:s + step + 1].copy()), d(matches), pairs[s:s + step], "homography", 3.0, 0.999,
                                256, 0)
        for k in range(4):
            assert np.array_equal(part[k].cpu().numpy(), whole[k][s:s + step])
        lo, hi = offsets[s], offsets[min(s + step, n_pairs)]
        assert np.array_equal(part[4].cpu().numpy()[lo:hi].astype(bool), whole[4][lo:hi])
    assert (whole[3] >= 0).any()


def test_degenerate_inputs_give_no_model():
    rng = np.random.RandomState(41)
    line = np.c_[np.arange(0, 400, 10), np.arange(0, 400, 10) // 2]
    one = np.tile([[100, 200]], (50, 1))
    xa, xb, _, _ = scene(rng, 30, 1.0, "homography")
    dup = (np.repeat(xa[:1], 40, 0), np.repeat(xb[:1], 40, 0))
    cases = {"homography": [(line, line + 5), (one, one + 1), dup, (line[:0], line[:0])],
             "fundamental": [(one, one + 1), dup, (line[:0], line[:0])]}
    for kind, sets in cases.items():
        kp, pairs, offsets, matches = pool(sets, 64)
        models, num, hyp, best, inl = _run(kp, pairs, offsets, matches, kind, max_iters=1000)
        assert (num == 0).all() and (best == -1).all() and (models == 0).all() and not inl.any(), (kind, num, best)
        for p, (a, b) in enumerate(sets):
            assert hyp[p] == V.ransac(a, b, *pairs[p], kind, max_iters=1000)["hypotheses"], (kind, p)
    out = _run(np.zeros((1, 8, 2), np.int32), np.zeros((0, 2), np.int64), np.zeros(1, np.int64), np.zeros((0, 2), np.int32),
               "fundamental")                                     # no pairs at all
    assert out[0].shape == (0, 3, 3) and out[4].shape == (0,)


def test_errors_and_guard_bands():
    import superpoint_nerf_pytorch_b200 as P
    ctx = P.Context(0)
    rng = np.random.RandomState(51)
    sets = [scene(rng, n, 0.7, "homography")[:2] for n in (50, 60, 70, 80)]
    kp, pairs, offsets, matches = pool(sets, 128)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()   # noqa: E731
    want = ctx.verify_pairs(d(kp), d(offsets), d(matches), pairs, "homography")
    for kw, msg in ((dict(model="essential"), "model must be one of"), (dict(threshold=0.0), "threshold"),
                    (dict(threshold=float("nan")), "threshold"), (dict(threshold=-2.0), "threshold"),
                    (dict(confidence=0.0), "confidence"), (dict(confidence=1.0), "confidence"), (dict(max_iters=0), "max_iters")):
        with pytest.raises(P.NativeError, match=msg):
            ctx.verify_pairs(d(kp), d(offsets), d(matches), pairs, **dict(dict(model="homography"), **kw))
    with pytest.raises(P.NativeError, match="offsets"):
        ctx.verify_pairs(d(kp), d(offsets[:-1]), d(matches), pairs, "homography")
    # out-of-range offsets and indices on the device: -1 for that pair only
    bad_off = offsets.copy()
    bad_off[2] = offsets[3] + 1                                   # pair 1 holds more than cap matches, pair 2 ends before it starts
    bad_m = matches.copy()
    bad_m[offsets[3] + 5, 1] = 128                                # keypoint index == cap in pair 3
    bad_m[offsets[0] + 1, 0] = -1                                 # negative index in pair 0
    big = offsets.copy()
    big[4] = matches.shape[0] + 1                                 # last pair runs past M
    for off, m, bad in ((bad_off, matches, {1, 2}), (offsets, bad_m, {0, 3}), (big, matches, {3})):
        got = ctx.verify_pairs(d(kp), d(off), d(m), pairs, "homography")
        num = got[1].cpu().numpy()
        for p in range(4):
            if p in bad:
                assert num[p] == -1 and got[3][p].item() == -1 and (got[0][p] == 0).all(), (p, num)
            elif off[p] == offsets[p] and off[p + 1] == offsets[p + 1]:
                assert num[p] == want[1][p].item(), (p, num)
    again = ctx.verify_pairs(d(kp), d(offsets), d(matches), pairs, "homography")
    for x, y in zip(want, again):
        assert torch.equal(x, y)
    # every cap up to 16384 is accepted: a pair at the largest cap, both models
    xa, xb, _, _ = scene(rng, 16384, 0.9, "fundamental")
    kp, pairs, offsets, matches = pool([(xa, xb)], 16384)
    for kind in KINDS:
        out = ctx.verify_pairs(d(kp), d(offsets), d(matches), pairs, kind, max_iters=256)
        assert out[1][0].item() > 0 if kind == "fundamental" else out[1][0].item() >= 0
    assert ctx.check_guards() == 0
    ctx.close()


def test_cli_end_to_end(tmp_path, monkeypatch):
    """geometry.npz equals verify.verify_pairs on the tensors rebuilt from features.npz / matches.npz, is byte-stable,
    and the other outputs are the bytes of a run without the verification block."""
    import cv2
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import settings, verify
    root = tmp_path / "data" / "imgs"
    root.mkdir(parents=True)
    for i in range(5):
        img = (smooth_image(96, 128, 80 + i % 3) * 255).astype(np.uint8)
        cv2.imwrite(str(root / f"im{i}.png"), img)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(M.Path(M.__file__).parent / "configs" / "superpoint_match_verify.yaml"))
    cfg["data"].update(name="imgs", batch_size=2, preprocessing={"resize": [96, 128]})
    cfg["model"]["detector_head"].update(det_thresh=0.001, top_k=200)
    cfg["matching"].update(ratio=0.0)
    cfg["verification"].update(model="homography", min_inliers=10, max_iters=2000, seed=7)

    def run(name, c):
        c = copy.deepcopy(c)
        c["data"]["experiment_name"] = name
        path = tmp_path / f"{name}.yaml"
        path.write_text(yaml.safe_dump(c))
        M.main(config_path=str(path), random_init=True)
        out = tmp_path / "exper" / "matches" / name
        return out, {f.name: f.read_bytes() for f in out.iterdir()}

    out_dir, files = run("ver", cfg)
    assert sorted(files) == ["features.npz", "geometry.npz", "matches.npz"]
    _, again = run("ver", cfg)
    assert again == files
    plain = copy.deepcopy(cfg)
    del plain["verification"]
    _, base = run("plain", plain)
    assert sorted(base) == ["features.npz", "matches.npz"]
    assert base["features.npz"] == files["features.npz"] and base["matches.npz"] == files["matches.npz"]

    g, f, m = (np.load(out_dir / k) for k in ("geometry.npz", "features.npz", "matches.npz"))
    N, cap = len(f["names"]), 200
    kp = np.zeros((N, cap, 2), np.int32)
    for n in range(N):
        rows = f["keypoints"][f["offsets"][n]:f["offsets"][n + 1]]
        kp[n, :len(rows)] = rows
    models, num, hyp, best, inl = (x.cpu().numpy() for x in verify.verify_pairs(
        torch.from_numpy(kp).cuda(), torch.from_numpy(m["offsets"]).cuda(), torch.from_numpy(m["matches"]).cuda(), m["pairs"],
        "homography", 3.0, 0.999, 2000, 7))
    assert np.array_equal(g["pairs"], m["pairs"]) and np.array_equal(g["models"], models)
    assert np.array_equal(g["num_inliers"], num) and np.array_equal(g["hypotheses"], hyp) and np.array_equal(g["best"], best)
    assert g["inliers"].dtype == bool and np.array_equal(g["inliers"], inl) and len(g["inliers"]) == len(m["matches"])
    assert np.array_equal(g["verified"], num >= 10) and str(g["model"]) == "homography" and int(g["seed"]) == 7
    assert g["verified"].any(), num                               # the repeated images verify
