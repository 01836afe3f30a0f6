"""spn_match_pairs (include/spn_match.h) and matching.py on the GPU: indices, keep decisions and distances against the
fp64 oracle (oracle/match_oracle.py) for every filter combination, equality with spn_mutual_nn_match, argument errors,
guard bands, the per-call pair limit and the CLI end to end."""
import copy
import itertools
import math

import numpy as np
import pytest
import torch

from conftest import SP_MODEL, smooth_image
from oracle import match_oracle as O

pytestmark = pytest.mark.gpu

MARGIN = 1e-5      # decisions are compared where the oracle is at least this far (in d^2) from flipping them
DIST_TOL = 1e-5    # the matcher tolerance of DESIGN.md section 4: on d^2 everywhere, and on d where d >= 0.5 (the
                   # square root divides the few-1e-6 error of d^2 by 2d: ~1e-3 near 0, 3e-5 at d = 0.06)
FILTERS = list(itertools.product((False, True), (0.0, 0.8, 1.0), (math.inf, 1.1)))   # mutual x ratio x max_dist


def _unit(shape, rng):
    x = rng.randn(*shape).astype(np.float32)
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def _pool_random(N, cap, counts, seed, C=256):
    rng = np.random.RandomState(seed)
    desc = np.zeros((N, cap, C), np.float32)
    for n, c in enumerate(counts):
        desc[n, :c] = _unit((c, C), rng)
    return desc


def _pool_duplicates(seed, cap=300, C=256):
    """Sets with exact copies of rows inside a set and across sets, and near-copies (noise 0.05)."""
    rng = np.random.RandomState(seed)
    counts = [300, 250, 180, 1]
    desc = _pool_random(4, cap, counts, seed, C)
    desc[1, :60] = desc[0, :60]                              # b shares rows with a
    desc[1, 60:70] = desc[0, 5]                              # ten more copies of a5 in b (b5 is one): ties to the lower index
    desc[0, 200:210] = desc[0, 7]                            # copies of a7 inside a: the mutual check keeps a7
    near = desc[0, 100:160] + 0.05 * rng.randn(60, C).astype(np.float32)
    desc[2, :60] = near / np.linalg.norm(near, axis=1, keepdims=True)
    desc[3, 0] = desc[0, 0]
    return desc, counts


def _pool_superpoint(top_k=300, n_img=6):
    from oracle import spn_oracle
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    cfg = copy.deepcopy(SP_MODEL)
    cfg["detector_head"]["top_k"] = top_k
    cfg["precision"] = "f16"
    model = get_model(cfg, "cuda").eval()
    model.load_state_dict(spn_oracle.make_state_dict("superpoint", seed=1, logit_gain=10.0))
    imgs = np.stack([smooth_image(120, 160, 900 + i) for i in range(n_img)])
    x = torch.from_numpy(imgs)[:, None].cuda()
    x[1] = x[0]                                              # an identical image: identical descriptor sets
    x[2] = torch.flip(x[0], dims=[2])
    out = model(x, keypoints=True)
    return out["descriptor_output"]["desc_sparse"].cpu().numpy(), out["detector_output"]["keypoint_count"].cpu().numpy()


def _compare(desc, counts, pairs, label):
    """Every filter combination against the oracle; returns the number of queries the margin rule excluded."""
    from superpoint_nerf_pytorch_b200 import _native
    ctx = _native.get_context(0)
    d, c = torch.from_numpy(desc).cuda(), torch.from_numpy(np.asarray(counts, np.int32)).cuda()
    excluded = total = 0
    for mutual, ratio, max_dist in FILTERS:
        m, dist = ctx.match_pairs(d, c, pairs, mutual, ratio, max_dist)
        m, dist = m.cpu().numpy(), dist.cpu().numpy()
        want = O.match_pairs(desc, counts, pairs, mutual, ratio, max_dist)
        sure = want["margin"] > MARGIN
        assert np.array_equal(m[sure], want["match"][sure]), (label, mutual, ratio, max_dist)
        kept = sure & (m >= 0)
        got_d, want_d = dist[kept].astype(np.float64), want["dist"][kept]
        assert np.abs(got_d ** 2 - want_d ** 2).max(initial=0) <= DIST_TOL, (label, mutual, ratio, max_dist)
        far = want_d >= 0.5
        assert np.abs(got_d[far] - want_d[far]).max(initial=0) <= DIST_TOL, (label, mutual, ratio, max_dist)
        assert (dist[m < 0] == 0).all()
        cap = desc.shape[1]
        n_a = np.clip(np.asarray(counts)[[a for a, _ in pairs]], 0, cap)
        assert (m[np.arange(cap)[None] >= n_a[:, None]] == -1).all()
        excluded += int((~sure & (np.arange(cap)[None] < n_a[:, None])).sum())
        total += int(n_a.sum())
    print(f"{label}: {len(pairs)} pairs x {len(FILTERS)} filter settings, {excluded} of {total} queries within the "
          f"{MARGIN:g} decision margin (not compared)")
    return excluded, total


def test_random_unit_vectors_ragged_counts():
    rng = np.random.RandomState(11)
    counts = [0, 1, 1000, 999, 517, 130, 129, 128, 2]
    desc = _pool_random(len(counts), 1000, counts, 1)
    pairs7 = [(2, 3), (3, 2), (4, 5), (6, 7), (0, 4), (4, 0), (8, 1)]
    _compare(desc, counts, pairs7, "N=9 cap=1000 P=7")
    _compare(desc, counts, [(4, 2)], "N=9 cap=1000 P=1")
    counts = rng.randint(0, 200, 40)
    counts[:3] = [0, 1, 199]
    desc = _pool_random(40, 199, counts, 2)
    pairs = [tuple(p) for p in rng.randint(0, 40, (300, 2))]
    ex, tot = _compare(desc, counts, pairs, "N=40 cap=199 P=300")
    assert ex < 0.01 * tot


def test_planted_duplicates():
    desc, counts = _pool_duplicates(3)
    pairs = [(0, 1), (1, 0), (0, 2), (2, 0), (0, 3), (3, 0), (0, 0), (1, 1)]
    _compare(desc, counts, pairs, "duplicates")
    from superpoint_nerf_pytorch_b200 import _native
    ctx = _native.get_context(0)
    m, _ = ctx.match_pairs(torch.from_numpy(desc).cuda(), torch.tensor(counts, dtype=torch.int32).cuda(), [(0, 1)], False)
    assert m[0, 5].item() == 5                               # the first of the eleven copies of a5 in b
    m, _ = ctx.match_pairs(torch.from_numpy(desc).cuda(), torch.tensor(counts, dtype=torch.int32).cuda(), [(0, 1)], False, 1.0)
    assert m[0, 5].item() == -1                              # d1 == d2 fails the strict ratio test


def test_superpoint_descriptors():
    desc, counts = _pool_superpoint()
    assert counts.min() > 20
    pairs = [(a, b) for a in range(len(counts)) for b in range(len(counts)) if a != b] + [(0, 0)]
    ex, tot = _compare(desc, counts, pairs, "SuperPoint descriptors")
    assert tot - ex >= 1000


def test_mutual_only_equals_mutual_nn_match():
    from superpoint_nerf_pytorch_b200 import _native
    ctx = _native.get_context(0)
    rng = np.random.RandomState(5)
    random_counts = rng.randint(0, 1001, 12)
    for desc, counts in ((_pool_random(12, 1000, random_counts, 6), random_counts), _pool_superpoint()):
        N = len(counts)
        d, c = torch.from_numpy(desc).cuda(), torch.from_numpy(np.asarray(counts, np.int32)).cuda()
        pairs = np.array([(a, b) for a in range(N) for b in range(N)], np.int64)
        m, dist = ctx.match_pairs(d, c, pairs, True, 0.0, math.inf)
        ia, ib = torch.from_numpy(pairs[:, 0]).cuda(), torch.from_numpy(pairs[:, 1]).cuda()
        m_ref, d_ref = ctx.mutual_nn_match(d.index_select(0, ia), c.index_select(0, ia), d.index_select(0, ib), c.index_select(0, ib))
        assert torch.equal(m, m_ref) and torch.equal(dist, d_ref)
        if counts is not random_counts:
            continue          # these SuperPoint sets hold near-duplicate descriptors: no identity on (a, a)
        for a in range(N):                                   # (a, a): the identity
            q = a * N + a
            n = int(counts[a])
            assert torch.equal(m[q, :n].cpu(), torch.arange(n, dtype=torch.int32)) and (m[q, n:] == -1).all()


def test_python_api_compacts_and_splits_long_pair_lists(monkeypatch):
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200._native import Context
    counts = np.random.RandomState(8).randint(0, 300, 20)
    desc = _pool_random(20, 300, counts, 9)
    d, c = torch.from_numpy(desc).cuda(), torch.from_numpy(counts.astype(np.int32)).cuda()
    pairs = M.pair_list([str(i) for i in range(20)], "exhaustive")
    full = M.match_pairs(d, c, pairs, True, 0.8, 1.2)
    monkeypatch.setattr(Context, "MATCH_MAX_PAIRS", 7)
    split = M.match_pairs(d, c, pairs, True, 0.8, 1.2)
    assert all(torch.equal(x, y) for x, y in zip(full, split))
    offsets, matches, distances = (x.cpu().numpy() for x in full)
    want = O.match_pairs(desc, counts, pairs, True, 0.8, 1.2)
    assert offsets[0] == 0 and offsets[-1] == len(matches) == len(distances)
    for q in range(len(pairs)):
        mq = matches[offsets[q]:offsets[q + 1]]
        sure = want["margin"][q, mq[:, 0]] > MARGIN
        assert np.all(np.diff(mq[:, 0]) > 0)                 # keypoint order of a
        assert np.array_equal(mq[sure, 1], want["match"][q, mq[sure, 0]])
    empty = M.match_pairs(d, c, [])
    assert empty[0].tolist() == [0] and empty[1].shape == (0, 2) and empty[2].shape == (0,)


def test_errors_and_guard_bands():
    import superpoint_nerf_pytorch_b200 as P
    ctx = P.Context(0)
    rng = np.random.RandomState(4)
    counts = rng.randint(0, 260, 9).astype(np.int32)
    counts[0] = 300                                          # above cap: clamped
    d = torch.from_numpy(_pool_random(9, 257, np.minimum(counts, 257), 4)).cuda()
    c = torch.from_numpy(counts).cuda()
    pairs = [(0, 1), (2, 3), (8, 8)]
    want = ctx.match_pairs(d, c, pairs, True, 0.8, 1.0)
    for kw, msg in ((dict(ratio=1.5), r"ratio must be in \[0, 1\]"), (dict(max_dist=float("nan")), "max_dist must not be NaN"),
                    (dict(pairs=[(0, 1), (2, 9)]), r"pair 1 = \(2, 9\) has a set index outside \[0, 9\)"),
                    (dict(pairs=[(-1, 0)]), "set index outside")):
        args = dict(pairs=pairs, mutual=True, ratio=0.8, max_dist=1.0) | kw
        with pytest.raises(P.NativeError, match=msg):
            ctx.match_pairs(d, c, args["pairs"], args["mutual"], args["ratio"], args["max_dist"])
    with pytest.raises(P.NativeError, match="multiple of 64"):
        ctx.match_pairs(d[..., :100].contiguous(), c, pairs)
    with pytest.raises(P.NativeError, match="must be"):
        ctx.match_pairs(d, c.to(torch.int64), pairs)
    again = ctx.match_pairs(d, c, pairs, True, 0.8, 1.0)    # the context still works
    assert torch.equal(want[0], again[0]) and torch.equal(want[1], again[1])
    empty = ctx.match_pairs(d, c, [])                        # P = 0: a no-op
    assert empty[0].shape == (0, 257)
    for N, cap in ((5, 1), (7, 129), (3, 640), (11, 1000)):
        cnt = rng.randint(0, cap + 1, N).astype(np.int32)
        desc = _pool_random(N, cap, cnt, N * cap)
        pr = [tuple(p) for p in rng.randint(0, N, (2 * N, 2))]
        for mutual in (False, True):
            m, _ = ctx.match_pairs(torch.from_numpy(desc).cuda(), torch.from_numpy(cnt).cuda(), pr, mutual, 0.9)
            w = O.match_pairs(desc, cnt, pr, mutual, 0.9)
            sure = w["margin"] > MARGIN
            assert np.array_equal(m.cpu().numpy()[sure], w["match"][sure])
    assert ctx.check_guards() == 0
    ctx.close()


def test_cli_matching_end_to_end(tmp_path, monkeypatch):
    """The CLI on an image folder equals extract_features + match_pairs called directly; a second run changes no byte."""
    import cv2
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.data.ImageFolder import ImageFolder
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    root = tmp_path / "data" / "imgs"
    (root / "seq").mkdir(parents=True)
    for i, (h, w) in enumerate([(96, 128), (96, 128), (100, 150), (96, 128), (130, 120)]):
        img = (smooth_image(h, w, 40 + i) * 255).astype(np.uint8)
        cv2.imwrite(str(root / ("seq" if i % 2 else ".") / f"im{i}.png"), img)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(M.Path(M.__file__).parent / "configs" / "superpoint_match.yaml"))
    cfg["data"].update(name="imgs", batch_size=2, preprocessing={"resize": [96, 128]}, experiment_name="cli")
    cfg["model"]["detector_head"].update(det_thresh=0.001, top_k=200)
    cfg["matching"].update(pairs="sequential", window=3, ratio=0.9)
    cfg_path = tmp_path / "match.yaml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    M.main(config_path=str(cfg_path), random_init=True)
    out_dir = tmp_path / "exper" / "matches" / "cli"
    feats, res = np.load(out_dir / "features.npz"), np.load(out_dir / "matches.npz")
    assert feats["names"].tolist() == ["im0.png", "im2.png", "im4.png", "seq/im1.png", "seq/im3.png"]
    assert feats["shapes"].tolist() == [[96, 128], [100, 150], [130, 120], [96, 128], [96, 128]]
    assert feats["resize_geometry"].shape == (5, 4) and res["pairs"].shape == (9, 2)
    assert len(res["matches"]) > 0 and float(res["ratio"]) == 0.9 and bool(res["mutual"])

    torch.manual_seed(0)
    model = get_model(copy.deepcopy(cfg["model"]), device="cuda:0").eval()
    ds = ImageFolder(cfg["data"], device="cuda:0")
    items, kp, counts, desc = M.extract_features(model, ds, 2)
    offsets, matches, distances = M.match_pairs(desc, counts, res["pairs"].tolist(), True, 0.9, math.inf)
    assert np.array_equal(res["offsets"], offsets.cpu().numpy()) and np.array_equal(res["matches"], matches.cpu().numpy())
    assert np.array_equal(res["distances"], distances.cpu().numpy())
    cnt = counts.cpu().numpy()
    assert np.array_equal(feats["offsets"], np.r_[0, np.cumsum(cnt)])
    assert np.array_equal(feats["keypoints"], np.concatenate([kp[n, :cnt[n]].cpu().numpy() for n in range(5)]))
    before = {f.name: f.read_bytes() for f in out_dir.iterdir()}
    M.main(config_path=str(cfg_path), random_init=True)
    assert {f.name: f.read_bytes() for f in out_dir.iterdir()} == before
    cfg["data"]["preprocessing"] = None                      # without resize: 100x150 is not a multiple of 8
    cfg_path.write_text(yaml.safe_dump(cfg))
    with pytest.raises(ValueError, match=r"im2.png: size 100x150 is not a multiple of 8"):
        M.main(config_path=str(cfg_path), random_init=True)
