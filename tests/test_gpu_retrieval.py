"""spn_knn, spn_residual_sums (include/spn_retrieval.h) and retrieval.py on the GPU: neighbours against the fp64 oracle
(oracle/retrieval_oracle.py) at ragged sizes, the same d^2 bits as spn_match_pairs, bit-equal residual sums, k-means
steps, retrieval quality on planted scenes, duplicate images, argument errors, guard bands and the CLI end to end."""
import copy
import math

import numpy as np
import pytest
import torch

from conftest import SP_MODEL, smooth_image
from oracle import retrieval_oracle as R

pytestmark = pytest.mark.gpu

MARGIN = 1e-5      # orders are compared where the oracle is at least this far (in d^2) from flipping them (DESIGN.md
DIST_TOL = 1e-5    # section 4, the matcher's rule); d^2 within this everywhere


def _unit(shape, rng):
    x = rng.randn(*shape).astype(np.float32)
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def _ctx():
    from superpoint_nerf_pytorch_b200 import _native
    return _native.get_context(0)


def _check_knn(q, t, k, exclude_self, label):
    idx, d2 = _ctx().knn(torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda(), k, exclude_self)
    idx, d2 = idx.cpu().numpy(), d2.cpu().numpy()
    w_idx, w_d2, margin = R.knn(q, t, k, exclude_self)
    pad = w_idx < 0
    assert (idx[pad] == -1).all() and np.isposinf(d2[pad]).all(), label
    sure = margin > MARGIN
    assert np.array_equal(idx[sure], w_idx[sure]), label
    assert np.abs(d2[~pad].astype(np.float64) - w_d2[~pad]).max(initial=0) <= DIST_TOL, label
    assert (d2[:, 1:] >= d2[:, :-1]).all(), label                         # ascending; +inf >= +inf in the padding
    return int((~sure).sum())


def test_knn_against_the_oracle_at_ragged_sizes():
    rng = np.random.RandomState(0)
    sizes = (1, 127, 128, 129, 1000)
    excluded = 0
    for nq in sizes:
        for nt in sizes:
            q, t = _unit((nq, 64), rng), _unit((nt, 64), rng)
            for k in (1, 2, 5, 128):
                excluded += _check_knn(q, t, k, False, (nq, nt, k))
        q = _unit((nq, 128), rng)
        for k in (1, 2, 5, 128):
            excluded += _check_knn(q, q, k, True, (nq, "self", k))
    q, t = _unit((300, 1024), rng), _unit((77, 1024), rng)             # k > nt, and a longer K loop
    excluded += _check_knn(q, t, 100, False, "k > nt")
    print(f"knn: {excluded} query rows within the {MARGIN:g} margin (not compared)")


def test_knn_planted_duplicates_and_empty_train():
    rng = np.random.RandomState(1)
    q = _unit((200, 256), rng)
    t = np.concatenate([_unit((150, 256), rng), q[[7, 7, 7]], q[[2]]])
    idx, _ = _ctx().knn(torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda(), 3)
    assert idx[7].tolist() == [150, 151, 152] and idx[2, 0].item() == 153
    _check_knn(q, t, 5, False, "duplicates")
    idx, d2 = _ctx().knn(torch.from_numpy(q).cuda(), torch.zeros((0, 256), device="cuda"), 4)
    assert (idx == -1).all() and torch.isinf(d2).all()
    idx, d2 = _ctx().knn(torch.zeros((0, 256), device="cuda"), torch.from_numpy(t).cuda(), 4)
    assert idx.shape == (0, 4)


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
    with torch.no_grad():
        out = model(x, keypoints=True)
    return out["descriptor_output"]["desc_sparse"].contiguous(), out["detector_output"]["keypoint_count"].contiguous()


def test_knn_has_the_same_bits_as_match_pairs():
    rng = np.random.RandomState(2)
    random_pool = torch.from_numpy(np.stack([_unit((500, 256), rng), _unit((500, 256), rng)])).cuda()
    pools = [(random_pool, torch.tensor([500, 437], dtype=torch.int32, device="cuda")), _pool_superpoint()]
    for desc, counts in pools:
        cnt = counts.cpu().tolist()
        pairs = [(a, b) for a in range(len(cnt)) for b in range(len(cnt)) if a != b]
        match, dist = _ctx().match_pairs(desc, counts, pairs, False, 0.0, math.inf)
        for p, (a, b) in enumerate(pairs):
            idx, d2 = _ctx().knn(desc[a, :cnt[a]], desc[b, :cnt[b]], 2)
            assert torch.equal(idx[:, 0], match[p, :cnt[a]]), (a, b)
            assert np.array_equal(np.sqrt(d2[:, 0].cpu().numpy()).view(np.int32), dist[p, :cnt[a]].cpu().numpy().view(np.int32))


def test_residual_sums_are_bit_equal_to_the_oracle():
    rng = np.random.RandomState(3)
    for N, cap, C, K in ((5, 300, 256, 64), (3, 1, 64, 1), (4, 700, 320, 37), (2, 40, 256, 256)):
        desc = rng.randn(N, cap, C).astype(np.float32)
        counts = rng.randint(0, cap + 1, N).astype(np.int32)
        counts[0] = cap + 5                                          # above cap: clamped
        if N > 2:
            counts[1] = 0
        assign = rng.randint(-1, K + 1, (N, cap)).astype(np.int32)  # -1 and K are skipped
        assign[:, ::7] = 0                                           # a crowded word ...
        assign[assign == K // 2] = K                                 # ... and one with no members
        words = rng.randn(K, C).astype(np.float32)
        sums, n = _ctx().residual_sums(*(torch.from_numpy(x).cuda() for x in (desc, counts, assign, words)))
        w_sums, w_n = R.residual_sums(desc, counts, assign, words)
        assert np.array_equal(sums.cpu().numpy(), w_sums), (N, cap, C, K)
        assert np.array_equal(n.cpu().numpy(), w_n), (N, cap, C, K)


def _valid_rows(desc, counts):
    cap = desc.shape[1]
    return np.arange(cap)[None] < np.clip(counts, 0, cap)[:, None]


def test_kmeans_steps_against_the_oracle():
    from superpoint_nerf_pytorch_b200 import retrieval
    rng = np.random.RandomState(4)
    N, cap, C, K, iters = 12, 400, 256, 32, 6
    centres = _unit((20, C), rng)
    desc = np.zeros((N, cap, C), np.float32)
    counts = rng.randint(50, cap + 1, N).astype(np.int32)
    for n in range(N):
        x = centres[rng.randint(0, 20, cap)] + 0.05 * rng.randn(cap, C).astype(np.float32)
        desc[n, :counts[n]] = (x / np.linalg.norm(x, axis=1, keepdims=True))[:counts[n]]
    d, c = torch.from_numpy(desc).cuda(), torch.from_numpy(counts).cuda()
    valid = _valid_rows(desc, counts)
    flat = desc[valid]
    words = [flat[np.random.RandomState(0).choice(len(flat), K, replace=False)]]     # the draw of iteration 0
    words += [retrieval.kmeans(d, c, K, t).cpu().numpy() for t in range(1, iters + 1)]
    excluded, objective = 0, []
    for t in range(iters):
        assign = retrieval.assign_words(d, c, torch.from_numpy(words[t]).cuda()).cpu().numpy()
        assert (assign[~valid] == -1).all()
        w_idx, _, margin = R.knn(flat, words[t], 1)
        sure = margin > MARGIN
        assert np.array_equal(assign[valid][sure], w_idx[sure, 0]), t
        excluded += int((~sure).sum())
        want = R.kmeans_step(desc, counts, assign, words[t])
        assert np.abs(words[t + 1] - want).max() <= 1e-6, t
        objective.append(R.objective(desc, counts, assign, words[t]))
    for a, b in zip(objective, objective[1:]):
        assert b <= a * (1 + 1e-6), objective
    assert np.array_equal(retrieval.kmeans(d, c, K, iters).cpu().numpy(), words[iters])   # run to run
    print(f"kmeans: objective {objective[0]:.2f} -> {objective[-1]:.2f}, {excluded} assignments within the margin")
    with pytest.raises(ValueError, match="retrieval.vocab_size"):
        retrieval.kmeans(d, torch.full_like(c, 1), 13, 1)


def _planted_scenes(seed, S=8, V=4, L=400, keep=300, distractors=50, C=256, sigma=0.1):
    """S scenes of L random unit landmarks; each of V views holds `keep` of its scene's landmarks with noise and
    `distractors` random unit rows.  sigma is the noise's scale relative to the unit-norm descriptor (per-component
    standard deviation sigma / sqrt(C), so the noise vector has norm ~sigma) before re-normalisation."""
    rng = np.random.RandomState(seed)
    desc = np.zeros((S * V, keep + distractors, C), np.float32)
    for s in range(S):
        landmarks = _unit((L, C), rng)
        for v in range(V):
            x = landmarks[rng.choice(L, keep, replace=False)] + sigma / math.sqrt(C) * rng.randn(keep, C).astype(np.float32)
            rows = np.concatenate([x / np.linalg.norm(x, axis=1, keepdims=True), _unit((distractors, C), rng)])
            desc[s * V + v] = rows[rng.permutation(len(rows))]
    return desc


def test_retrieval_finds_the_views_of_a_scene():
    from superpoint_nerf_pytorch_b200 import retrieval
    S, V = 8, 4
    desc = torch.from_numpy(_planted_scenes(5, S, V)).cuda()
    counts = torch.full((S * V,), desc.shape[1], dtype=torch.int32, device="cuda")
    words = retrieval.kmeans(desc, counts, 64, 20)
    vec = retrieval.vlad(desc, counts, words)
    assert torch.allclose(vec.norm(dim=1), torch.ones(S * V, device="cuda"), atol=1e-5)
    index, dist2 = retrieval.neighbors(vec, counts, V - 1)
    scene = np.arange(S * V) // V
    precision = float((scene[index.cpu().numpy()] == scene[:, None]).mean())
    print(f"mean precision@{V - 1} of same-scene neighbours: {precision:.4f} (chance {(V - 1) / (S * V - 1):.3f})")
    assert precision >= 0.95
    # a different view of the same collection with two images emptied: their rows are -1, nobody pairs with them
    counts[[3, 17]] = 0
    vec = retrieval.vlad(desc, counts, words)
    assert (vec[[3, 17]] == 0).all()
    index, dist2 = retrieval.neighbors(vec, counts, 30)
    idx = index.cpu().numpy()
    assert (idx[[3, 17]] == -1).all() and torch.isinf(dist2[[3, 17]]).all()
    assert not np.isin(idx, [3, 17]).any() and (idx[0, 29:] == -1).all() and (idx[0, :29] >= 0).all()


def test_duplicate_images_are_each_others_first_neighbour():
    from superpoint_nerf_pytorch_b200 import retrieval
    desc, counts = _pool_superpoint()
    assert counts.min().item() > 20
    words = retrieval.kmeans(desc, counts, 16, 5)
    vec = retrieval.vlad(desc, counts, words)
    assert torch.equal(vec[0], vec[1])
    index, _ = retrieval.neighbors(vec, counts, 2)
    assert index[0, 0].item() == 1 and index[1, 0].item() == 0


def test_errors_and_guard_bands():
    import superpoint_nerf_pytorch_b200 as P
    ctx = P.Context(0)
    rng = np.random.RandomState(6)
    q = torch.from_numpy(_unit((300, 256), rng)).cuda()
    want = ctx.knn(q, q[:100], 5)
    for args, msg in (((q, q[:100], 0), r"k = 0 outside \[1, 128\]"), ((q, q[:100], 129), "k = 129"),
                      ((q, q[:100], 5, True), "exclude_self needs the same set")):
        with pytest.raises(P.NativeError, match=msg):
            ctx.knn(*args)
    with pytest.raises(P.NativeError, match="multiple of 64"):
        ctx.knn(q[:, :100].contiguous(), q[:, :100].contiguous(), 2)
    with pytest.raises(P.NativeError, match="must be"):
        ctx.knn(q.double(), q, 2)
    with pytest.raises(P.NativeError, match="same C"):
        ctx.knn(q, q[:, :128].contiguous(), 2)
    with pytest.raises(P.NativeError, match="do not fit together"):
        ctx.residual_sums(q.view(3, 100, 256), torch.zeros(3, dtype=torch.int32, device="cuda"),
                          torch.zeros((3, 99), dtype=torch.int32, device="cuda"), q[:4])
    again = ctx.knn(q, q[:100], 5)                                   # the context still works
    assert torch.equal(want[0], again[0]) and torch.equal(want[1], again[1])
    for nq, nt, C, k in ((1, 1, 64, 1), (129, 257, 128, 7), (1000, 33, 256, 128), (257, 257, 64, 128)):
        a, b = torch.from_numpy(_unit((nq, C), rng)).cuda(), torch.from_numpy(_unit((nt, C), rng)).cuda()
        ctx.knn(a, b, k)
        ctx.knn(b, b, k, exclude_self=True)
    for N, cap, C, K in ((1, 1, 1, 1), (7, 129, 300, 33), (3, 1000, 256, 256)):
        desc = torch.randn((N, cap, C), device="cuda")
        counts = torch.randint(0, cap + 2, (N,), dtype=torch.int32, device="cuda")
        assign = torch.randint(-2, K + 2, (N, cap), dtype=torch.int32, device="cuda")
        ctx.residual_sums(desc, counts, assign, torch.randn((K, C), device="cuda"))
    assert ctx.check_guards() == 0
    ctx.close()


def test_cli_retrieval_end_to_end(tmp_path, monkeypatch):
    """The CLI in retrieval mode equals extract_features -> kmeans -> vlad -> neighbors -> retrieval_pairs ->
    match_pairs called directly; a second run changes no byte; a loaded vocabulary reproduces the words and pairs;
    num_neighbors >= N - 1 gives the exhaustive run's matches."""
    import cv2
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import retrieval, settings
    from superpoint_nerf_pytorch_b200.data.ImageFolder import ImageFolder
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    root = tmp_path / "data" / "imgs"
    root.mkdir(parents=True)
    for i in range(7):
        img = (smooth_image(96, 128, 60 + i % 6) * 255).astype(np.uint8)     # im6 repeats im0
        cv2.imwrite(str(root / f"im{i}.png"), img)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(M.Path(M.__file__).parent / "configs" / "superpoint_match_retrieval.yaml"))
    cfg["data"].update(name="imgs", batch_size=3, preprocessing={"resize": [96, 128]}, experiment_name="ret")
    cfg["model"]["detector_head"].update(det_thresh=0.001, top_k=200)
    cfg["matching"].update(ratio=0.9)
    cfg["retrieval"].update(num_neighbors=2, vocab_size=8, kmeans_iters=4)

    def run(name, **retrieval_block):
        c = copy.deepcopy(cfg)
        c["data"]["experiment_name"] = name
        c["retrieval"] = retrieval_block if retrieval_block else c["retrieval"]
        path = tmp_path / f"{name}.yaml"
        path.write_text(yaml.safe_dump(c))
        M.main(config_path=str(path), random_init=True)
        out = tmp_path / "exper" / "matches" / name
        return out, {f.name: np.load(f) for f in out.iterdir()}

    out_dir, files = run("ret")
    assert sorted(files) == ["features.npz", "matches.npz", "retrieval.npz"]
    ret, res, feats = files["retrieval.npz"], files["matches.npz"], files["features.npz"]
    assert ret["words"].shape == (8, 256) and ret["words"].dtype == np.float32 and ret["neighbors"].shape == (7, 2)
    assert int(ret["num_neighbors"]) == 2 and int(ret["kmeans_iters"]) == 4
    assert ret["neighbors"][0, 0] == 6 and ret["neighbors"][6, 0] == 0          # the repeated image

    torch.manual_seed(0)
    model = get_model(copy.deepcopy(cfg["model"]), device="cuda:0").eval()
    ds = ImageFolder(cfg["data"], device="cuda:0")
    items, kp, counts, desc = M.extract_features(model, ds, 3)
    words = retrieval.kmeans(desc, counts, 8, 4)
    index, dist2 = retrieval.neighbors(retrieval.vlad(desc, counts, words), counts, 2)
    pairs = retrieval.retrieval_pairs(index)
    offsets, matches, distances = M.match_pairs(desc, counts, pairs, True, 0.9, math.inf)
    assert np.array_equal(ret["words"], words.cpu().numpy()) and np.array_equal(ret["neighbors"], index.cpu().numpy())
    assert np.array_equal(ret["dist2"], dist2.cpu().numpy()) and res["pairs"].tolist() == [list(p) for p in pairs]
    assert np.array_equal(res["offsets"], offsets.cpu().numpy()) and np.array_equal(res["matches"], matches.cpu().numpy())
    assert np.array_equal(res["distances"], distances.cpu().numpy())
    assert np.array_equal(feats["offsets"], np.r_[0, np.cumsum(counts.cpu().numpy())])

    before = {f.name: f.read_bytes() for f in out_dir.iterdir()}
    run("ret")
    assert {f.name: f.read_bytes() for f in out_dir.iterdir()} == before

    _, loaded = run("vocab", num_neighbors=2, vocabulary=str(out_dir / "retrieval.npz"))
    assert np.array_equal(loaded["retrieval.npz"]["words"], ret["words"]) and int(loaded["retrieval.npz"]["kmeans_iters"]) == -1
    assert np.array_equal(loaded["matches.npz"]["pairs"], res["pairs"])

    _, wide = run("wide", num_neighbors=6, vocab_size=8, kmeans_iters=4)
    c = copy.deepcopy(cfg)
    c["matching"]["pairs"] = "exhaustive"
    c["data"]["experiment_name"] = "exh"
    path = tmp_path / "exh.yaml"
    path.write_text(yaml.safe_dump(c))
    M.main(config_path=str(path), random_init=True)
    exh_dir = tmp_path / "exper" / "matches" / "exh"
    assert sorted(f.name for f in exh_dir.iterdir()) == ["features.npz", "matches.npz"]
    exh = np.load(exh_dir / "matches.npz")
    for key in ("pairs", "offsets", "matches", "distances"):
        assert np.array_equal(wide["matches.npz"][key], exh[key]), key
