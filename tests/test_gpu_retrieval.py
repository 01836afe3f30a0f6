"""spn_knn, spn_residual_sums (include/spn_retrieval.h) and retrieval.py on the GPU: neighbours against the fp64 oracle
(oracle/retrieval_oracle.py) at ragged sizes, at the VLAD widths of retrieval (D up to 65 536) on random rows, on
near-duplicate ladders and on VLAD vectors of planted scenes, the same d^2 bits as spn_match_pairs and
spn_mutual_nn_match at every width, bit-equal residual sums, k-means steps, retrieval quality on planted scenes,
duplicate images, argument errors, guard bands and the CLI end to end."""
import copy
import math

import numpy as np
import pytest
import torch

from conftest import SP_MODEL, smooth_image
from oracle import retrieval_oracle as R
from retrieval_scenes import planted_scenes as _planted_scenes
from retrieval_scenes import unit as _unit

pytestmark = pytest.mark.gpu

MARGIN = 1e-5      # orders are compared where the oracle is at least this far (in d^2) from flipping them (DESIGN.md
DIST_TOL = 1e-5    # section 4, the matcher's rule); d^2 within this everywhere


def _ctx():
    from superpoint_nerf_pytorch_b200 import _native
    return _native.get_context(0)


def _pair_d2(q, t, idx):
    """fp64 d^2 of query row i and train row idx[i, s] (idx >= 0)."""
    q, t = q.astype(np.float64), t.astype(np.float64)
    d = (q * q).sum(1)[:, None] + (t * t).sum(1)[None, :] - 2.0 * (q @ t.T)
    return np.maximum(d, 0.0)[np.arange(len(q))[:, None], np.maximum(idx, 0)]


def _check_knn(q, t, k, exclude_self, label, got=None):
    """spn_knn(q, t, k) (or `got` = its (index, dist2) from elsewhere) against the oracle.  -> (queries within the
    margin, largest |d^2 - fp64 d^2 of the returned pair|)."""
    idx, d2 = got if got is not None else _ctx().knn(torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda(), k, exclude_self)
    idx, d2 = idx.cpu().numpy(), d2.cpu().numpy()
    w_idx, w_d2, margin = R.knn(q, t, k, exclude_self)
    pad = w_idx < 0
    assert (idx[pad] == -1).all() and np.isposinf(d2[pad]).all(), label
    sure = margin > MARGIN
    assert np.array_equal(idx[sure], w_idx[sure]), label
    assert np.abs(d2[~pad].astype(np.float64) - w_d2[~pad]).max(initial=0) <= DIST_TOL, label
    err = np.abs(d2[~pad].astype(np.float64) - _pair_d2(q, t, idx)[~pad]).max(initial=0)
    assert err <= DIST_TOL, label                                          # also right for the row it names
    assert (d2[:, 1:] >= d2[:, :-1]).all(), label                         # ascending; +inf >= +inf in the padding
    return int((~sure).sum()), float(err)


def test_knn_against_the_oracle_at_ragged_sizes():
    rng = np.random.RandomState(0)
    sizes = (1, 127, 128, 129, 1000)
    excluded = 0
    for nq in sizes:
        for nt in sizes:
            q, t = _unit((nq, 64), rng), _unit((nt, 64), rng)
            for k in (1, 2, 5, 128):
                excluded += _check_knn(q, t, k, False, (nq, nt, k))[0]
        q = _unit((nq, 128), rng)
        for k in (1, 2, 5, 128):
            excluded += _check_knn(q, q, k, True, (nq, "self", k))[0]
    q, t = _unit((300, 1024), rng), _unit((77, 1024), rng)             # k > nt, and a longer K loop
    excluded += _check_knn(q, t, 100, False, "k > nt")[0]
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


def test_knn_against_the_oracle_at_vlad_widths():
    """Random unit rows at the widths retrieval runs spn_knn on (D = vocab_size x 256), ragged nq / nt, k up to 128.
    Random rows at large D have d^2 = 2 +- 2 / sqrt(D), so among a few hundred rows adjacent ranks are often closer
    than the margin: for k > 1 most queries fall within it by construction of the input.  The d^2 bound holds on every
    entry, and with k = 1 fewer than 1 % of the queries may fall within the margin."""
    rng = np.random.RandomState(7)
    first = first_total = 0
    for D in (4096, 16384, 65536):
        pool = _unit((512, D), rng)
        excluded, total, worst = {}, {}, 0.0
        for k in (1, 20, 128):
            cases = [(pool[:nq], pool[-nt:], False, (D, nq, nt, k)) for nq, nt in ((1, 300), (127, 129), (129, 1), (300, 127))]
            cases += [(pool[:n], pool[:n], True, (D, n, "self", k)) for n in (1, 129, 300)]
            for q, t, self_, label in cases:
                ex, err = _check_knn(q, t, k, self_, label)
                excluded[k] = excluded.get(k, 0) + ex
                total[k] = total.get(k, 0) + len(q)
                worst = max(worst, err)
        first, first_total = first + excluded[1], first_total + total[1]
        print(f"knn D={D}: largest d^2 error {worst:.2e}; queries within the {MARGIN:g} margin (not compared) "
              + ", ".join(f"k={k}: {excluded[k]} of {total[k]}" for k in excluded))
    assert first < 0.01 * first_total, (first, first_total)


def _ladder(D, nq, rng, rungs=40, copies=2, others=50):
    """nq unit queries and a train set holding, per query, `copies` exact copies of it, rungs normalise(q + eps n) with
    eps from 1e-4 to 1 (true d^2 ~1e-8 to ~0.6, n a random unit row) and `others` random unit rows.  -> q, t, the
    train indices of the copies (nq, copies)."""
    q = _unit((nq, D), rng)
    eps = np.logspace(-4, 0, rungs)
    blocks, copy_idx = [], []
    for i in range(nq):
        near = q[i] + eps[:, None].astype(np.float32) * _unit((rungs, D), rng)
        near /= np.linalg.norm(near, axis=1, keepdims=True)
        start = sum(len(b) for b in blocks)
        copy_idx.append(start + np.arange(copies))
        blocks.append(np.concatenate([np.repeat(q[i:i + 1], copies, 0), near, _unit((others, D), rng)]))
    return q, np.concatenate(blocks).astype(np.float32), np.array(copy_idx)


@pytest.mark.parametrize("D", [256, 1024, 4096, 16384, 65536])
def test_knn_near_duplicate_ladder(D):
    """True d^2 from 0 to ~2 at one width: d^2 within 1e-5 of fp64 at every rank, and the d^2 of an exact copy of the
    query, which is the accumulation error of the dot product alone (|q|^2 = |t|^2 bit for bit)."""
    rng = np.random.RandomState(D)
    q, t, copy_idx = _ladder(D, 4, rng)
    k = 128
    idx, d2 = _ctx().knn(torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda(), k)
    ex, err = _check_knn(q, t, k, False, ("ladder", D), got=(idx, d2))
    idx, d2 = idx.cpu().numpy(), d2.cpu().numpy()
    copy_d2 = []
    for i in range(len(q)):
        at = np.isin(idx[i], copy_idx[i])
        assert at.sum() == copy_idx.shape[1], (D, i)                       # every copy is among the k nearest ...
        assert len(set(d2[i, at].view(np.int32).tolist())) == 1, (D, i)   # ... with one d^2: identical rows, identical bits
        copy_d2.append(float(d2[i, at][0]))
    assert max(copy_d2) <= DIST_TOL
    print(f"ladder D={D}: largest d^2 error {err:.2e}, exact-copy d^2 {max(copy_d2):.2e} (of {len(q)} queries), "
          f"{ex} of {len(q)} queries within the {MARGIN:g} margin (the rungs below 1e-5 are, by design)")


def test_knn_on_vlad_vectors_of_planted_scenes():
    """spn_knn on intra-normalised VLAD vectors as retrieval makes them (k-means and VLAD on the GPU, 128 scenes x 4
    views, D = 16 384 and 65 536) against the fp64 oracle on the same fp32 vectors, through retrieval.neighbors, with
    two images without keypoints.  k = 3 is the other views of the scene: fewer than 1 % of the queries may fall within
    the margin.  k = 20 adds views of other scenes, whose d^2 to the query crowd near 2."""
    from superpoint_nerf_pytorch_b200 import retrieval
    S, V = 128, 4
    desc = torch.from_numpy(_planted_scenes(7, S, V)).cuda()
    counts = torch.full((S * V,), desc.shape[1], dtype=torch.int32, device="cuda")
    counts[[5, 300]] = 0
    has = torch.nonzero(counts > 0).view(-1)
    has_np = has.cpu().numpy()
    for K in (64, 256):
        words = retrieval.kmeans(desc, counts, K, 5)
        vec = retrieval.vlad(desc, counts, words)
        assert vec.shape == (S * V, K * 256) and (vec[[5, 300]] == 0).all()
        v = vec[has].cpu().numpy()
        for k in (V - 1, 20):
            index, dist2 = retrieval.neighbors(vec, counts, k)
            assert (index[[5, 300]] == -1).all() and torch.isinf(dist2[[5, 300]]).all()
            local = torch.from_numpy(np.searchsorted(has_np, np.maximum(index[has].cpu().numpy(), 0))).to(torch.int32)
            local = torch.where(index[has].cpu() >= 0, local, -1)                        # image ids -> rows of v
            ex, err = _check_knn(v, v, k, True, ("vlad", K, k), got=(local, dist2[has].cpu()))
            print(f"vlad D={K * 256} k={k}: largest d^2 error {err:.2e}, {ex} of {len(v)} queries within the "
                  f"{MARGIN:g} margin (not compared)")
            if k == V - 1:
                assert ex < 0.01 * len(v), ex


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


def _near_copy_pool(C, rng):
    """Two random unit sets of 500 rows at width C, the second holding near-copies (noise 0.01) of 63 rows of the
    first, so that dot products near 1 go through every chunk of the tile; counts 500 and 470."""
    xa = _unit((500, C), rng)
    xb = np.concatenate([_unit((437, C), rng), xa[:63] + 0.01 * _unit((63, C), rng)])
    pool = torch.from_numpy(np.stack([xa, xb / np.linalg.norm(xb, axis=1, keepdims=True)])).cuda()
    return pool, torch.tensor([500, 470], dtype=torch.int32, device="cuda")


def test_knn_has_the_same_bits_as_match_pairs():
    """The three consumers of nn_tc.cuh's distance tile give the same d^2 bits at every width, from one chunk (C <= 256)
    to 64 chunks: knn's first neighbour and sqrtf of its d^2 equal match_pairs' match and distance, and match_pairs
    with the mutual check only equals spn_mutual_nn_match."""
    rng = np.random.RandomState(2)
    random_pool = torch.from_numpy(np.stack([_unit((500, 256), rng), _unit((500, 256), rng)])).cuda()
    pools = [(256, random_pool, torch.tensor([500, 437], dtype=torch.int32, device="cuda")), (256, *_pool_superpoint())]
    pools += [(C, *_near_copy_pool(C, rng)) for C in (64, 128, 256, 1024, 16384)]
    for C, desc, counts in pools:
        cnt = counts.cpu().tolist()
        pairs = [(a, b) for a in range(len(cnt)) for b in range(len(cnt)) if a != b]
        match, dist = _ctx().match_pairs(desc, counts, pairs, False, 0.0, math.inf)
        for p, (a, b) in enumerate(pairs):
            idx, d2 = _ctx().knn(desc[a, :cnt[a]], desc[b, :cnt[b]], 2)
            assert torch.equal(idx[:, 0], match[p, :cnt[a]]), (C, a, b)
            assert np.array_equal(np.sqrt(d2[:, 0].cpu().numpy()).view(np.int32), dist[p, :cnt[a]].cpu().numpy().view(np.int32))
        pairs = [(a, b) for a in range(len(cnt)) for b in range(len(cnt))]
        m, dist = _ctx().match_pairs(desc, counts, pairs, True, 0.0, math.inf)
        ia = torch.tensor([a for a, _ in pairs], device="cuda")
        ib = torch.tensor([b for _, b in pairs], device="cuda")
        m_ref, d_ref = _ctx().mutual_nn_match(desc.index_select(0, ia), counts.index_select(0, ia),
                                              desc.index_select(0, ib), counts.index_select(0, ib))
        assert torch.equal(m, m_ref) and torch.equal(dist, d_ref), C


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
