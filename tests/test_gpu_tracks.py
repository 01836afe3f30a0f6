"""spn_track_labels / spn_track_table (include/spn_tracks.h) and tracks.py on the GPU: every output array-equal to the
oracle (oracle/tracks_oracle.py) on random graphs, ragged images and the deepest chain; invariance to the order and
split of the edges; planted multi-view scenes; bad input and guard bands; the matching CLI end to end."""
import copy

import numpy as np
import pytest
import torch

from conftest import smooth_image
from oracle import tracks_oracle as T
from track_scenes import planted

pytestmark = pytest.mark.gpu


def _ctx():
    from superpoint_nerf_pytorch_b200 import _native
    return _native.get_context(0)


def _ragged(rng, K, N):
    """N images holding K keypoints between them, some of them without keypoints."""
    counts = rng.multinomial(K, np.full(N, 1.0 / N)) if N > 1 else np.array([K])
    if N > 3:
        empty = rng.choice(N, N // 4, replace=False)
        moved = counts[empty].sum()
        counts[empty] = 0
        counts[np.setdiff1d(np.arange(N), empty)[0]] += moved
    return counts.astype(np.int64)


def _gpu(edges, K, img_off, min_length=2, splits=1):
    """The two C entry points -> (labels, track_offsets, observations, consistent, track_of) as numpy."""
    ctx = _ctx()
    d = torch.from_numpy(np.ascontiguousarray(edges, dtype=np.int32).reshape(-1, 2)).cuda()
    labels = None
    for part in torch.tensor_split(d, splits):
        labels, bad = ctx.track_labels(part.contiguous(), K, labels)
        assert bad.item() == 0
    off, obs, cons, tof, totals, bad = ctx.track_table(labels, torch.from_numpy(np.asarray(img_off, np.int64)).cuda(), min_length)
    n_t, n_o = totals.tolist()
    assert bad.item() == 0
    return (labels.cpu().numpy(), off[:n_t + 1].cpu().numpy(), obs[:n_o].cpu().numpy(), cons[:n_t].cpu().numpy().astype(bool),
            tof.cpu().numpy())


def _oracle(edges, K, img_off, min_length=2):
    lab = T.labels(edges, K)
    return (lab, *T.tracks(lab, img_off, min_length))


def _equal(got, want, label=""):
    names = ("labels", "track_offsets", "observations", "consistent", "track_of")
    for name, g, w in zip(names, got, want):
        assert g.shape == w.shape and np.array_equal(g, w), (label, name, g.shape, w.shape)


# ---------------------------------------------------------------------------------------------------------- oracle
def test_random_graphs_equal_the_oracle():
    rng = np.random.RandomState(1)
    for K in (1, 2, 1000, 10 ** 5, 10 ** 6):
        for density in (0.0, 0.2, 0.5, 1.0, 3.0):              # sparse ... one giant component
            E = int(density * K) + (1 if K <= 2 else 0)
            edges = rng.randint(0, K, (E, 2))
            N = max(1, K // 500)
            img_off = np.r_[0, np.cumsum(_ragged(rng, K, N))]
            for min_length in (2, 3):
                _equal(_gpu(edges, K, img_off, min_length), _oracle(edges, K, img_off, min_length), (K, density, min_length))
    # image-local structure: edges inside a window of rows, so many images hold two keypoints of one track
    K = 20000
    img_off = np.r_[0, np.cumsum(_ragged(rng, K, 400))]
    u = rng.randint(0, K - 40, 15000)
    edges = np.c_[u, u + rng.randint(0, 40, len(u))]
    got = _gpu(edges, K, img_off)
    _equal(got, _oracle(edges, K, img_off), "local")
    assert got[3].any() and not got[3].all()


def test_empty_duplicate_and_self_loop_edges():
    K, img_off = 1000, np.r_[0, np.cumsum([300, 0, 500, 200])]
    got = _gpu(np.zeros((0, 2)), K, img_off)                    # E = 0: all singletons, no tracks
    assert np.array_equal(got[0], np.arange(K)) and got[1].tolist() == [0] and got[2].shape == (0, 2) and (got[4] == -1).all()
    loops = np.c_[np.arange(K), np.arange(K)]
    _equal(_gpu(loops, K, img_off), got, "self-loops")
    rng = np.random.RandomState(2)
    edges = rng.randint(0, K, (300, 2))
    dup = np.r_[edges, edges, edges[:, ::-1], loops[:50]]
    _equal(_gpu(dup, K, img_off), _gpu(edges, K, img_off), "duplicates")
    _equal(_gpu(dup, K, img_off), _oracle(dup, K, img_off), "duplicates vs oracle")


def test_descending_chain_of_a_million_rows():
    K = 10 ** 6
    r = np.arange(K - 2, -1, -1)
    edges = np.c_[r, r + 1]                                      # (K-2, K-1), ..., (0, 1): the deepest forest
    img_off = np.arange(K + 1)                                   # one keypoint per image: one consistent track
    got = _gpu(edges, K, img_off)
    assert (got[0] == 0).all() and got[1].tolist() == [0, K] and got[3].tolist() == [True]
    _equal(got, _oracle(edges, K, img_off), "chain")
    img_off = np.r_[np.arange(0, K, 2), K]                       # two keypoints per image: inconsistent
    assert _gpu(edges, K, img_off)[3].tolist() == [False]


def test_order_and_split_invariance():
    rng = np.random.RandomState(3)
    K = 200000
    img_off = np.r_[0, np.cumsum(_ragged(rng, K, 300))]
    edges = rng.randint(0, K, (180000, 2))
    first = _gpu(edges, K, img_off)
    _equal(_gpu(edges, K, img_off), first, "again")
    _equal(_gpu(edges[rng.permutation(len(edges))], K, img_off), first, "permuted")
    _equal(_gpu(edges[:, ::-1], K, img_off), first, "swapped endpoints")
    for splits in (2, 7):
        _equal(_gpu(edges, K, img_off, splits=splits), first, f"{splits} launches")
    _equal(_gpu(edges[rng.permutation(len(edges))], K, img_off, splits=5), first, "permuted, 5 launches")
    _equal(first, _oracle(edges, K, img_off), "oracle")


# ---------------------------------------------------------------------------------------------------------- scenes
def _build(counts, pairs, offsets, matches, keep=None, min_length=2):
    from superpoint_nerf_pytorch_b200 import tracks
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()   # noqa: E731
    out = tracks.build_tracks(d(counts), pairs, d(offsets), d(matches), None if keep is None else d(keep), min_length)
    return [x.cpu().numpy() for x in out]


def _same_as_oracle(got, want, label):
    for name, g, w in zip(("track_offsets", "observations", "consistent", "track_of"), got, want):
        assert g.shape == w.shape and np.array_equal(g, w), (label, name)


def test_planted_scenes():
    rng = np.random.RandomState(4)
    # no outliers: the tracks are exactly the landmarks seen at least twice, all consistent
    counts, pairs, offsets, matches, land = planted(rng)
    got = _build(counts, pairs, offsets, matches)
    _same_as_oracle(got, T.build_tracks(counts, pairs, offsets, matches)[:4], "clean")
    t_off, obs, cons, tof = got
    img_off = np.r_[0, np.cumsum(counts)]
    rows = img_off[obs[:, 0]] + obs[:, 1]
    seen_twice = np.nonzero(np.bincount(land[land >= 0], minlength=400) >= 2)[0]
    assert len(cons) == len(seen_twice) and cons.all()
    for t in range(len(cons)):
        lm = land[rows[t_off[t]:t_off[t + 1]]]
        assert (lm == lm[0]).all() and lm[0] >= 0 and len(lm) == (land == lm[0]).sum()
    # chance outliers between distractors: every landmark track is still its landmark
    counts, pairs, offsets, matches, land = planted(rng, outliers=3)
    got = _build(counts, pairs, offsets, matches)
    _same_as_oracle(got, T.build_tracks(counts, pairs, offsets, matches)[:4], "outliers")
    t_off, obs, cons, tof = got
    img_off = np.r_[0, np.cumsum(counts)]
    for lm in np.nonzero(np.bincount(land[land >= 0], minlength=400) >= 2)[0]:
        members = np.nonzero(land == lm)[0]
        t = tof[members[0]]
        assert t >= 0 and (tof[members] == t).all() and t_off[t + 1] - t_off[t] == len(members) and cons[t]
    # outliers that join two keypoints of one image: those tracks are flagged, everything else equals the oracle
    counts, pairs, offsets, matches, land = planted(rng, outliers=2, clashes=12)
    got = _build(counts, pairs, offsets, matches)
    _same_as_oracle(got, T.build_tracks(counts, pairs, offsets, matches)[:4], "clashes")
    t_off, obs, cons, tof = got
    assert (~cons).sum() >= 1
    for t in np.nonzero(~cons)[0]:
        img = obs[t_off[t]:t_off[t + 1], 0]
        assert (np.diff(img) == 0).any() and (land[(np.r_[0, np.cumsum(counts)][img] + obs[t_off[t]:t_off[t + 1], 1])] < 0).any()
    # keep masks: all false gives no tracks; a random mask equals the oracle; a permuted pair list changes nothing
    keep = np.zeros(len(matches), bool)
    t_off, obs, cons, tof = _build(counts, pairs, offsets, matches, keep)
    assert t_off.tolist() == [0] and obs.shape == (0, 2) and cons.shape == (0,) and (tof == -1).all() and len(tof) == counts.sum()
    keep = rng.rand(len(matches)) < 0.7
    _same_as_oracle(_build(counts, pairs, offsets, matches, keep, 3), T.build_tracks(counts, pairs, offsets, matches, keep, 3)[:4],
                    "keep")
    perm = rng.permutation(len(pairs))
    seg = [matches[offsets[p]:offsets[p + 1]] for p in perm]
    off_p = np.r_[0, np.cumsum([len(s) for s in seg])].astype(np.int64)
    base = _build(counts, pairs, offsets, matches)
    for x, y in zip(_build(counts, pairs[perm], off_p, np.concatenate(seg)), base):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------------------------------------------------- errors
def test_bad_input_and_guard_bands():
    import superpoint_nerf_pytorch_b200 as P
    from superpoint_nerf_pytorch_b200 import tracks
    rng = np.random.RandomState(5)
    counts, pairs, offsets, matches, _ = planted(rng, n_images=6, n_land=100, outliers=2)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()   # noqa: E731
    for col, value in ((0, None), (1, None), (0, -1)):
        bad = matches.copy()
        p = 4
        a, b = pairs[p]
        bad[offsets[p] + 1, col] = value if value is not None else counts[a if col == 0 else b]
        with pytest.raises(ValueError, match="keypoint index outside"):
            tracks.build_tracks(d(counts), pairs, d(offsets), d(bad))
    with pytest.raises(ValueError, match="offsets"):
        tracks.build_tracks(d(counts), pairs, d(offsets[:-1]), d(matches))
    with pytest.raises(ValueError, match="min_length"):
        tracks.build_tracks(d(counts), pairs, d(offsets), d(matches), min_length=1)
    ctx = P.Context(0)
    K = 5000
    img_off = d(np.r_[0, np.cumsum(_ragged(rng, K, 20))])
    edges = rng.randint(0, K, (4000, 2))
    want, _ = ctx.track_labels(d(edges.astype(np.int32)), K)
    # out-of-range edges are counted and not applied
    wild = np.r_[edges, [[K, 0], [-1, 3], [7, K + 100], [2 ** 31 - 1, 5]]][rng.permutation(len(edges) + 4)]
    got, bad = ctx.track_labels(d(wild.astype(np.int32)), K)
    assert bad.item() == 4 and torch.equal(got, want)
    # resumed labels outside [0, r] are counted and reset; a label that does not point at a root is counted by the table
    lab = torch.arange(K, dtype=torch.int32, device="cuda")
    lab[10], lab[20] = 11, -4
    got, bad = ctx.track_labels(d(np.zeros((0, 2), np.int32)), K, lab)
    assert bad.item() == 2 and got[10].item() == 10 and got[20].item() == 20
    lab = want.clone()
    lab[K - 1] = int(torch.nonzero(want != torch.arange(K, device="cuda"))[0, 0])    # a row that is not a root
    assert ctx.track_table(lab, img_off, 2)[5].item() == 1
    out = ctx.track_table(want, d(np.r_[0, K - 10]), 2)             # offsets that do not end at K
    assert out[5].item() == 1
    with pytest.raises(P.NativeError, match="min_length"):
        ctx.track_table(want, img_off, 1)
    with pytest.raises(P.NativeError, match="edges must be"):
        ctx.track_labels(d(np.zeros((4, 3), np.int32)), K)
    with pytest.raises(P.NativeError, match="K = 0"):
        ctx.track_labels(d(edges.astype(np.int32)), 0)
    assert ctx.check_guards() == 0
    ctx.close()


# ---------------------------------------------------------------------------------------------------------- CLI
def test_cli_end_to_end(tmp_path, monkeypatch):
    """tracks.npz equals tracks.build_tracks and the oracle on the tensors rebuilt from features.npz, matches.npz and
    geometry.npz, is byte-stable, and the other outputs are the bytes of a run without the tracks block."""
    import cv2
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    from superpoint_nerf_pytorch_b200 import settings
    root = tmp_path / "data" / "imgs"
    root.mkdir(parents=True)
    for i in range(5):
        img = (smooth_image(96, 128, 80 + i % 3) * 255).astype(np.uint8)
        cv2.imwrite(str(root / f"im{i}.png"), img)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(M.Path(M.__file__).parent / "configs" / "superpoint_match_tracks.yaml"))
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

    out_dir, files = run("trk", cfg)
    assert sorted(files) == ["features.npz", "geometry.npz", "matches.npz", "tracks.npz"]
    _, again = run("trk", cfg)
    assert again == files
    plain = copy.deepcopy(cfg)
    del plain["tracks"]
    _, base = run("plain", plain)
    assert sorted(base) == ["features.npz", "geometry.npz", "matches.npz"]
    for k in base:
        assert base[k] == files[k], k

    t, f, m, g = (np.load(out_dir / k) for k in ("tracks.npz", "features.npz", "matches.npz", "geometry.npz"))
    counts = np.diff(f["offsets"]).astype(np.int32)
    keep = g["inliers"] & np.repeat(g["verified"], np.diff(m["offsets"]))
    got = _build(counts, m["pairs"], m["offsets"], m["matches"], keep)
    want = T.build_tracks(counts, m["pairs"], m["offsets"], m["matches"], keep)
    for name, x, y in zip(("offsets", "observations", "consistent", "track_of"), got, want):
        assert np.array_equal(t[name], x) and np.array_equal(t[name], y) and t[name].dtype == x.dtype, name
    assert len(t["track_of"]) == len(f["keypoints"]) and int(t["min_length"]) == 2
    assert len(t["consistent"]) > 0, "the repeated images give tracks"
