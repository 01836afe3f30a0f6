"""Retrieval without a GPU: the numpy oracle on closed forms, pair lists from neighbour lists, the ``retrieval`` config
block and the vocabulary file checks, and the C ABI of include/spn_retrieval.h."""
import copy
import math
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import retrieval_oracle as R


def _unit(n, c=64, seed=0):
    x = np.random.RandomState(seed).randn(n, c)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


# ---------------------------------------------------------------------------------------------------------- oracle
def test_oracle_identical_sets():
    a = _unit(30)
    idx, d2, margin = R.knn(a, a, 3)
    assert idx[:, 0].tolist() == list(range(30)) and np.abs(d2[:, 0]).max() < 1e-12
    assert (np.diff(d2, axis=1) >= 0).all() and (margin > 0).all()
    idx, d2, _ = R.knn(a, a, 3, exclude_self=True)
    assert (idx != np.arange(30)[:, None]).all()
    want, _, _ = R.knn(a, a, 4)
    assert np.array_equal(idx, want[:, 1:])                                  # self is rank 0 when it is not excluded


def test_oracle_permuted_set():
    a = _unit(40, seed=1)
    perm = np.random.RandomState(2).permutation(40)
    idx, _, _ = R.knn(a, a[perm], 1)
    assert np.array_equal(perm[idx[:, 0]], np.arange(40))


def test_oracle_planted_duplicates_tie_to_the_lower_index():
    a = _unit(10, seed=3)
    t = np.concatenate([_unit(5, seed=4), a[[7, 7, 7]], a[[2]]])            # a7 at 5, 6, 7; a2 at 8
    idx, d2, margin = R.knn(a, t, 3)
    assert idx[7].tolist() == [5, 6, 7] and (d2[7] < 1e-12).all()
    assert idx[2, 0] == 8
    assert np.isfinite(margin[7]) and margin[7] > 0.1                          # the copies are not a margin; rank 3 is
    t2 = np.concatenate([t, t[[0]]])                                         # a copy of t0 at rank k / k + 1
    _, _, m2 = R.knn(t[:1], t2, 1)
    assert m2[0] > 0.1


def test_oracle_k_larger_than_the_set():
    a, t = _unit(4, seed=5), _unit(3, seed=6)
    idx, d2, _ = R.knn(a, t, 5)
    assert (idx[:, 3:] == -1).all() and np.isinf(d2[:, 3:]).all() and sorted(idx[0, :3]) == [0, 1, 2]
    idx, d2, _ = R.knn(t, t, 5, exclude_self=True)
    assert (idx[:, 2:] == -1).all() and np.isinf(d2[:, 2:]).all()
    idx, d2, margin = R.knn(a, t[:0], 2)
    assert (idx == -1).all() and np.isinf(d2).all() and np.isinf(margin).all()
    assert R.knn(a[:0], t, 2)[0].shape == (0, 2)


def test_oracle_residual_sums_and_vlad():
    rng = np.random.RandomState(7)
    desc = rng.randn(3, 5, 4).astype(np.float32)
    words = rng.randn(2, 4).astype(np.float32)
    assign = np.array([[0, 1, 0, -1, 2], [1, 1, 1, 1, 1], [0, 0, 0, 0, 0]])
    sums, n = R.residual_sums(desc, [5, 3, 0], assign, words)
    assert n.tolist() == [[2, 1], [0, 3], [0, 0]]
    want = np.float32(desc[0, 0] - words[0]) + np.float32(desc[0, 2] - words[0])
    assert np.array_equal(sums[0, 0], want.astype(np.float32)) and (sums[2] == 0).all()
    v = R.vlad(sums)
    assert v.shape == (3, 8) and (v[2] == 0).all() and np.allclose(np.linalg.norm(v[:2], axis=1), 1)
    assert np.allclose(np.linalg.norm(v[1, :4]), 0) and np.allclose(np.linalg.norm(v[0, :4]), np.sqrt(0.5))
    step = R.kmeans_step(desc, [5, 3, 0], np.where(assign == 2, 0, assign), words)
    assert np.allclose(step[0], desc[0, [0, 2, 4]].astype(np.float64).mean(0))


# ---------------------------------------------------------------------------------------------------------- pairs
def test_retrieval_pairs_from_neighbour_lists():
    from superpoint_nerf_pytorch_b200.matching import pair_list
    from superpoint_nerf_pytorch_b200.retrieval import retrieval_pairs
    index = np.array([[1, 2], [0, -1], [3, 0], [-1, -1]])
    assert retrieval_pairs(index) == R.retrieval_pairs(index) == [(0, 1), (0, 2), (2, 3)]
    for N in (1, 2, 5, 9):                                                   # k >= N - 1: the exhaustive list
        full = np.array([[j for j in range(N) if j != i] + [-1] for i in range(N)]).reshape(N, N)
        assert retrieval_pairs(full) == pair_list([str(i) for i in range(N)], "exhaustive")
    assert retrieval_pairs(np.zeros((0, 3), np.int32)) == []
    with pytest.raises(ValueError, match="retrieval needs the descriptors"):
        pair_list(["a", "b"], "retrieval")


# ---------------------------------------------------------------------------------------------------------- config
def _config():
    import yaml
    return yaml.safe_load((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match_retrieval.yaml").read_text())


def test_match_config_accepts_retrieval():
    from superpoint_nerf_pytorch_b200.matching import match_config, retrieval_config
    cfg = _config()
    assert match_config(cfg)["pairs"] == "retrieval"
    assert retrieval_config(cfg) == {"num_neighbors": 20, "vocab_size": 64, "kmeans_iters": 20, "vocabulary": None}
    assert retrieval_config({}) == retrieval_config({"retrieval": None}) == retrieval_config(cfg)


def test_retrieval_config_names_the_key():
    from superpoint_nerf_pytorch_b200.matching import retrieval_config
    cfg = _config()
    bad = [("neighbours", 3), ("num_neighbors", 0), ("num_neighbors", 129), ("num_neighbors", 2.0), ("num_neighbors", True),
           ("vocab_size", 0), ("vocab_size", 257), ("vocab_size", "64"), ("kmeans_iters", 0), ("kmeans_iters", None),
           ("vocabulary", 3), ("vocabulary", "")]
    for key, value in bad:
        c = dict(cfg, retrieval=dict(cfg["retrieval"], **{key: value}))
        with pytest.raises(ValueError, match=f"retrieval.{key}"):
            retrieval_config(c)
    with pytest.raises(ValueError, match="retrieval: expected a mapping"):
        retrieval_config({"retrieval": [1]})
    for key in ("vocab_size", "kmeans_iters"):                              # a loaded vocabulary excludes k-means keys
        with pytest.raises(ValueError, match=f"retrieval.vocabulary: .*retrieval.{key}"):
            retrieval_config({"retrieval": {"vocabulary": "r.npz", key: 8}})
    assert retrieval_config({"retrieval": {"vocabulary": "r.npz", "num_neighbors": 5}})["vocabulary"] == "r.npz"


def test_vocabulary_file_checks(tmp_path):
    from superpoint_nerf_pytorch_b200.matching import load_vocabulary
    from superpoint_nerf_pytorch_b200.utils.npz import write_npz
    good = np.random.RandomState(0).randn(16, 256).astype(np.float32)
    write_npz(tmp_path / "ok.npz", {"words": good, "neighbors": np.zeros((3, 2), np.int32)})
    assert np.array_equal(load_vocabulary(tmp_path / "ok.npz"), good)
    nan = good.copy()
    nan[3, 4] = np.nan
    cases = [({"words": good.astype(np.float64)}, "float32"), ({"words": good[:, :128]}, r"\(K, 256\)"),
             ({"words": good[0]}, r"\(K, 256\)"), ({"words": np.zeros((0, 256), np.float32)}, r"1 <= K <= 256"),
             ({"words": np.zeros((257, 256), np.float32)}, r"1 <= K <= 256"), ({"words": nan}, "non-finite"),
             ({"neighbors": np.zeros(2)}, "no 'words' array")]
    for i, (arrays, msg) in enumerate(cases):
        f = tmp_path / f"bad{i}.npz"
        write_npz(f, arrays)
        with pytest.raises(ValueError, match="retrieval.vocabulary: " + re.escape(str(f)) + ": .*" + msg):
            load_vocabulary(f)
    (tmp_path / "junk.npz").write_bytes(b"not a zip")
    for f in (tmp_path / "junk.npz", tmp_path / "missing.npz"):
        with pytest.raises(ValueError, match="retrieval.vocabulary: " + re.escape(str(f)) + ": cannot be read"):
            load_vocabulary(f)


def test_cli_validates_the_retrieval_block(tmp_path, monkeypatch):
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    cfg = _config()
    cfg["retrieval"]["num_neighbors"] = 500
    path = tmp_path / "bad.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("WORLD_SIZE", "1")
    with pytest.raises(ValueError, match="retrieval.num_neighbors"):
        M.main(config_path=str(path))
    other = copy.deepcopy(cfg)                                               # not consulted in the other modes
    other["matching"]["pairs"] = "exhaustive"
    assert M.match_config(other)["pairs"] == "exhaustive"


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_cabi_exports_the_retrieval_symbols(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_retrieval.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.RETRIEVAL_PROTOTYPES) == ["spn_knn",
                                                                                                       "spn_residual_sums"]
    others = set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES) | set(N.NERF_PROTOTYPES) | set(N.POSED_PROTOTYPES) | set(N.MATCH_PROTOTYPES)
    assert not set(N.RETRIEVAL_PROTOTYPES) & others
    lib = ctypes.CDLL(str(built_lib))
    assert all(hasattr(lib, name) for name in N.RETRIEVAL_PROTOTYPES)


def test_retrieval_calls_reject_null_and_out_of_range_arguments(built_lib):
    """NULL or zero arguments and out-of-range values -> SPN_E_INVALID (-1) and a message, before any CUDA call (child
    process; the stand-in context and buffers are never dereferenced on these paths)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
for name, (res, args) in N.RETRIEVAL_PROTOTYPES.items():
    rc = getattr(lib, name)(*[None if a in (C.c_void_p, C.c_char_p) else a(0) for a in args])
    assert rc == -1 and "null pointer" in lib.spn_last_error().decode(), (name, rc)
fake = C.create_string_buffer(64)
def knn(nq=10, nt=10, Cc=256, k=4, excl=0, q=fake, t=fake, out=fake):
    rc = lib.spn_knn(fake, q, nq, t, nt, Cc, k, excl, out, out, None)
    return rc, lib.spn_last_error().decode()
def res(N_=2, cap=8, Cc=256, K=4, ptr=fake):
    rc = lib.spn_residual_sums(fake, ptr, ptr, ptr, ptr, N_, cap, Cc, K, ptr, ptr, None)
    return rc, lib.spn_last_error().decode()
cases = [(knn, dict(k=0), "k = 0 outside [1, 128]"), (knn, dict(k=129), "k = 129"), (knn, dict(Cc=0), "C = 0"),
         (knn, dict(Cc=100), "multiple of 64"), (knn, dict(Cc=65600), "up to 65536"), (knn, dict(nq=-1), "nq = -1"),
         (knn, dict(nq=(1 << 26) + 1), "query rows outside"), (knn, dict(nt=-2), "nt = -2"),
         (knn, dict(nt=(1 << 26) + 1), "train rows outside"), (knn, dict(excl=1, nt=9), "exclude_self needs the same set"),
         (knn, dict(q=None), "null pointer"), (knn, dict(t=None), "null pointer"), (knn, dict(out=None), "null pointer"),
         (res, dict(N_=-1), "N = -1"), (res, dict(N_=(1 << 26) + 1), "images outside"), (res, dict(cap=0), "cap = 0"),
         (res, dict(cap=(1 << 20) + 1), "cap = 1048577"), (res, dict(Cc=0), "C = 0"), (res, dict(Cc=65537), "C = 65537"),
         (res, dict(K=0), "K = 0"), (res, dict(K=65537), "K = 65537"), (res, dict(ptr=None), "null pointer")]
for fn, kw, msg in cases:
    rc, err = fn(**kw)
    assert rc == -1 and msg in err, (fn.__name__, kw, rc, err)
assert knn(nq=0, nt=0, q=None, t=None, out=None)[0] == 0                 # nq = 0: a no-op
assert knn(nq=0, q=None, out=None)[0] == 0
assert res(N_=0, ptr=None)[0] == 0                                       # N = 0: a no-op
print("checked", len(cases) + 5)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 27" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
