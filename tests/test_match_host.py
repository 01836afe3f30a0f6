"""Feature matching without a GPU: the fp64 matching oracle against closed forms, pair lists, config validation, the
image folder, the output writer, the C ABI of include/spn_match.h and the CLI's single-process rule."""
import math
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import match_oracle as O


def _unit(n, c=64, seed=0):
    x = np.random.RandomState(seed).randn(n, c)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


# ---------------------------------------------------------------------------------------------------------- oracle
def test_oracle_identical_sets_give_identity_matches():
    a = _unit(50)
    for mutual in (False, True):
        r = O.match(a, a, mutual=mutual, ratio=0.8)
        assert r["match"].tolist() == list(range(50))
        assert np.abs(r["dist"]).max() < 1e-7


def test_oracle_permuted_set_gives_the_permutation():
    a = _unit(40, seed=1)
    perm = np.random.RandomState(2).permutation(40)
    r = O.match(a, a[perm])
    assert np.array_equal(a[perm][r["match"]], a)
    assert np.array_equal(perm[r["match"]], np.arange(40))


def test_oracle_ratio_and_threshold_on_hand_built_distances():
    # a = e0; b0 = e0 + 0.5 e1 (d = 0.5), b1 = e0 + e2 (d = 1): both exact in binary
    a = np.zeros((1, 4))
    a[0, 0] = 1.0
    b = np.array([[1.0, 0.5, 0, 0], [1.0, 0, 1.0, 0]])
    r = O.match(a, b, mutual=False)
    assert r["best"].tolist() == [0] and r["d1"].tolist() == [0.5] and r["d2"].tolist() == [1.0]
    assert O.match(a, b, mutual=False, ratio=0.8)["match"].tolist() == [0]       # 0.5 < 0.8
    assert O.match(a, b, mutual=False, ratio=0.5)["match"].tolist() == [-1]      # 0.5 < 0.5 is false: strict
    assert O.match(a, b, mutual=False, ratio=0.51)["match"].tolist() == [0]
    assert O.match(a, b, mutual=False, max_dist=0.5)["match"].tolist() == [0]    # d1 <= max_dist
    assert O.match(a, b, mutual=False, max_dist=0.49)["match"].tolist() == [-1]
    r = O.match(a, b, mutual=False, ratio=0.8, max_dist=0.75)
    assert r["match"].tolist() == [0] and r["dist"].tolist() == [0.5]
    assert r["margin"][0] == pytest.approx(min(1 - 0.25, abs(0.25 - 0.64), abs(0.25 - 0.5625)))   # in d^2


def test_oracle_duplicate_rows_tie_to_the_lower_index():
    a = _unit(10, seed=3)
    b = np.concatenate([_unit(5, seed=4), a[[7, 7]], a[[2]], a[[2]]])   # a7 at 5 and 6, a2 at 7 and 8
    r = O.match(a, b, mutual=False)
    assert r["best"][7] == 5 and r["best"][2] == 7
    assert r["d1"][7] == r["d2"][7] and np.isfinite(r["margin"][7])      # an exact copy is not a margin
    assert O.match(a, b, mutual=False, ratio=1.0)["match"][[2, 7]].tolist() == [-1, -1]   # d1 = d2 fails d1 < d2
    # duplicates in a: both copies pick the same row of b, the mutual check keeps the lower one
    a2 = np.concatenate([a, a[[4]]])
    r = O.match(a2, a2, mutual=True)
    assert r["match"][4] == 4 and r["match"][10] == -1


def test_oracle_empty_and_single_row_sets():
    a = _unit(6, seed=5)
    assert O.match(a[:0], a)["match"].shape == (0,)
    r = O.match(a, a[:0], ratio=0.8)
    assert r["match"].tolist() == [-1] * 6 and r["dist"].tolist() == [0.0] * 6
    r = O.match(a, a[:1], mutual=False, ratio=0.8)                    # second = inf: the ratio test passes
    assert r["match"].tolist() == [0] * 6 and np.isinf(r["d2"]).all()
    r = O.match(a, a[:1], mutual=True)                                 # only a0 is b0's nearest
    assert r["match"].tolist() == [0, -1, -1, -1, -1, -1]
    pool = np.zeros((3, 8, 64))
    pool[0, :6], pool[1, :1] = a, a[:1]
    out = O.match_pairs(pool, [6, 1, 0], [(0, 1), (0, 2), (2, 0), (0, 0)], mutual=False)
    assert out["match"][0, :6].tolist() == [0] * 6 and (out["match"][0, 6:] == -1).all()
    assert (out["match"][1:3] == -1).all() and out["match"][3, :6].tolist() == list(range(6))


# ---------------------------------------------------------------------------------------------------------- pairs
def test_pair_list_modes():
    from superpoint_nerf_pytorch_b200.matching import pair_list
    names = ["a.png", "b.png", "c.png", "d.png"]
    assert pair_list(names, "exhaustive") == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    assert len(pair_list([str(i) for i in range(32)], "exhaustive")) == 496
    assert pair_list(names, "sequential", 1) == [(0, 1), (1, 2), (2, 3)]
    assert pair_list(names, "sequential", 2) == [(0, 1), (0, 2), (1, 2), (1, 3), (2, 3)]
    assert pair_list(names, "sequential", 10) == pair_list(names, "exhaustive")
    assert pair_list(names[:1], "exhaustive") == [] and pair_list([], "sequential", 3) == []
    for w in (0, -1, None, 1.5, True):
        with pytest.raises(ValueError, match="window"):
            pair_list(names, "sequential", w)
    with pytest.raises(ValueError, match="pair mode"):
        pair_list(names, "all")


def test_pair_list_from_file(tmp_path):
    from superpoint_nerf_pytorch_b200.matching import pair_list
    names = ["a.png", "sub/b.png", "c.png"]
    f = tmp_path / "pairs.txt"
    f.write_text("# comment\na.png sub/b.png\n\n  c.png a.png  \nsub/b.png c.png\n")
    assert pair_list(names, "file", pairs_file=f) == [(0, 1), (2, 0), (1, 2)]
    bad = [("a.png x.png\n", r":1: unknown image name 'x.png'"),
           ("a.png c.png\nc.png c.png\n", r":2: pairs an image with itself"),
           ("a.png c.png\n#\nc.png a.png\n", r":3: duplicate of the pair on line 1"),
           ("a.png c.png\na.png c.png\n", r":2: duplicate of the pair on line 1"),
           ("a.png\n", r":1: expected 'name_a name_b'"),
           ("a.png c.png sub/b.png\n", r":1: expected 'name_a name_b'")]
    for text, msg in bad:
        f.write_text(text)
        with pytest.raises(ValueError, match=re.escape(str(f)) + msg):
            pair_list(names, "file", pairs_file=f)


# ---------------------------------------------------------------------------------------------------------- config
def _config():
    import yaml
    return yaml.safe_load((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match.yaml").read_text())


def test_config_validation_names_the_key():
    from superpoint_nerf_pytorch_b200.matching import MATCH_DEFAULTS, match_config
    cfg = _config()
    assert match_config(cfg) == {"pairs": "exhaustive", "window": 5, "pairs_file": None, "mutual": True, "ratio": 0.0,
                                 "max_dist": math.inf}
    assert match_config({k: v for k, v in cfg.items() if k != "matching"}) == MATCH_DEFAULTS
    bad = [("pair", "exhaustive"), ("pairs", "all"), ("window", 0), ("window", 2.5), ("window", True), ("pairs_file", 3),
           ("mutual", "yes"), ("ratio", 1.5), ("ratio", -0.1), ("ratio", "0.8"), ("ratio", float("nan")), ("max_dist", -1.0),
           ("max_dist", float("nan")), ("max_dist", True)]
    for key, value in bad:
        c = dict(cfg, matching=dict(cfg["matching"], **{key: value}))
        with pytest.raises(ValueError, match=f"matching.{key}"):
            match_config(c)
    with pytest.raises(ValueError, match="matching.window: required"):
        match_config(dict(cfg, matching={"pairs": "sequential"}))
    with pytest.raises(ValueError, match="matching.pairs_file: required"):
        match_config(dict(cfg, matching={"pairs": "file"}))
    import copy
    mp = copy.deepcopy(cfg)
    mp["model"]["model_name"] = "magicpoint"
    del mp["model"]["descriptor_head"]
    with pytest.raises(ValueError, match="MagicPoint"):
        match_config(mp)
    for top_k in (0, None, -5):
        c = copy.deepcopy(cfg)
        c["model"]["detector_head"]["top_k"] = top_k
        with pytest.raises(ValueError, match="model.detector_head.top_k"):
            match_config(c)
    c = copy.deepcopy(cfg)
    c["data"]["batch_size"] = 0
    with pytest.raises(ValueError, match="data.batch_size"):
        match_config(c)


# ---------------------------------------------------------------------------------------------------------- images
def test_image_folder_listing_and_errors(tmp_path, monkeypatch):
    import cv2
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.data.ImageFolder import ImageFolder
    root = tmp_path / "imgs"
    (root / "sub").mkdir(parents=True)
    rng = np.random.RandomState(0)
    cv2.imwrite(str(root / "b.png"), rng.randint(0, 255, (16, 24), np.uint8))
    cv2.imwrite(str(root / "sub" / "a.jpg"), rng.randint(0, 255, (16, 24, 3), np.uint8))
    cv2.imwrite(str(root / "a.jpeg"), rng.randint(0, 255, (20, 30), np.uint8))
    (root / "notes.txt").write_text("not an image")
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path))
    ds = ImageFolder({"name": "imgs"}, device="cpu")
    assert ds.names == ["a.jpeg", "b.png", "sub/a.jpg"]
    it = ds[1]
    assert it["name"] == "b.png" and it["shape"] == (16, 24) and it["image"].dtype == np.uint8 and it["geometry"] is None
    assert ds[2]["image"].shape == (16, 24)                              # colour converted to grayscale
    with pytest.raises(ValueError, match=re.escape(str(root / "a.jpeg")) + ": size 20x30 is not a multiple of 8"):
        ds[0]
    rs = ImageFolder({"name": "imgs", "preprocessing": {"resize": [32, 48]}}, device="cpu")
    assert rs[0]["geometry"] == (32, 48, 0, 0)
    (root / "c.png").write_bytes(b"\x89PNG broken")
    with pytest.raises(ValueError, match=re.escape(str(root / "c.png")) + ": cannot be decoded"):
        ImageFolder({"name": "imgs"}, device="cpu")[2]
    for resize in ([30, 48], [32], "32x48"):
        with pytest.raises(ValueError, match="data.preprocessing.resize"):
            ImageFolder({"name": "imgs", "preprocessing": {"resize": resize}}, device="cpu")
    (tmp_path / "empty").mkdir()
    with pytest.raises(ValueError, match="no .png/.jpg/.jpeg images"):
        ImageFolder({"name": "empty"}, device="cpu")
    with pytest.raises(ValueError, match="no such image folder"):
        ImageFolder({"name": "missing"}, device="cpu")


def test_writer_is_shared_and_deterministic(tmp_path):
    from superpoint_nerf_pytorch_b200.evaluations import posed_evaluation
    from superpoint_nerf_pytorch_b200.utils.npz import write_npz
    assert posed_evaluation._write_npz is write_npz
    arrays = {"names": np.array(["a.png", "sub/b.png"]), "offsets": np.array([0, 3, 5]), "max_dist": np.array(np.inf),
              "distances": np.arange(4, dtype=np.float32)}
    write_npz(tmp_path / "one.npz", arrays)
    write_npz(tmp_path / "two.npz", dict(reversed(list(arrays.items()))))
    assert (tmp_path / "one.npz").read_bytes() == (tmp_path / "two.npz").read_bytes()
    z = np.load(tmp_path / "one.npz")
    assert sorted(z.files) == sorted(arrays) and all(np.array_equal(z[k], v) for k, v in arrays.items())


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_cabi_exports_the_match_pairs_symbol(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_match.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.MATCH_PROTOTYPES) == ["spn_match_pairs"]
    others = set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES) | set(N.NERF_PROTOTYPES) | set(N.POSED_PROTOTYPES)
    assert not set(N.MATCH_PROTOTYPES) & others
    assert hasattr(ctypes.CDLL(str(built_lib)), "spn_match_pairs")


def test_match_pairs_rejects_null_and_out_of_range_arguments(built_lib):
    """NULL context and out-of-range arguments -> SPN_E_INVALID (-1) and a message, before any CUDA call (child
    process; the stand-in context and buffers are never dereferenced on these paths)."""
    code = r'''
import sys, math, ctypes as C
import numpy as np
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
for name, (res, args) in N.MATCH_PROTOTYPES.items():
    rc = getattr(lib, name)(*[None if a in (C.c_void_p, C.c_char_p) else a(0) for a in args])
    assert rc == -1 and "null pointer" in lib.spn_last_error().decode(), (name, rc)
fake = C.create_string_buffer(64)
pairs = np.array([[0, 1], [1, 0]], np.int32)
P = C.c_void_p(pairs.ctypes.data)
def call(N_=2, cap=100, Cc=256, pairs=P, n=2, mutual=1, ratio=0.0, max_dist=math.inf, out=fake):
    rc = lib.spn_match_pairs(fake, fake, fake, N_, cap, Cc, pairs, n, mutual, C.c_float(ratio), C.c_float(max_dist), out, out, None)
    return rc, lib.spn_last_error().decode()
cases = [(dict(N_=0), "N = 0"), (dict(N_=(1 << 20) + 1), "descriptor sets outside"), (dict(cap=0), "cap = 0"),
         (dict(cap=16385), "cap = 16385"), (dict(Cc=100), "multiple of 64"), (dict(Cc=0), "C = 0"), (dict(n=-1), "P = -1"),
         (dict(n=65536), "P = 65536"), (dict(ratio=1.5), "ratio must be in [0, 1]"), (dict(ratio=-0.1), "ratio"),
         (dict(ratio=float("nan")), "ratio"), (dict(max_dist=float("nan")), "max_dist must not be NaN"),
         (dict(pairs=None), "null pointer"), (dict(out=None), "null pointer"), (dict(N_=1), "pair 0 = (0, 1) has a set index outside [0, 1)")]
for kw, msg in cases:
    rc, err = call(**kw)
    assert rc == -1 and msg in err, (kw, rc, err)
neg = np.array([[0, 1], [1, -1]], np.int32)
rc, err = call(pairs=C.c_void_p(neg.ctypes.data))
assert rc == -1 and "pair 1 = (1, -1)" in err, err
assert call(n=0, pairs=None, out=None)[0] == 0          # P = 0 is a no-op
print("checked", len(cases) + 3)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 18" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


# ---------------------------------------------------------------------------------------------------------- CLI
def test_cli_is_single_process(tmp_path, monkeypatch):
    from superpoint_nerf_pytorch_b200 import matching as M
    cfg = tmp_path / "match.yaml"
    cfg.write_text((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match.yaml").read_text())
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit, match="single process"):
        M.main(config_path=str(cfg))
    monkeypatch.setenv("WORLD_SIZE", "1")
    bad = tmp_path / "bad.yaml"
    bad.write_text(cfg.read_text().replace("ratio: 0.0", "ratio: 2.0"))
    with pytest.raises(ValueError, match="matching.ratio"):
        M.main(config_path=str(bad))
    if not torch.cuda.is_available():
        with pytest.raises(SystemExit, match="CUDA is not available"):
            M.main(config_path=str(cfg), random_init=True)
