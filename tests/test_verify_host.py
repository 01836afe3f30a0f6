"""Geometric verification without a GPU: the oracle's sampler and solvers (oracle/verify_oracle.py), the
``verification`` config block and the C ABI of include/spn_verify.h."""
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import verify_oracle as V
from verify_scenes import camera_pair, scene, true_fundamental, true_homography


# ---------------------------------------------------------------------------------------------------------- sampler
def test_sampler_draws_distinct_indices_as_a_pure_function():
    for n, s in ((7, 7), (8, 7), (4, 4), (5, 4), (1000, 7), (16384, 4)):
        for h in range(50):
            idx = V.sample(3, 10, 11, h, n, s)
            assert idx is not None and len(set(idx)) == s and all(0 <= i < n for i in idx), (n, s, h, idx)
            assert idx == V.sample(3, 10, 11, h, n, s)
    draws = [tuple(V.sample(0, 1, 2, h, 1000, 7)) for h in range(64)]
    assert len(set(draws)) == 64
    assert V.sample(0, 1, 2, 5, 1000, 7) != V.sample(1, 1, 2, 5, 1000, 7)    # seed, a, b and h all enter the key
    assert V.sample(0, 1, 2, 5, 1000, 7) != V.sample(0, 2, 1, 5, 1000, 7)
    assert V.sample(0, 1, 2, 5, 1000, 7) != V.sample(0, 1, 3, 5, 1000, 7)
    batch, ok = V.samples(V.pair_key(3, 10, 11), np.arange(50), 1000, 7)
    assert ok.all() and [V.sample(3, 10, 11, h, 1000, 7) for h in range(50)] == batch.tolist()


def test_splitmix64_matches_the_reference_values():
    # SplitMix64 outputs for the state sequence 0x9E3779B97F4A7C15 * k from seed 0 (Vigna's reference generator)
    assert int(V.splitmix64(np.uint64(0))) == 0xE220A8397B1DCDAF
    assert int(V.splitmix64(np.uint64(0x9E3779B97F4A7C15))) == 0x6E789E6AA1B965F4


# ---------------------------------------------------------------------------------------------------------- solvers
def _exact_f(seed, n):
    rng = np.random.RandomState(seed)
    K, R, t = camera_pair(rng)
    X = np.c_[rng.uniform(-4, 4, n), rng.uniform(-3, 3, n), rng.uniform(4, 12, n)]
    pa, pb = (K @ X.T).T, (K @ (R @ X.T + t[:, None])).T
    return pa[:, :2] / pa[:, 2:], pb[:, :2] / pb[:, 2:], true_fundamental(K, R, t)


def _exact_h(seed, n):
    rng = np.random.RandomState(seed)
    Hm = true_homography(rng)
    xa = np.c_[rng.uniform(0, 640, n), rng.uniform(0, 480, n)]
    p = (Hm @ np.c_[xa, np.ones(n)].T).T
    return xa, p[:, :2] / p[:, 2:], Hm


def test_seven_point_recovers_a_planted_fundamental_matrix():
    for seed in range(5):
        xa, xb, F = _exact_f(seed, 40)
        T = V.normalisation(xa, xb)
        models, nominal, _, _ = V.solve7(xa[None, :7], xb[None, :7], T)
        found = [V.canonical(models[0, k], "fundamental") for k in range(4) if nominal[0, k]]
        assert found and min(np.abs(m - V.canonical(F, "fundamental")).max() for m in found) < 1e-10, seed


def test_four_point_recovers_a_planted_homography():
    for seed in range(5):
        xa, xb, Hm = _exact_h(seed, 20)
        T = V.normalisation(xa, xb)
        models, nominal, _, _ = V.solve4(np.rint(xa[None, :4]), np.rint(xa[None, :4]), T)   # identity on rounded points
        assert nominal[0, 0] and np.abs(models[0, 0] - np.eye(3)).max() < 1e-10
        models, nominal, _, _ = V.solve4(xa[None, :4] * 0 + xa[None, :4], xb[None, :4], T)
        assert nominal[0, 0] and np.abs(models[0, 0] - Hm).max() / np.abs(Hm).max() < 1e-10, seed
    line = np.array([[[0, 0], [10, 10], [20, 20], [5, 40]]])                     # three collinear points
    T = V.normalisation(np.array([[0, 0], [30, 1], [1, 30.0]]), np.array([[0, 0], [30, 1], [1, 30.0]]))
    assert not V.solve4(line, line + [[1, 2]], T)[1].any()


def test_refit_recovers_the_model_from_all_inliers():
    xa, xb, F = _exact_f(7, 200)
    fit, _ = V.refit(xa, xb, np.ones(200, bool), V.normalisation(xa, xb), "fundamental")
    assert np.abs(V.canonical(fit, "fundamental") - V.canonical(F, "fundamental")).max() < 1e-10
    assert abs(np.linalg.det(fit)) < 1e-12 * np.abs(fit).max() ** 3
    xa, xb, Hm = _exact_h(8, 200)
    fit, _ = V.refit(xa, xb, np.ones(200, bool), V.normalisation(xa, xb), "homography")
    assert np.abs(fit - Hm).max() / np.abs(Hm).max() < 1e-10


def test_ransac_on_planted_scenes_and_degenerate_pairs():
    rng = np.random.RandomState(1)
    for kind in ("fundamental", "homography"):
        xa, xb, true, model = scene(rng, 300, 0.6, kind)
        r = V.ransac(xa, xb, 0, 1, kind)
        err = V.errors(model, xa, xb, kind)
        good = true & (err < 1.5)
        assert (r["inliers"] & good).sum() >= 0.99 * good.sum() and r["num_inliers"] == r["inliers"].sum()
        assert r["hypotheses"] % 256 == 0 and 0 <= r["best"] < r["hypotheses"]
        again = V.ransac(xa, xb, 0, 1, kind)
        assert np.array_equal(again["model"], r["model"]) and again["best"] == r["best"]
        assert V.ransac(xa[:3], xb[:3], 0, 1, kind)["best"] == -1
        same = V.ransac(np.zeros((50, 2)), np.zeros((50, 2)), 0, 1, kind)
        assert same["num_inliers"] == 0 and same["hypotheses"] == 0
    line = np.c_[np.arange(40), 2 * np.arange(40)]
    r = V.ransac(line, line + 3, 0, 1, "homography", max_iters=300)
    assert r["best"] == -1 and r["num_inliers"] == 0 and r["hypotheses"] == 512


# ---------------------------------------------------------------------------------------------------------- config
def _config():
    import yaml
    return yaml.safe_load((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match_verify.yaml").read_text())


def test_verify_config_defaults_and_absence():
    from superpoint_nerf_pytorch_b200.matching import match_config, verify_config
    cfg = _config()
    assert verify_config(cfg) == {"model": "fundamental", "threshold": 3.0, "confidence": 0.999, "max_iters": 10000,
                                  "min_inliers": 15, "seed": 0}
    assert verify_config({"verification": {"model": "homography"}})["model"] == "homography"
    assert verify_config({}) is None and verify_config({"verification": None}) is None
    assert match_config(cfg)["pairs"] == "exhaustive"


def test_verify_config_names_the_key():
    from superpoint_nerf_pytorch_b200.matching import verify_config
    bad = [("modell", "fundamental"), ("model", None), ("model", "essential"), ("threshold", 0), ("threshold", -1.0),
           ("threshold", float("nan")), ("threshold", float("inf")), ("threshold", "3"), ("threshold", True),
           ("confidence", 0), ("confidence", 1), ("confidence", 1.5), ("confidence", float("nan")), ("max_iters", 0),
           ("max_iters", 2.5), ("max_iters", (1 << 24) + 1), ("max_iters", True), ("min_inliers", -1),
           ("min_inliers", 1.0), ("seed", -1), ("seed", 2 ** 64), ("seed", "0")]
    for key, value in bad:
        block = {"model": "fundamental", key: value}
        if key == "model" and value is None:
            block = {"threshold": 3.0}
            key = "model"
        with pytest.raises(ValueError, match=f"verification.{key}"):
            verify_config({"verification": block})
    with pytest.raises(ValueError, match="verification: expected a mapping"):
        verify_config({"verification": [1]})


def test_cli_validates_the_verification_block(tmp_path, monkeypatch):
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    cfg = _config()
    cfg["verification"]["confidence"] = 2
    path = tmp_path / "bad.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("WORLD_SIZE", "1")
    with pytest.raises(ValueError, match="verification.confidence"):
        M.main(config_path=str(path))


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_cabi_exports_the_verify_symbol(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_verify.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.VERIFY_PROTOTYPES) == ["spn_verify_pairs"]
    others = (set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES) | set(N.NERF_PROTOTYPES) | set(N.POSED_PROTOTYPES)
              | set(N.MATCH_PROTOTYPES) | set(N.RETRIEVAL_PROTOTYPES))
    assert not set(N.VERIFY_PROTOTYPES) & others
    assert hasattr(ctypes.CDLL(str(built_lib)), "spn_verify_pairs")


def test_verify_rejects_null_and_out_of_range_arguments(built_lib):
    """A NULL context and out-of-range values -> SPN_E_INVALID (-1) and a message, before any CUDA call (child process;
    the stand-in context and buffers are never dereferenced on these paths)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
fake = C.create_string_buffer(64)
pairs = (C.c_int32 * 4)(0, 1, 1, 0)
def call(ctx=fake, N_=2, cap=8, pr=pairs, P=2, M=4, model=0, t=3.0, conf=0.999, iters=100, ptr=fake, mptr=fake):
    rc = lib.spn_verify_pairs(ctx, ptr, N_, cap, pr, P, ptr, mptr, M, model, t, conf, iters, 0, ptr, ptr, ptr, ptr, mptr, None)
    return rc, lib.spn_last_error().decode()
cases = [(dict(ctx=None), "null pointer (ctx)"), (dict(N_=0), "N = 0"), (dict(N_=(1 << 20) + 1), "keypoint sets outside"),
         (dict(cap=0), "cap = 0"), (dict(cap=16385), "cap = 16385"), (dict(P=-1), "P = -1"), (dict(P=65536), "P = 65536"),
         (dict(M=-1), "M = -1"), (dict(model=2), "model = 2"), (dict(model=-1), "model = -1"), (dict(t=0.0), "threshold"),
         (dict(t=-1.0), "threshold"), (dict(t=float("nan")), "threshold"), (dict(t=float("inf")), "threshold"),
         (dict(conf=0.0), "confidence"), (dict(conf=1.0), "confidence"), (dict(conf=float("nan")), "confidence"),
         (dict(iters=0), "max_iters = 0"), (dict(iters=(1 << 24) + 1), "max_iters"), (dict(ptr=None), "null pointer"),
         (dict(pr=None), "null pointer"), (dict(mptr=None), "null pointer (matches / inlier"),
         (dict(pr=(C.c_int32 * 4)(0, 1, 2, 0)), "pair 1 = (2, 0)"), (dict(pr=(C.c_int32 * 4)(0, -1, 1, 0)), "pair 0 = (0, -1)")]
for kw, msg in cases:
    rc, err = call(**kw)
    assert rc == -1 and msg in err, (kw, rc, err)
assert call(P=0, pr=None, ptr=None, mptr=None)[0] == 0                 # P = 0: a no-op
print("checked", len(cases) + 1)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 25" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
