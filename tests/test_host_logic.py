"""CPU: host-side mirror of the reference interface, and the C-ABI library (loads, exports every declared symbol,
refuses to run without a GPU).  No compute calls here."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import HA_CFG, MP_MODEL, ROOT, SP_MODEL
from oracle import spn_oracle as O


@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def declared_symbols():
    text = (ROOT / "include" / "spn_b200.h").read_text()
    return sorted(set(re.findall(r"SPN_API\s+[\w\s\*]+?\b(spn_\w+)\s*\(", text)))


def test_cabi_exports_every_declared_symbol(built_lib):
    names = declared_symbols()
    assert len(names) >= 16, names
    lib = ctypes.CDLL(str(built_lib))
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/spn_b200.h but not exported"
    import superpoint_nerf_pytorch_b200._native as N
    assert sorted(N.PROTOTYPES) == names, "ctypes prototypes and header are out of sync"
    lib.spn_version.restype = ctypes.c_int
    assert lib.spn_version() >= 100


def test_no_silent_cpu_fallback(built_lib):
    import superpoint_nerf_pytorch_b200 as P
    from superpoint_nerf_pytorch_b200.models.model_utils.sp_utils import box_nms
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    if torch.cuda.is_available():
        pytest.skip("this check is for the GPU-less container")
    with pytest.raises(P.NativeError):
        P.Context()
    with pytest.raises(P.NativeError):
        box_nms(torch.zeros(8, 8), 4)
    m = get_model(MP_MODEL, "cpu")
    with pytest.raises(P.NativeError):
        m(torch.zeros(1, 1, 16, 16))
    lib = ctypes.CDLL(str(built_lib))
    h = ctypes.c_void_p()
    lib.spn_last_error.restype = ctypes.c_char_p
    assert lib.spn_create(ctypes.byref(h), 0) != 0
    assert b"no CPU fallback" in lib.spn_last_error() or b"CUDA" in lib.spn_last_error()


def test_state_dict_is_reference_compatible():
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    for cfg in (MP_MODEL, SP_MODEL):
        m = get_model(cfg, "cpu")
        sd = O.make_state_dict(cfg["model_name"], seed=0)
        assert set(sd) == set(m.state_dict())
        assert all(sd[k].shape == v.shape for k, v in m.state_dict().items())
        m.load_state_dict(sd)  # engine.py:108-117 style loading works
    with pytest.raises(Exception):
        get_model(MP_MODEL, "cpu").train()


def test_host_sampler_bit_equal_to_reference(golden):
    from superpoint_nerf_pytorch_b200.data.data_utils.homographic_augmentation import (Homographic_aug,
                                                                                      perspective_from_corners,
                                                                                      sample_corners)
    g = golden("homographies.npz")
    aug = Homographic_aug({"params": HA_CFG["params"], "valid_border_margin": 3}, "cpu")
    for s in range(6):
        np.random.seed(s)
        got = torch.cat([aug.sample_homography((240, 320), **HA_CFG["params"]) for _ in range(3)]).numpy()
        assert np.array_equal(got, g[f"s{s}"])
    np.random.seed(100)
    p2 = dict(HA_CFG["params"], allow_artifacts=False, patch_ratio=0.5, n_scales=5, n_angles=25, translation_overflow=0.0)
    got = torch.cat([aug.sample_homography((120, 160), **p2) for _ in range(3)]).numpy()
    assert np.array_equal(got, g["noartifact"])
    import cv2
    np.random.seed(1)
    s, d = sample_corners(**HA_CFG["params"])
    wh = np.array([[320, 240.0]])
    M = cv2.getPerspectiveTransform(np.float32(s * wh), np.float32(d * wh))
    assert np.abs(M - perspective_from_corners(s * wh, d * wh)).max() < 1e-5


def test_move_to_device_and_get_model():
    from superpoint_nerf_pytorch_b200.utils.train_utils import move_to_device
    d = {"a": torch.zeros(2), "b": [torch.ones(1), "x"], "name": ["n"]}
    out = move_to_device(d, "cpu")
    assert out["name"] == ["n"] and out["b"][1] == "x" and torch.equal(out["a"], d["a"])


def test_shard_plan():
    from superpoint_nerf_pytorch_b200.utils.sharding import shard_indices
    for n in (0, 1, 7, 10000):
        for world in (1, 2, 4, 8):
            parts = [shard_indices(n, r, world) for r in range(world)]
            allidx = sorted(i for p in parts for i in p)
            assert allidx == list(range(n))
            assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_preprocessing_host_side_matches_reference(golden):
    from superpoint_nerf_pytorch_b200.data.preprocessing import adapt_homography_to_resize, resize_geometry
    import torchvision.transforms.functional as TF
    g = golden("preprocess.npz")
    h = adapt_homography_to_resize(g["h_in"], [480.0, 640.0], [427.0, 600.0], (240, 320))
    assert np.array_equal(h.numpy(), g["h_out"])
    # crop geometry == what torchvision's center_crop does on the resized image (incl. the zero-padded case)
    for src, tgt in [((96, 128), (48, 64)), ((107, 160), (48, 64)), ((160, 120), (48, 64)), ((61, 80), (60, 80)), ((50, 70), (48, 64)),
                     ((427, 640), (240, 320)), ((333, 500), (240, 320)), ((30, 90), (48, 64))]:
        nh, nw, top, left = resize_geometry(src, tgt)
        probe = torch.arange(nh * nw, dtype=torch.float32).reshape(nh, nw) + 1.0
        want = TF.center_crop(probe, list(tgt))
        got = torch.zeros(tgt)
        for y in range(tgt[0]):
            for x in range(tgt[1]):
                ry, rx = y + top, x + left
                if 0 <= ry < nh and 0 <= rx < nw:
                    got[y, x] = probe[ry, rx]
        assert torch.equal(got, want), (src, tgt)


def test_npz_writer_pool_is_transparent(tmp_path):
    """The HPatches exports hand np.savez_compressed to a bounded thread pool: same bytes as a synchronous save, bounded
    number of files in flight, and a writer's exception surfaces in the caller."""
    from superpoint_nerf_pytorch_b200.engine_solvers.export import _NpzWriter
    rng = np.random.RandomState(3)
    items = [{"image": rng.rand(24, 32).astype(np.float32), "prob": rng.rand(24, 32).astype(np.float32),
              "homography": np.eye(3, dtype=np.float32) * (k + 1)} for k in range(9)]
    w = _NpzWriter(workers=3, depth=4)
    for k, it in enumerate(items):
        w.save(tmp_path / f"a{k}.npz", it)
        assert len(w.pending) <= 4
    w.close()
    for k, it in enumerate(items):
        np.savez_compressed(tmp_path / f"b{k}.npz", **it)
        assert (tmp_path / f"a{k}.npz").read_bytes() == (tmp_path / f"b{k}.npz").read_bytes()
    w = _NpzWriter(workers=1, depth=1)
    w.save(tmp_path / "missing_dir" / "x.npz", items[0])
    with pytest.raises(Exception):
        w.close()


def test_weights_key_tracks_parameter_updates():
    """The packed-weight cache key must change when weights are loaded or modified in place."""
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    m = get_model(MP_MODEL, "cpu")
    k0 = m._weights_key()
    assert m._weights_key() == k0
    m.load_state_dict(O.make_state_dict("magicpoint", seed=1))
    k1 = m._weights_key()
    assert k1 != k0
    with torch.no_grad():
        m.detector_head.convPb.conv2d.bias.add_(1.0)
    assert m._weights_key() != k1


def test_kornia_geometry_mirror_matches_the_shim():
    """utils/kornia_geometry.sampling_matrices (what the binding uploads for host homographies) == the matrices the
    restated kornia.warp_perspective builds (oracle/kornia_shim.py), bit for bit, and == the committed reference bits."""
    from oracle import kornia_shim as K
    from superpoint_nerf_pytorch_b200.utils.kornia_geometry import sampling_matrices
    g = np.load(ROOT / "tests" / "golden" / "ha_masks.npz")
    for ci in range(int(g["n"])):
        h, w, _margin, n = (int(v) for v in g[f"c{ci}_par"])
        Hc = torch.from_numpy(g[f"c{ci}_H"])
        fwd, bwd = sampling_matrices(Hc, (h, w))
        for i in range(n):
            a = K._inverse_cast(K.normalize_homography(Hc[i:i + 1], (h, w), (h, w)))[0]
            b = K._inverse_cast(K.normalize_homography(torch.inverse(Hc[i:i + 1]), (h, w), (h, w)))[0]
            assert torch.equal(fwd[i], a) and torch.equal(bwd[i], b)
        assert np.array_equal(fwd.numpy(), g[f"c{ci}_ainv"]) and np.array_equal(bwd.numpy(), g[f"c{ci}_ainv_back"])


def test_move_to_device_handles_loader_containers():
    from collections import defaultdict, namedtuple
    from superpoint_nerf_pytorch_b200.utils.train_utils import move_to_device
    Pair = namedtuple("Pair", "a b")
    dd = defaultdict(list)
    dd["x"] = torch.zeros(2)
    batch = {"raw": {"image": torch.ones(1, 1, 4, 4)}, "name": ["n"], "pair": Pair(torch.zeros(1), "s"), "dd": dd,
             "rng": range(3), "tup": (torch.zeros(1), 2)}
    out = move_to_device(batch, "cpu")
    assert isinstance(out["pair"], Pair) and out["pair"].b == "s" and torch.equal(out["pair"].a, torch.zeros(1))
    assert out["dd"]["x"].shape == (2,) and out["rng"] == range(3) and isinstance(out["tup"], tuple)
    assert out["name"] == ["n"] and out["raw"]["image"].shape == (1, 1, 4, 4)


def test_cli_accepts_reference_flag_groups():
    """engine.py:14-59 of the reference: --training.* and --pseudo_labels.* parse; out-of-scope tasks are rejected at
    dispatch, not by the parser."""
    import tyro
    from superpoint_nerf_pytorch_b200 import engine
    seen = {}

    def fake_main(**kw):
        seen.update(kw)
    import inspect
    sig = inspect.signature(engine.main)
    assert {"config_path", "task", "training", "pseudo_labels"} <= set(sig.parameters)
    with pytest.raises(SystemExit) as e:
        tyro.cli(engine.main, use_underscores=True,
                 args=["--config_path", "x.yaml", "--task", "train", "--training.validate_training", "True",
                       "--training.include_mask_loss", "False", "--pseudo_labels.split", "validation"])
    assert "outside the B200 hot path" in str(e.value)


def test_sharded_loader_partitions_items():
    from superpoint_nerf_pytorch_b200.engine import ShardedLoader
    items = list(range(11))
    parts = [list(ShardedLoader(items, r, 3)) for r in range(3)]
    assert sorted(sum(parts, [])) == items and [len(ShardedLoader(items, r, 3)) for r in range(3)] == [len(p) for p in parts]


def test_prefetch_loader_order_sharding_and_dataset_listing(tmp_path, monkeypatch):
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.utils.data_loaders import PrefetchLoader

    class Fake:
        def __len__(self):
            return 23

        def decode(self, i):
            return i

        def finish(self, d):
            return {"v": d * 10}

        def batch_collator(self, batch):
            return [b["v"] for b in batch]

    assert list(PrefetchLoader(Fake(), batch_size=1, workers=4)) == [[10 * i] for i in range(23)]
    assert sum(list(PrefetchLoader(Fake(), batch_size=4, workers=3)), []) == [10 * i for i in range(23)]
    parts = [sum(list(PrefetchLoader(Fake(), 1, workers=2, rank=r, world=3)), []) for r in range(3)]
    assert sorted(sum(parts, [])) == [10 * i for i in range(23)] and parts[1][0] == 10
    assert len(PrefetchLoader(Fake(), 4, rank=1, world=3)) == 2
    # dataset listing (COCO.py:34-56): <DATA_PATH>/<name>/images/<split>/*
    import cv2
    d = tmp_path / "COCO" / "images" / "validation"
    d.mkdir(parents=True)
    for k in range(4):
        cv2.imwrite(str(d / f"im{k}.jpg"), np.full((20, 30), 40 * k, np.uint8))
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path))
    from superpoint_nerf_pytorch_b200.data.COCO import COCO
    cfg = {"name": "COCO", "preprocessing": {"resize": [16, 24]}, "has_labels": False, "warped_pair": False, "truncate": 0.5,
           "augmentation": {"photometric": {"enable": False}, "homographic": {"enable": False}}}
    ds = COCO(cfg, task="validation", device="cpu")
    assert len(ds) == 2 and all(n.startswith("im") for n in ds.samples["names"])
    img, name = ds.decode(0)
    assert img.dtype == torch.uint8 and tuple(img.shape) == (20, 30) and name in ("im0", "im1", "im2", "im3")
    with pytest.raises(NotImplementedError):
        COCO(dict(cfg, has_labels="outputs/x"), task="training")


def test_packed_label_reader(tmp_path):
    from superpoint_nerf_pytorch_b200.engine_solvers.export import load_packed_labels
    a, b, c = np.array([[1, 2], [3, 4]], np.int32), np.zeros((0, 2), np.int32), np.array([[7, 8]], np.int32)
    np.savez(tmp_path / "packed_rank000.npz", names=np.array(["x", "y"]), keypoints=np.concatenate([a, b]), offsets=np.array([0, 2, 2]),
             global_offset=np.array(0))
    np.savez(tmp_path / "packed_rank001.npz", names=np.array(["z"]), keypoints=c, offsets=np.array([0, 1]), global_offset=np.array(2))
    got = load_packed_labels(tmp_path)
    assert sorted(got) == ["x", "y", "z"] and np.array_equal(got["x"], a) and got["y"].shape == (0, 2) and got["z"].dtype == np.int64


def test_nerf_point_reprojection_mirror_matches_the_oracle(golden):
    """data/data_utils/kp_utils.warp_points_NeRF (5x5 depth rule evaluated with pooling instead of the reference's
    per-point Python loop) and filter_points on CPU tensors: bit-equal to the oracle restatement, which
    tests/test_oracle_golden.py pins to the unmodified reference's ExportNeRFDetections.step."""
    import torch
    from conftest import make_nerf_batch
    from oracle import eval_oracle as EO
    from superpoint_nerf_pytorch_b200.data.data_utils.kp_utils import filter_points, warp_points_NeRF
    rng = np.random.RandomState(2)
    for seed, nv, j, k in ((0, 4, 1, 3), (1, 5, 0, 2)):
        bt = make_nerf_batch(seed, n_views=nv)
        raw = bt["raw"]
        h, w = raw["input_depth"].shape[-2:]
        pts = torch.from_numpy(np.unique(np.stack([rng.randint(0, h, 300), rng.randint(0, w, 300)], 1), axis=0))   # incl. borders
        got = warp_points_NeRF(pts.to(torch.float32), raw["input_depth"][k][None], bt["camera_intrinsic_matrix"][j][None],
                               raw["input_rotation"][k][None], raw["input_translation"][k][None], raw["input_rotation"][j][None],
                               raw["input_translation"][j][None]).reshape(-1, 2)
        want = EO.nerf_reproject_points(pts, raw["input_depth"][k], bt["camera_intrinsic_matrix"][j], raw["input_rotation"][k],
                                        raw["input_translation"][k], raw["input_rotation"][j], raw["input_translation"][j])
        assert torch.equal(got, want)
        kept, mask = filter_points(got, (h, w), return_mask=True)
        ok = (want[:, 0] >= 0) & (want[:, 0] < h - 1) & (want[:, 1] >= 0) & (want[:, 1] < w - 1)
        assert torch.equal(mask, ok) and torch.equal(kept, want[ok]) and 0 < int(ok.sum()) < len(pts)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (CPU): one JSON line with the native arm's metric / unit / config, exactly the
    requested steps and warm-up, cpu_baseline describing the run and an e2e object with zero copies; ranks other than 0
    print nothing."""
    import json
    import os
    import subprocess
    import sys
    import types
    from conftest import ROOT
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1", "--ref-budget-s", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, WORLD_SIZE="2", RANK="0"))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pseudo-label img/s (240x320, 100 H)" and d["unit"] == "img/s"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 2 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "2 timed steps (+1 warm-up)" in d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    sys.path.insert(0, str(ROOT))
    import bench
    args = types.SimpleNamespace(images_per_step=128, precision="f16", streams=1)
    assert d["config"] == bench.workload_config(args, 2)          # the same object the native arm prints
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=120, cwd=ROOT, env=dict(os.environ, WORLD_SIZE="2", RANK="1"))
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_bench_rejects_arguments_it_cannot_honour():
    """No step count is silently changed: --steps 0 or a negative --warmup is an argument error (exit 2, no JSON line),
    as is --dump-outputs with the reference arm, which has no native outputs to write."""
    import subprocess
    import sys
    from conftest import ROOT
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--steps", "0"],
                  ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and not [l for l in out.stdout.splitlines() if l.startswith("{")], (extra, out.stderr[-500:])


def test_cabi_rejects_null_context_without_a_gpu(built_lib):
    """Error behaviour at the boundary (include/spn_b200.h: 'return 0 or a negative SPN_E_* code with spn_last_error()'):
    every entry point called with a NULL context and zeroed arguments returns a negative code and sets a message - no
    crash, no CUDA call needed.  Runs in a child process so that a null dereference could not take pytest down."""
    import subprocess
    import sys
    from conftest import ROOT
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
skip = {"spn_last_error", "spn_version", "spn_create", "spn_destroy", "spn_launch_count"}
n = 0
for name, (res, args) in N.PROTOTYPES.items():
    if name in skip:
        continue
    vals = [None if (a in (C.c_void_p, C.c_char_p) or hasattr(a, "contents")) else a(0) for a in args]
    rc = getattr(lib, name)(*vals)
    msg = lib.spn_last_error().decode()
    assert rc < 0 and msg, (name, rc, msg)
    n += 1
assert lib.spn_launch_count(None) == -1 and lib.spn_destroy(None) == 0 and lib.spn_version() >= 100
print("checked", n)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "checked 26" in out.stdout, out.stdout


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_bench_native_arm_fails_loudly_without_a_gpu():
    """`python bench.py` (native arm) must not produce a number on a machine without a GPU: non-zero exit, no JSON line
    (a silent CPU or library fallback would print one)."""
    import subprocess
    import sys
    from conftest import ROOT
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]
