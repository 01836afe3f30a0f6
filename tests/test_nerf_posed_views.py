"""export_NeRF_labels without a GPU: the PosedViews dataset (layout, chunking, order, sharding, error cases), the loader
and CLI wiring, and the C ABI of include/spn_nerf.h."""
import json
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from nerf_scenes import write_scene, write_tree


def _dataset(tmp_path, monkeypatch, batch_size=2, resize=(64, 96), split="training"):
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.data.PosedViews import PosedViews
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path))
    cfg = {"name": "PosedViews", "class_name": "PosedViews", "batch_size": batch_size,
           "preprocessing": {"resize": list(resize) if resize else None}}
    return PosedViews(cfg, task=split, device="cpu")


def test_items_hold_what_was_written(tmp_path, monkeypatch):
    scenes = write_tree(tmp_path)
    ds = _dataset(tmp_path, monkeypatch, batch_size=8)
    assert len(ds) == 3
    for item, (scene, bt) in zip((ds[i] for i in range(3)), sorted(scenes.items())):
        raw = item["raw"]
        V = len(bt["name"])
        assert set(item) == {"raw", "camera_intrinsic_matrix", "name"}
        assert set(raw) == {"image", "input_depth", "input_rotation", "input_translation"}
        shapes = {"image": (V, 1, 64, 96), "input_depth": (V, 64, 96), "input_rotation": (V, 3, 3), "input_translation": (V, 3, 1)}
        for k, shp in shapes.items():
            assert raw[k].dtype == torch.float32 and tuple(raw[k].shape) == shp, (k, raw[k].dtype, raw[k].shape)
        assert item["camera_intrinsic_matrix"].dtype == torch.float32 and tuple(item["camera_intrinsic_matrix"].shape) == (V, 3, 3)
        assert np.array_equal(raw["image"].numpy(), bt["written_image"])
        for k in ("input_depth", "input_rotation", "input_translation"):
            assert np.array_equal(raw[k].numpy().view(np.uint32), bt["raw"][k].numpy().view(np.uint32)), k   # bit-equal
        assert np.array_equal(item["camera_intrinsic_matrix"].numpy().view(np.uint32), bt["camera_intrinsic_matrix"].numpy().view(np.uint32))
        assert item["name"] == bt["frame_names"]


def test_chunks_follow_frames_order_and_never_cross_scenes(tmp_path, monkeypatch):
    write_tree(tmp_path)                                        # scenes of 5, 3 and 4 frames
    ds = _dataset(tmp_path, monkeypatch, batch_size=2)
    names = [ds[i]["name"] for i in range(len(ds))]
    assert names == [["sceneA_f000", "sceneA_f001"], ["sceneA_f002", "sceneA_f003"], ["sceneA_f004"],
                     ["sceneB_f000", "sceneB_f001"], ["sceneB_f002"], ["sceneC_f000", "sceneC_f001"], ["sceneC_f002", "sceneC_f003"]]
    assert [len(c) for c in (ds[i]["raw"]["input_depth"] for i in range(len(ds)))] == [2, 2, 1, 2, 1, 2, 2]
    # frames come in the order cameras.json lists them, not in file-name order
    cams_path = tmp_path / "PosedViews" / "training" / "sceneB" / "cameras.json"
    cams = json.loads(cams_path.read_text())
    cams["frames"] = cams["frames"][::-1]
    cams_path.write_text(json.dumps(cams))
    ds = _dataset(tmp_path, monkeypatch, batch_size=3)
    assert ds[2]["name"] == ["sceneB_f002", "sceneB_f001", "sceneB_f000"]


def test_loader_serves_chunks_in_order_and_shards_by_rank(tmp_path, monkeypatch):
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.utils.data_loaders import get_loader
    write_tree(tmp_path)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path))
    cfg = {"data": {"name": "PosedViews", "class_name": "PosedViews", "batch_size": 2, "preprocessing": {"resize": [64, 96]},
                    "loader_workers": 3}}
    every = [b["name"] for b in get_loader(cfg, "export_NeRF_labels", device="cpu", export_split="training")]
    assert len(every) == 7 and every[0] == ["sceneA_f000", "sceneA_f001"] and every[-1] == ["sceneC_f002", "sceneC_f003"]
    parts = [[b["name"] for b in get_loader(cfg, "export_NeRF_labels", device="cpu", export_split="training", rank=r, world=3)]
             for r in range(3)]
    assert parts == [every[r::3] for r in range(3)]
    assert len(get_loader(cfg, "export_NeRF_labels", device="cpu", export_split="training", rank=1, world=3)) == 2


def _expect(ds_or_fn, path_part):
    with pytest.raises(ValueError) as e:
        ds_or_fn()
    assert path_part in str(e.value), str(e.value)
    return str(e.value)


def test_errors_name_the_file(tmp_path, monkeypatch):
    import cv2
    root = tmp_path / "PosedViews" / "training"
    write_scene(root, "s", 3, 4)
    scene = root / "s"
    # preprocessing.resize different from the stored size
    _expect(lambda: _dataset(tmp_path, monkeypatch, resize=(64, 88))[0], str(scene / "images" / "f000.png"))
    # no resize key at all: the stored size is taken as is
    assert tuple(_dataset(tmp_path, monkeypatch, resize=None)[0]["raw"]["image"].shape) == (2, 1, 64, 96)
    # mixed sizes within a chunk
    cv2.imwrite(str(scene / "images" / "f001.png"), np.zeros((56, 96), np.uint8))
    np.save(scene / "depth" / "f001.npy", np.ones((56, 96), np.float32))
    msg = _expect(lambda: _dataset(tmp_path, monkeypatch, resize=None)[0], str(scene / "images" / "f001.png"))
    assert "other views" in msg
    # a size that is not a multiple of 8
    cv2.imwrite(str(scene / "images" / "f001.png"), np.zeros((60, 96), np.uint8))
    np.save(scene / "depth" / "f001.npy", np.ones((60, 96), np.float32))
    assert "multiple of 8" in _expect(lambda: _dataset(tmp_path, monkeypatch, resize=None)[0], str(scene / "images" / "f001.png"))
    cv2.imwrite(str(scene / "images" / "f001.png"), np.zeros((64, 96), np.uint8))
    # mis-shaped and mistyped depth
    np.save(scene / "depth" / "f001.npy", np.ones((64, 95), np.float32))
    _expect(lambda: _dataset(tmp_path, monkeypatch)[0], str(scene / "depth" / "f001.npy"))
    np.save(scene / "depth" / "f001.npy", np.ones((64, 96), np.float64))
    _expect(lambda: _dataset(tmp_path, monkeypatch)[0], str(scene / "depth" / "f001.npy"))
    np.save(scene / "depth" / "f001.npy", np.ones((64, 96), np.float32))
    assert len(_dataset(tmp_path, monkeypatch)[0]["name"]) == 2
    # missing depth file, missing image
    (scene / "depth" / "f003.npy").rename(scene / "depth" / "moved.npy")
    _expect(lambda: _dataset(tmp_path, monkeypatch), str(scene / "depth" / "f003.npy"))
    (scene / "depth" / "moved.npy").rename(scene / "depth" / "f003.npy")
    (scene / "images" / "f002.png").unlink()
    _expect(lambda: _dataset(tmp_path, monkeypatch), str(scene / "images" / "f002"))
    cv2.imwrite(str(scene / "images" / "f002.png"), np.zeros((64, 96), np.uint8))
    assert len(_dataset(tmp_path, monkeypatch)) == 2
    # malformed camera entries
    cams_path = scene / "cameras.json"
    good = json.loads(cams_path.read_text())
    bad_cases = [
        dict(good, frames=[dict(good["frames"][0], R=[[1, 0], [0, 1]])] + good["frames"][1:]),      # R not 3x3
        dict(good, frames=[dict(good["frames"][0], t=[0.0, "x", 1.0])] + good["frames"][1:]),         # t not numeric
        dict(good, frames=[{k: v for k, v in good["frames"][0].items() if k != "t"}] + good["frames"][1:]),   # no t
        dict(good, frames=[{"R": good["frames"][0]["R"], "t": good["frames"][0]["t"]}] + good["frames"][1:]),  # no name
        {"frames": good["frames"]},                                                                  # no K anywhere
        dict(good, K=[[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, float("nan")]]),                 # non-finite K
        {"K": good["K"]},                                                                            # no frames
    ]
    for case in bad_cases:
        cams_path.write_text(json.dumps(case))
        _expect(lambda: _dataset(tmp_path, monkeypatch), str(cams_path))
    cams_path.write_text("{not json")
    _expect(lambda: _dataset(tmp_path, monkeypatch), str(cams_path))
    cams_path.write_text(json.dumps(good))
    assert len(_dataset(tmp_path, monkeypatch)) == 2


def test_cabi_exports_the_nerf_fuse_symbol(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_nerf.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.NERF_PROTOTYPES) == ["spn_nerf_fuse"]
    assert not set(N.NERF_PROTOTYPES) & (set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES))
    assert hasattr(ctypes.CDLL(str(built_lib)), "spn_nerf_fuse")


def test_nerf_fuse_rejects_null_arguments(built_lib):
    """NULL context and zero arguments -> a negative code and a message, no CUDA call (child process)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
for name, (res, args) in N.NERF_PROTOTYPES.items():
    rc = getattr(lib, name)(*[None if a in (C.c_void_p, C.c_char_p) else a(0) for a in args])
    msg = lib.spn_last_error().decode()
    assert rc == -1 and "null pointer" in msg, (name, rc, msg)
print("checked", len(N.NERF_PROTOTYPES))
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 1" in out.stdout, out.stderr[-2000:]


@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_cli_dispatches_export_nerf_labels(tmp_path):
    """export_NeRF_labels gets past dispatch (it used to be rejected there) and stops where every export task stops on a
    machine without a GPU; train is still rejected at dispatch."""
    import tyro
    from superpoint_nerf_pytorch_b200 import engine
    cfg = tmp_path / "nerf.yaml"
    cfg.write_text((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "magicpoint_nerf_export.yaml").read_text())
    with pytest.raises(SystemExit) as e:
        tyro.cli(engine.main, use_underscores=True, args=["--config_path", str(cfg), "--task", "export_NeRF_labels"])
    assert "CUDA is not available" in str(e.value)
    with pytest.raises(SystemExit) as e:
        tyro.cli(engine.main, use_underscores=True, args=["--config_path", str(cfg), "--task", "train"])
    assert "outside the B200 hot path" in str(e.value)
