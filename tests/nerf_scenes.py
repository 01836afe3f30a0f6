"""Posed-view scene trees in the layout of data/PosedViews.py, written from conftest.make_nerf_batch (shared by the CPU
dataset tests and the GPU export tests)."""
import json
from pathlib import Path

import numpy as np

from conftest import make_nerf_batch


def write_scene(root, scene, seed, n_views, h=64, w=96, shared_K=True, ext=".png"):
    """One scene directory from make_nerf_batch(seed, n_views, h, w); frames are named f000, f001, ... Returns the batch
    (images as written: uint8-rounded / 255)."""
    import cv2
    bt = make_nerf_batch(seed, n_views=n_views, h=h, w=w)
    d = Path(root, scene)
    (d / "images").mkdir(parents=True, exist_ok=True)
    (d / "depth").mkdir(parents=True, exist_ok=True)
    frames, imgs = [], []
    K = bt["camera_intrinsic_matrix"].numpy()
    for i in range(n_views):
        name = f"f{i:03d}"
        img = np.round(bt["raw"]["image"][i, 0].numpy() * 255.0).astype(np.uint8)
        cv2.imwrite(str(d / "images" / f"{name}{ext}"), img)
        imgs.append(img.astype(np.float32) / np.float32(255.0))
        np.save(d / "depth" / f"{name}.npy", bt["raw"]["input_depth"][i].numpy())
        fr = {"name": name, "R": bt["raw"]["input_rotation"][i].numpy().tolist(),
              "t": bt["raw"]["input_translation"][i].numpy().reshape(3).tolist()}
        if not shared_K:
            fr["K"] = K[i].tolist()
        frames.append(fr)
    cams = {"frames": frames}
    if shared_K:
        cams["K"] = K[0].tolist()
    (d / "cameras.json").write_text(json.dumps(cams))
    bt["written_image"] = np.stack(imgs)[:, None]
    bt["frame_names"] = [f"{scene}_f{i:03d}" for i in range(n_views)]
    return bt


def write_tree(data_path, name="PosedViews", split="training", scenes=(("sceneA", 0, 5), ("sceneB", 1, 3), ("sceneC", 2, 4)),
               h=64, w=96):
    """A split directory with several scenes -> {scene: batch}."""
    root = Path(data_path, name, split)
    return {s: write_scene(root, s, seed, nv, h, w, shared_K=(k % 2 == 0)) for k, (s, seed, nv) in enumerate(scenes)}
