"""Posed multi-view scenes for ``export_NeRF_labels``: images, per-pixel ray depth and camera poses in this package's own
on-disk layout (not the reference's NeRF dataset layout, which this package does not read).

Layout, under ``<DATA_PATH>/<data.name>/<split>/``, one directory per scene (scenes in sorted order)::

    <scene>/images/<frame>.png | .jpg | .jpeg   grayscale after decoding (colour images are converted), divided by 255
    <scene>/depth/<frame>.npy                   float32 (H, W): the DISTANCE ALONG THE PIXEL'S RAY, not z-depth
                                                (warp_points_NeRF scales the unit ray K^-1 (x, y, 1) / |.| by it)
    <scene>/cameras.json                        {"K": 3x3 (shared, optional),
                                                 "frames": [{"name": <frame>, "R": 3x3, "t": 3 or 3x1, "K": 3x3 (optional)}]}

``R`` and ``t`` are camera-to-world in OpenCV axes (x right, y down, z forward): ``X_world = R X_cam + t``.  A frame
takes its own ``K`` if it has one, else the shared one.

One item is a chunk of up to ``data.batch_size`` consecutive frames of one scene, in ``frames`` order; chunks never
cross scenes.  The item is the dictionary ExportNeRFDetections consumes::

    {"raw": {"image": (V,1,H,W), "input_depth": (V,H,W), "input_rotation": (V,3,3), "input_translation": (V,3,1)},
     "camera_intrinsic_matrix": (V,3,3), "name": [<scene>_<frame>, ...]}      all float32 CPU tensors

Nothing is resized: resizing would have to rescale K and the depth maps too.  A ``preprocessing.resize`` that differs
from the stored size, an image size that is not a multiple of 8, mixed sizes in a chunk, a missing or mis-shaped depth
file and a malformed camera entry raise ValueError naming the file.
"""
import json
from pathlib import Path

import numpy as np
import torch
from torch.utils.data import Dataset

from .. import settings

IMAGE_EXTENSIONS = (".png", ".jpg", ".jpeg")


def _matrix(value, shape, where):
    try:
        m = np.asarray(value, dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError(f"{where}: expected a {shape[0]}x{shape[1]} matrix of numbers, got {value!r}") from None
    if m.size != shape[0] * shape[1] or not np.isfinite(m).all():
        raise ValueError(f"{where}: expected {shape[0] * shape[1]} finite numbers for a {shape[0]}x{shape[1]} matrix, "
                         f"got {value!r}")
    return m.reshape(shape).astype(np.float32)


def read_image(path):
    """-> (H, W) uint8 grayscale (colour images are converted); ValueError naming the file if it cannot be decoded."""
    import cv2
    img = cv2.imread(str(path), cv2.IMREAD_GRAYSCALE)
    if img is None:
        raise ValueError(f"{path}: cannot be decoded as an image")
    if img.dtype != np.uint8:
        raise ValueError(f"{path}: expected 8-bit samples, got {img.dtype}")
    return img


class PosedViews(Dataset):
    def __init__(self, data_config, task="training", device="cuda") -> None:
        super().__init__()
        self.config = data_config
        self.device = device
        self.split = task
        self.chunk = int(data_config.get("batch_size", 1) or 1)
        if self.chunk < 1:
            raise ValueError(f"data.batch_size must be >= 1, got {data_config.get('batch_size')!r}")
        resize = (data_config.get("preprocessing") or {}).get("resize")
        self.resize = tuple(int(v) for v in resize) if resize else None
        self.root = Path(settings.DATA_PATH, data_config["name"], self.split)
        self.items = self._init_dataset()

    def _scene_frames(self, scene):
        """-> list of frame records of one scene, validated against the files."""
        cam_path = scene / "cameras.json"
        try:
            cams = json.loads(cam_path.read_text())
        except FileNotFoundError:
            raise ValueError(f"{cam_path}: missing") from None
        except json.JSONDecodeError as e:
            raise ValueError(f"{cam_path}: not valid JSON ({e})") from None
        if not isinstance(cams, dict) or not isinstance(cams.get("frames"), list):
            raise ValueError(f"{cam_path}: expected an object with a 'frames' list")
        shared_K = _matrix(cams["K"], (3, 3), f"{cam_path}: 'K'") if "K" in cams else None
        frames = []
        for i, fr in enumerate(cams["frames"]):
            where = f"{cam_path}: frames[{i}]"
            if not isinstance(fr, dict) or not isinstance(fr.get("name"), str) or not fr["name"]:
                raise ValueError(f"{where}: expected an object with a non-empty 'name'")
            name = fr["name"]
            for key in ("R", "t"):
                if key not in fr:
                    raise ValueError(f"{where} ({name}): missing '{key}'")
            if "K" not in fr and shared_K is None:
                raise ValueError(f"{where} ({name}): no 'K' for this frame and no shared 'K'")
            K = _matrix(fr["K"], (3, 3), f"{where} ({name}): 'K'") if "K" in fr else shared_K
            R = _matrix(fr["R"], (3, 3), f"{where} ({name}): 'R'")
            t = _matrix(fr["t"], (3, 1), f"{where} ({name}): 't'")
            images = [scene / "images" / f"{name}{ext}" for ext in IMAGE_EXTENSIONS if (scene / "images" / f"{name}{ext}").is_file()]
            if len(images) != 1:
                raise ValueError(f"{scene / 'images' / name}.{{png,jpg,jpeg}}: expected exactly one image for frame "
                                 f"'{name}' of {cam_path}, found {len(images)}")
            depth = scene / "depth" / f"{name}.npy"
            if not depth.is_file():
                raise ValueError(f"{depth}: missing depth file for frame '{name}' of {cam_path}")
            frames.append({"name": f"{scene.name}_{name}", "image": images[0], "depth": depth, "K": K, "R": R, "t": t})
        return frames

    def _init_dataset(self):
        if not self.root.is_dir():
            raise ValueError(f"{self.root}: no such split directory")
        items, seen = [], {}
        for scene in sorted(p for p in self.root.iterdir() if p.is_dir()):
            frames = self._scene_frames(scene)
            for fr in frames:
                if fr["name"] in seen:
                    raise ValueError(f"{fr['image']}: output name '{fr['name']}' is also the name of {seen[fr['name']]}")
                seen[fr["name"]] = fr["image"]
            items += [frames[s:s + self.chunk] for s in range(0, len(frames), self.chunk)]
        return items

    def __len__(self):
        return len(self.items)

    def __getitem__(self, index):
        """Host only (thread-safe): decode and check one chunk -> the item dictionary (CPU tensors)."""
        images, depths, shape = [], [], None
        for fr in self.items[index]:
            img = read_image(fr["image"])
            H, W = img.shape
            if H % 8 or W % 8:
                raise ValueError(f"{fr['image']}: size {H}x{W} is not a multiple of 8")
            if self.resize is not None and (H, W) != self.resize:
                raise ValueError(f"{fr['image']}: size {H}x{W} differs from preprocessing.resize {list(self.resize)} "
                                 "(views are not resized: K and the depth maps would have to be rescaled too)")
            if shape is not None and (H, W) != shape:
                raise ValueError(f"{fr['image']}: size {H}x{W} differs from {shape[0]}x{shape[1]} of the other views "
                                 "of its chunk")
            shape = (H, W)
            try:
                depth = np.load(fr["depth"], allow_pickle=False)
            except (OSError, ValueError) as e:
                raise ValueError(f"{fr['depth']}: cannot be read as .npy ({e})") from None
            if depth.dtype != np.float32 or depth.shape != (H, W):
                raise ValueError(f"{fr['depth']}: expected float32 {(H, W)} (the image's shape), got {depth.dtype} {depth.shape}")
            images.append(img)
            depths.append(depth)
        frames = self.items[index]
        return {"raw": {"image": torch.from_numpy(np.stack(images).astype(np.float32)[:, None] / np.float32(255.0)),
                        "input_depth": torch.from_numpy(np.stack(depths)),
                        "input_rotation": torch.from_numpy(np.stack([f["R"] for f in frames])),
                        "input_translation": torch.from_numpy(np.stack([f["t"] for f in frames]))},
                "camera_intrinsic_matrix": torch.from_numpy(np.stack([f["K"] for f in frames])),
                "name": [f["name"] for f in frames]}

    def batch_collator(self, batch):
        """One chunk per batch: the chunk's dictionary as is."""
        if len(batch) != 1:
            raise ValueError("PosedViews items are whole chunks of views: load them with batch size 1")
        return batch[0]
