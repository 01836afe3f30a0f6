"""A folder of images for feature matching (matching.py): every ``.png``, ``.jpg`` and ``.jpeg`` file under
``<DATA_PATH>/<data.name>/``, in subdirectories too, sorted by the relative POSIX path, which is also the image's name.

Images are decoded to grayscale (colour images are converted) with the same decoder as data/PosedViews.py.  With
``data.preprocessing.resize: [H, W]`` (multiples of 8) every image goes through ``preprocessing.ratio_preserving_resize``
on the GPU; without it, an image whose size is not a multiple of 8 raises ValueError naming the file.
"""
from pathlib import Path

import numpy as np
import torch
from torch.utils.data import Dataset

from .. import settings
from .PosedViews import IMAGE_EXTENSIONS, read_image
from .preprocessing import ratio_preserving_resize, resize_geometry


class ImageFolder(Dataset):
    def __init__(self, data_config, device="cuda") -> None:
        super().__init__()
        self.device = device
        resize = (data_config.get("preprocessing") or {}).get("resize")
        if resize is not None:
            if (not isinstance(resize, (list, tuple)) or len(resize) != 2
                    or not all(isinstance(v, int) and not isinstance(v, bool) and v > 0 and v % 8 == 0 for v in resize)):
                raise ValueError(f"data.preprocessing.resize: expected [H, W], positive multiples of 8, got {resize!r}")
            resize = (int(resize[0]), int(resize[1]))
        self.resize = resize
        self.root = Path(settings.DATA_PATH, data_config["name"])
        if not self.root.is_dir():
            raise ValueError(f"{self.root}: no such image folder")
        paths = [p for p in self.root.rglob("*") if p.is_file() and p.suffix.lower() in IMAGE_EXTENSIONS]
        self.names = sorted(p.relative_to(self.root).as_posix() for p in paths)
        if not self.names:
            raise ValueError(f"{self.root}: no {'/'.join(IMAGE_EXTENSIONS)} images")

    def __len__(self):
        return len(self.names)

    def __getitem__(self, index):
        """-> {"name", "image": (H, W) uint8 numpy as decoded, "shape": (H0, W0), "geometry": (new_h, new_w, crop_top,
        crop_left) of the resize or None}."""
        path = self.root / self.names[index]
        img = read_image(path)
        H, W = img.shape
        if self.resize is None:
            if H % 8 or W % 8:
                raise ValueError(f"{path}: size {H}x{W} is not a multiple of 8 (set data.preprocessing.resize)")
            geometry = None
        else:
            geometry = resize_geometry((H, W), self.resize)
        return {"name": self.names[index], "image": img, "shape": (H, W), "geometry": geometry}

    def network_input(self, item):
        """(H, W) fp32 CUDA image / 255 at the network's input size."""
        if self.resize is None:
            return torch.from_numpy(item["image"].astype(np.float32) / np.float32(255.0)).to(self.device)
        return ratio_preserving_resize(torch.from_numpy(item["image"]), self.resize, device=self.device)
