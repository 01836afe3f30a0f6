"""COCO image dataset for the export tasks, with the reference's class interface (data/COCO.py:14-139).

Export configuration only (``has_labels: False``, no augmentation, no warped pair - what
``configs/magicpoint_coco_export.yaml`` selects); the training-time branches of the reference class (labels,
photometric / homographic augmentation, warped pairs) are outside this package and rejected.  What differs underneath:
``read_image`` decodes to uint8 on a host thread (torchvision's decoder, as the reference) and everything after the
decode - bilinear ratio-preserving resize, centre crop, /255 - is ONE kernel (spn_resize_crop) on the uint8 image.
``decode`` / ``finish`` split ``__getitem__`` so that a prefetching loader can run the decodes on worker threads.

``data.decode: device`` (default ``host``) moves the JPEG decode to the GPU: the worker threads read the file and parse
its headers, a file the device decoder does not take (progressive, CMYK, not a JPEG, ...) is decoded on the host right
there, and ``finish_batch`` decodes the rest in batches (preprocessing.launch_jpeg_decode / finish_jpeg_decode).  The pixels are
bit-identical to the host decode, so the items do not depend on the mode; a file whose entropy data the device decoder
rejects is decoded on the host before it is returned.
"""
from pathlib import Path

import numpy as np
import torch
from torch.utils.data import Dataset

from .. import settings
from .._native import JPEG_OK, jpeg_plan
from .preprocessing import finish_jpeg_decode, launch_jpeg_decode, pin_host as _pin, ratio_preserving_resize


class _JpegFile:
    """File bytes left for the device decoder (COCO.decode in ``decode: device`` mode)."""
    __slots__ = ("data",)

    def __init__(self, data):
        self.data = data


class COCO(Dataset):
    def __init__(self, data_config, task="training", device="cuda") -> None:
        super().__init__()
        self.config = data_config
        self.device = device
        if torch.cuda.is_available() and torch.device(device).type == "cuda" and torch.device(device).index is None:
            self.device = f"cuda:{torch.cuda.current_device()}"   # resolved here: decode threads start with device 0 current
        self.action = "training" if task == "training" else "validation" if task == "validation" else "test"
        aug = data_config.get("augmentation", {})
        if data_config.get("has_labels") or data_config.get("warped_pair") or any(aug.get(k, {}).get("enable") for k in aug):
            raise NotImplementedError("the B200 COCO loader serves the export tasks (has_labels / warped_pair / augmentation "
                                      "are training-time features of the reference)")
        self.decode_mode = data_config.get("decode", "host")
        if self.decode_mode not in ("host", "device"):
            raise ValueError(f"data.decode must be 'host' or 'device', got {self.decode_mode!r}")
        if self.decode_mode == "device":
            self.finish_batch = self._finish_batch          # PrefetchLoader's batched device stage
        self.samples = self._init_dataset()

    def _init_dataset(self):
        """List of image paths and names (COCO.py:34-56)."""
        data_dir = Path(settings.DATA_PATH, self.config["name"], "images", self.action)
        image_paths = list(data_dir.iterdir())
        if self.config.get("truncate"):
            image_paths = image_paths[:int(self.config["truncate"] * len(image_paths))]
        return {"image_paths": [str(p) for p in image_paths], "names": [p.stem for p in image_paths]}

    def __len__(self):
        return len(self.samples["image_paths"])

    def read_image(self, image):
        """COCO.py:61-64, stopping at the decoded uint8 (H0,W0) image (the float conversion is fused into the resize)."""
        import torchvision
        data = torchvision.io.read_file(image)
        return _pin(torchvision.io.decode_image(data, torchvision.io.ImageReadMode.GRAY).squeeze(0), self.device)

    def ratio_preserving_resize(self, image, normalize=False):
        """COCO.py:66-76 on the device: (H0,W0) uint8 / fp32 -> (H,W) fp32."""
        # host images are uploaded by the module function on its side stream (never on the consumer's stream)
        return ratio_preserving_resize(image, self.config["preprocessing"]["resize"], normalize=normalize, device=self.device)

    def decode(self, index):
        """Host part of ``__getitem__`` (thread-safe): -> (uint8 image, name); in device mode the image is a _JpegFile
        when the device decoder takes the file."""
        path, name = self.samples["image_paths"][index], self.samples["names"][index]
        if self.decode_mode == "device":
            data = np.fromfile(path, dtype=np.uint8)
            if int(jpeg_plan(data, np.array([0, data.size], np.int64))[1][0, 0]) == JPEG_OK:
                return _JpegFile(data), name
            return self._host_decode(data), name
        return self.read_image(path), name

    def _host_decode(self, data):
        """read_image on bytes already read."""
        import torchvision
        return _pin(torchvision.io.decode_image(torch.from_numpy(data), torchvision.io.ImageReadMode.GRAY).squeeze(0), self.device)

    def finish(self, decoded):
        """Device part: resize + crop + /255 (COCO.py:89-90,135) -> the reference's item dictionary."""
        image, name = decoded
        if isinstance(image, _JpegFile):
            return next(self._finish_batch([decoded]))
        return {"raw": {"image": self.ratio_preserving_resize(image, normalize=True)}, "name": name}

    def _finish_batch(self, items):
        """``finish`` of several items in order, with one device JPEG decode for all the _JpegFile items among them.  The
        decode is launched here; the returned generator waits for it and yields the finished items one by one, so an
        item whose host re-decode raises lets every item before it through first, as in host mode."""
        idx = [k for k, (image, _) in enumerate(items) if isinstance(image, _JpegFile)]
        handle = launch_jpeg_decode([items[k][0].data for k in idx], device=self.device) if idx else None
        return self._finished(items, idx, handle)

    def _finished(self, items, idx, handle):
        imgs = dict(zip(idx, finish_jpeg_decode(handle, self.config["preprocessing"]["resize"]))) if handle else {}
        for k, (image, name) in enumerate(items):
            if k not in imgs:
                yield self.finish((image, name))
            elif imgs[k] is not None:
                yield {"raw": {"image": imgs[k]}, "name": name}
            else:                                             # entropy data the device decoder rejected
                yield self.finish((self._host_decode(image.data), name))

    def __getitem__(self, index):
        return self.finish(self.decode(index))

    def batch_collator(self, batch):
        """COCO.py:140-147 for label-free items."""
        assert len(batch) > 0 and isinstance(batch[0], dict)
        return {"raw": {"image": torch.stack([item["raw"]["image"].unsqueeze(0) for item in batch])},
                "name": [item["name"] for item in batch]}
