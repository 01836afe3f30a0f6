"""CLI with the reference's task names and flags (engine.py:43-208), export tasks only.

    python -m superpoint_nerf_pytorch_b200.engine --config_path configs/magicpoint_coco_export.yaml \
        --task export_pseudo_labels [--pseudo_labels.split training] [--pseudo_labels.enable_Homography_Adaptation True]

Same YAML schema as the reference (``data``, ``homography_adaptation``, ``model``, ``pretrained``).  What differs:
  * ``model.script`` / ``model.class_name`` resolve inside this package (models/SuperPoint.py), so an unmodified
    reference config selects the B200 implementation;
  * ``get_loader`` is this package's (utils/data_loaders.py): the reference's COCO / HPatches dataset classes mirrored for
    the export tasks, decoding on host threads and resizing on the GPU; ``--synthetic N`` feeds N synthetic images of
    the configured size instead;
  * ``export_NeRF_labels`` reads posed multi-view scenes in this package's own layout (data/PosedViews.py, config
    ``configs/magicpoint_nerf_export.yaml``, not the reference's NeRF dataset layout) and runs ExportNeRFDetections;
  * ``train`` is out of scope: its flags (``--training.*``) parse exactly as in the reference, the task itself is
    rejected at dispatch;
  * under ``torchrun`` (WORLD_SIZE > 1) every rank selects ``cuda:LOCAL_RANK``, joins the NCCL process group and takes
    the dataset items with index = rank (mod world): no two ranks write the same file (SURVEY.md section 8e).
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from pathlib import Path
from typing import Literal

import torch
import tyro
import yaml

from . import settings
from .engine_solvers.export import (Export_Hpatches_Descriptors, Export_Hpatches_Repeatability, ExportDetections,
                                   ExportNeRFDetections)
from .utils.get_model import get_model
from .utils.sharding import shard_indices


@dataclass
class options:
    """Training options (engine.py:14-28 of the reference; parsed for command-line compatibility, training itself is
    outside this package).

    Args:
        validate_training: Validate during training.
        include_mask_loss: Apply mask or no mask during loss (Do not include bordering artifacts by applying mask).
        nerf_loss: Whether to use Descriptor NeRF loss or normal SuperPoint Descriptor loss.
        train_nerf: Whether to enable training of NeRF datasets (Multiple datasets can be used for training)
    """
    validate_training: bool = False
    include_mask_loss: bool = True
    nerf_loss: bool = False
    train_nerf: bool = False


@dataclass
class export_pseudo_labels_split:
    """Export pseudo labels on train, validation or test split.

    Args:
        enable_Homography_Adaptation: Enable homography adaptation during export.
        split: The split to export pseudo labels on.
    """
    enable_Homography_Adaptation: bool = True
    split: Literal["training", "validation", "test"] = "training"


class ShardedLoader:
    """Rank-strided view of any loader that yields one item per batch: item i goes to rank i % world.  Used for the
    reference's DataLoaders under torchrun (a DataLoader cannot be re-sharded after construction); items of other ranks
    are skipped after loading, which costs host time only."""

    def __init__(self, loader, rank, world):
        self.loader, self.rank, self.world = loader, rank, world

    def __len__(self):
        n = len(self.loader)
        return (n - self.rank + self.world - 1) // self.world

    def __iter__(self):
        for i, item in enumerate(self.loader):
            if i % self.world == self.rank:
                yield item


def init_distributed():
    """-> (rank, world, device).  One process per GPU: cuda:LOCAL_RANK; NCCL group when WORLD_SIZE > 1."""
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        if local >= torch.cuda.device_count():
            raise SystemExit(f"LOCAL_RANK {local} but only {torch.cuda.device_count()} CUDA devices are visible")
        torch.cuda.set_device(local)
        if not torch.distributed.is_initialized():
            torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, f"cuda:{torch.cuda.current_device()}"


class SyntheticLoader:
    """Stand-in for the reference loaders: yields the batch dictionaries the export tasks consume."""

    def __init__(self, n, shape, task, rank=0, world=1, seed=0):
        self.ids = list(shard_indices(n, rank, world))
        self.shape, self.task, self.seed = tuple(shape), task, seed

    def __len__(self):
        return len(self.ids)

    def __iter__(self):
        for i in self.ids:
            g = torch.Generator().manual_seed(self.seed + i)
            img = torch.rand((1, 1, *self.shape), generator=g)
            if self.task == "export_pseudo_labels":
                yield {"raw": {"image": img}, "name": [f"synthetic_{i:08d}"]}
            else:
                h = torch.eye(3).unsqueeze(0)
                h[0, 0, 2], h[0, 1, 2] = 4.0, -3.0
                yield {"image": img, "warped_image": torch.roll(img, shifts=(-3, 4), dims=(2, 3)), "homography": h,
                       "name": [f"synthetic_{i:08d}"]}


def load_pretrained(model, config, device):
    """engine.py:108-117: copy the keys present in both dicts, then load_state_dict."""
    state = model.state_dict()
    ckpt = torch.load(Path(settings.CKPT_PATH, config["pretrained"]), map_location=device)
    for k, v in ckpt["model_state_dict"].items():
        if k in state:
            state[k] = v
    model.load_state_dict(state)
    print("\033[92m✅ Loaded pretrained model \033[0m")


@tyro.conf.configure(tyro.conf.FlagConversionOff)
def main(config_path: str,
         task: Literal["export_pseudo_labels", "export_HPatches_Repeatability", "export_HPatches_Descriptors",
                       "train", "export_NeRF_labels"],
         training: options = options(),
         pseudo_labels: export_pseudo_labels_split = export_pseudo_labels_split(),
         synthetic: int = 0, random_init: bool = False) -> None:
    """Run one export task.

    Args:
        config_path: Path to configuration.
        task: The task to be performed.
        synthetic: feed this many synthetic images instead of the dataset loader.
        random_init: skip loading `pretrained` (benchmarking with random-init weights, torch.manual_seed(0) on every rank).
    """
    if task == "train":
        raise SystemExit(f"task {task!r} is outside the B200 hot path (SURVEY.md section 8); use the reference for it")
    if task == "export_NeRF_labels" and synthetic:
        raise SystemExit("--synthetic feeds single images; export_NeRF_labels needs posed views (data/PosedViews.py)")
    with open(config_path, "r") as f:
        config = yaml.safe_load(f)
    if not torch.cuda.is_available():
        raise SystemExit("CUDA is not available: this implementation has no CPU fallback")
    rank, world, device = init_distributed()
    if random_init:
        torch.manual_seed(0)      # every rank (and every run) gets the same random-init weights
    model = get_model(config["model"], device=device)
    if not random_init:
        assert config["pretrained"], "Use pretrained model to export."
        load_pretrained(model, config, device)
    if synthetic:
        loader = SyntheticLoader(synthetic, config["data"]["preprocessing"]["resize"], task, rank, world)
    else:
        from .utils.data_loaders import get_loader
        loader = get_loader(config, task, device=device, export_split=pseudo_labels.split, rank=rank, world=world)
    if task == "export_pseudo_labels":
        if world > 1:   # device-sampler key = global dataset index: rank-strided items, see ExportDetections
            config.setdefault("homography_adaptation", {}).update(index_stride=world, index_offset=rank)
        ExportDetections(config, model, loader, pseudo_labels.split, pseudo_labels.enable_Homography_Adaptation, device)
    elif task == "export_NeRF_labels":
        ExportNeRFDetections(config, model, loader, pseudo_labels.split, device)
    elif task == "export_HPatches_Repeatability":
        Export_Hpatches_Repeatability(config, model, loader, device)
    else:
        Export_Hpatches_Descriptors(config, model, loader, device)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    tyro.cli(main, use_underscores=True)
