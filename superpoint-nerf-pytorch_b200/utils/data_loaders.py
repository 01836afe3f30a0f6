"""Loader factory with the reference's signature (utils/data_loaders.py:4-101), export tasks only.

``get_loader(config, task, device, export_split=...)`` imports ``data/<config.data.name>.py`` and instantiates
``config.data.class_name`` like the reference; instead of ``torch.utils.data.DataLoader(num_workers=0)`` (one image
decoded at a time on the loop's thread) it returns a ``PrefetchLoader``: the host part of ``__getitem__`` (file read +
JPEG/PPM decode, which release the GIL) runs on a thread pool a bounded number of items ahead, the device part (one
resize/crop/normalise kernel per image on the uint8 pixels) runs on the consumer's thread and stream.  It yields the
same collated batch dictionaries in the same order; rank sharding (``rank``/``world``) takes items with
index = rank (mod world) BEFORE anything is decoded.  ``export_NeRF_labels`` items are whole chunks of posed views
(data/PosedViews.py), loaded one per batch.  A dataset that has ``finish_batch`` (COCO with ``data.decode:
device``) gets up to ``device_batch`` ready items at a time, in order, for one batched device stage.  The stage is
launched when its items are ready and its results are taken one batch later, so the wait for one batch overlaps the
gathering and launch of the next.  Items before one that fails are yielded before the exception, as without the stage.
"""
import concurrent.futures as cf
import importlib
import itertools
import os

_DATA_PACKAGE = __name__.rsplit(".utils.", 1)[0] + ".data"


class PrefetchLoader:
    def __init__(self, dataset, batch_size=1, workers=None, depth=None, rank=0, world=1, device_batch=None):
        self.dataset = dataset
        self.device_batch = max(1, int(device_batch or 64))
        self.batch_size = max(1, int(batch_size))
        self.workers = workers or max(1, min(32, (os.cpu_count() or 2) - 1))
        self.depth = depth or 4 * self.workers
        if hasattr(dataset, "finish_batch"):
            self.depth = max(self.depth, 2 * self.device_batch)   # room for a full batch behind the one being decoded
        self.indices = list(range(rank, len(dataset), world))

    def __len__(self):
        return (len(self.indices) + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        ds = self.dataset
        split = hasattr(ds, "decode") and hasattr(ds, "finish")
        host_part = ds.decode if split else ds.__getitem__
        stage = getattr(ds, "finish_batch", None) if split else None
        with cf.ThreadPoolExecutor(max_workers=self.workers) as pool:
            pending, nxt, batch, inflight = [], 0, [], None
            while nxt < len(self.indices) or pending or inflight is not None:
                while nxt < len(self.indices) and len(pending) < self.depth:
                    pending.append(pool.submit(host_part, self.indices[nxt]))
                    nxt += 1
                items, failure, finished = [], None, []
                try:
                    if pending:
                        items.append(pending.pop(0).result())    # in order; re-raises a worker's exception here
                        while stage is not None and pending and len(items) < self.device_batch and pending[0].done():
                            items.append(pending.pop(0).result())
                except Exception as e:  # noqa: BLE001 - re-raised below, after the items before it
                    failure = e
                if stage is None:
                    finished = [ds.finish(it) if split else it for it in items]
                else:
                    launched = stage(items) if items else None
                    finished, inflight = (inflight or []), launched
                    if failure is not None and inflight is not None:
                        finished, inflight = itertools.chain(finished, inflight), None
                for it in finished:
                    batch.append(it)
                    if len(batch) == self.batch_size:
                        yield ds.batch_collator(batch)
                        batch = []
                if failure is not None:
                    raise failure
            if batch:
                yield ds.batch_collator(batch)


def get_loader(config, task, device="cuda", validate_training=False, export_split=None, nerf_train=False, rank=0, world=1):
    name, class_name = config["data"]["name"], config["data"]["class_name"]
    batch_size = config["data"]["batch_size"]
    cls = getattr(importlib.import_module(f"{_DATA_PACKAGE}.{name}"), class_name)
    if task in ("train", "test") or validate_training or nerf_train:
        raise NotImplementedError(f"task {task!r} is outside the B200 hot path (SURVEY.md section 8): use the reference's loader")
    if task == "export_NeRF_labels":              # one item = one chunk of posed views (data/PosedViews.py)
        dataset = cls(config["data"], task=export_split, device=device)
        return PrefetchLoader(dataset, 1, workers=config["data"].get("loader_workers"), rank=rank, world=world)
    if task == "export_pseudo_labels":
        dataset = cls(config["data"], task=export_split, device=device)
    elif task in ("export_HPatches_Repeatability", "export_HPatches_Descriptors"):
        dataset = cls(config["data"], device=device)
    else:
        raise ValueError(f"unknown task {task!r}")
    return PrefetchLoader(dataset, batch_size, workers=config["data"].get("loader_workers"), rank=rank, world=world,
                          device_batch=config["data"].get("decode_batch"))
