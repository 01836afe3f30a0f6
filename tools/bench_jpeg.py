#!/usr/bin/env python
"""Host vs device JPEG decode for the export loader (``data.decode``).

Writes N seeded 640x480 q90 4:2:0 JPEGs (as tools/bench_loader.py does) and reports, with the GPU's name, power limit
and clocks read in the same run:
  * decode-only img/s: host (torchvision decode_image GRAY on a thread pool: all workers, and 2) and device
    (spn_jpeg_decode_gray, batch 64 and 256, file bytes already on the host: plan + upload + decode + status read-back);
  * ExportDetections img/s (f16, 100 homographies, 240x320) fed by each mode with --workers 15 and 2 (2 threads
    emulates 8 ranks sharing 16 cores);
  * the export step time alone and with a concurrent device decode batch on the loader's side stream.

    python tools/bench_jpeg.py [--n 1024] [--out profiles/r3_jpeg_bench.json]
"""
import argparse
import concurrent.futures as cf
import copy
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from superpoint_nerf_pytorch_b200 import _native as N, settings  # noqa: E402
from superpoint_nerf_pytorch_b200.data.preprocessing import _upload_stream  # noqa: E402
from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportDetections  # noqa: E402
from superpoint_nerf_pytorch_b200.utils.data_loaders import get_loader  # noqa: E402
from superpoint_nerf_pytorch_b200.utils.get_model import get_model  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def host_decode_rate(files, workers):
    import torchvision
    ts = [torch.frombuffer(bytearray(f), dtype=torch.uint8) for f in files]
    dec = lambda t: torchvision.io.decode_image(t, torchvision.io.ImageReadMode.GRAY)  # noqa: E731
    with cf.ThreadPoolExecutor(workers) as pool:
        list(pool.map(dec, ts[:64]))
        t0 = time.perf_counter()
        list(pool.map(dec, ts))
        return len(ts) / (time.perf_counter() - t0)


class DeviceDecoder:
    """Batch decode with the bytes already on the host: plan + upload + decode + status read-back, on `stream`."""

    def __init__(self, files, batch, stream):
        self.batches = []
        dev = torch.device("cuda", 0)
        for k in range(0, len(files), batch):
            fs = files[k:k + batch]
            offsets = np.zeros(len(fs) + 1, np.int64)
            np.cumsum([len(f) for f in fs], out=offsets[1:])
            host = torch.empty(int(offsets[-1]), dtype=torch.uint8, pin_memory=True)
            host.numpy()[:] = np.frombuffer(b"".join(fs), np.uint8)
            _, _, cb, ob = N.jpeg_plan(host.numpy(), offsets)
            self.batches.append((host, offsets, torch.empty(cb // 2, dtype=torch.int16, device=dev),
                                 torch.empty(ob, dtype=torch.uint8, device=dev), torch.empty(len(fs), dtype=torch.int32, device=dev),
                                 torch.empty(len(fs), dtype=torch.int32, pin_memory=True)))
        self.ctx, self.stream, self.dev = N.get_context(dev), stream, dev

    def run(self, which=None):
        bad = 0
        for host, offsets, coef, out, st, st_h in (self.batches if which is None else [self.batches[which]]):
            plan = N.jpeg_plan(host.numpy(), offsets)[0]
            with torch.cuda.stream(self.stream):
                d = host.to(self.dev, non_blocking=True)
                p = torch.from_numpy(plan).pin_memory().to(self.dev, non_blocking=True)
                self.ctx.jpeg_decode_gray(p, d, len(offsets) - 1, coef, out, st)
                st_h.copy_(st, non_blocking=True)
        self.stream.synchronize()
        for b in (self.batches if which is None else [self.batches[which]]):
            bad += int((b[5] != 0).sum())
        return bad


def device_decode_rate(files, batch):
    dd = DeviceDecoder(files, batch, torch.cuda.Stream(0))
    dd.run()
    t0 = time.perf_counter()
    bad = dd.run()
    dt = time.perf_counter() - t0
    assert bad == 0, f"{bad} images not decoded on the device"
    # kernel-only time of one batch (CUDA events around the two kernels)
    host, offsets, coef, out, st, _ = dd.batches[0]
    plan = torch.from_numpy(N.jpeg_plan(host.numpy(), offsets)[0]).to(dd.dev)
    d = host.to(dd.dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        dd.ctx.jpeg_decode_gray(plan, d, len(offsets) - 1, coef, out, st)
    b.record()
    torch.cuda.synchronize()
    return len(files) / dt, a.elapsed_time(b) / 5


def export_rate(cfg, model, workers):
    cfg = copy.deepcopy(cfg)
    cfg["data"]["loader_workers"] = workers
    loader = get_loader(cfg, "export_pseudo_labels", device="cuda", export_split="training")
    warm = copy.deepcopy(cfg)
    warm["data"]["experiment_name"] = "warm"
    ExportDetections(warm, model, [b for _, b in zip(range(128), loader)], "training", True, "cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ExportDetections(cfg, model, loader, "training", True, "cuda")
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    files = len(list(Path(settings.EXPER_PATH, "outputs", cfg["data"]["experiment_name"], "training").glob("*.npy")))
    return files / dt


def step_time(model, cfg, dd, with_decode, reps=6):
    """ms per HA export step (64 images x 100 homographies, device sampler), alone or while a decode batch runs."""
    from superpoint_nerf_pytorch_b200.engine_solvers.export import HomographyAdaptation
    eng = HomographyAdaptation(cfg, model, "cuda")
    img = torch.rand(64, 1, 240, 320, device="cuda")
    eng.heatmaps(img)
    torch.cuda.synchronize()
    ts = []
    for r in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        if with_decode:
            dd.run_async(r % len(dd.batches))
        eng.heatmaps(img)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    import cv2
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_jpeg.py measures the GPU decoder: no CUDA device")
    res = {"gpu": gpu_info(), "jpeg": "640x480 q90 4:2:0 (cv2), seeded", "n": args.n}
    tmp = Path(tempfile.mkdtemp(prefix="spn_jpeg_"))
    try:
        d = tmp / "data" / "COCO" / "images" / "training"
        d.mkdir(parents=True)
        rng = np.random.RandomState(0)
        base = cv2.GaussianBlur(rng.randint(0, 256, (480, 640, 3)).astype(np.uint8), (0, 0), 2.0)
        files = []
        for k in range(args.n):
            ok, buf = cv2.imencode(".jpg", np.roll(base, k * 7, axis=1), [cv2.IMWRITE_JPEG_QUALITY, 90])
            files.append(buf.tobytes())
            (d / f"im{k:06d}.jpg").write_bytes(files[-1])
        res["decode_only_img_per_s"] = {"host_15_threads": host_decode_rate(files, 15), "host_2_threads": host_decode_rate(files, 2)}
        for batch in (64, 256):
            rate, ms = device_decode_rate(files, batch)
            res["decode_only_img_per_s"][f"device_batch{batch}"] = rate
            res[f"device_kernels_ms_per_batch{batch}"] = ms
        settings.DATA_PATH, settings.EXPER_PATH = str(tmp / "data"), str(tmp / "exper")
        data = {"name": "COCO", "class_name": "COCO", "experiment_name": "jpeg_bench", "preprocessing": {"resize": [240, 320]},
                "has_labels": False, "warped_pair": False, "batch_size": 1, "truncate": False,
                "augmentation": {"photometric": {"enable": False}, "homographic": {"enable": False}}}
        mcfg = dict(copy.deepcopy(bench.MODEL_CFG), precision="f16")
        cfg = {"data": data, "model": mcfg,
               "homography_adaptation": dict(copy.deepcopy(bench.HA_CFG), sampler="device", seed=1, images_per_launch=64, max_forwards=400)}
        model = get_model(mcfg, "cuda").eval()
        model.load_state_dict(bench.random_init_state_dict())
        res["export_img_per_s"] = {}
        for rep in range(2):
            for mode in ("host", "device"):
                for w in (15, 2):
                    c = copy.deepcopy(cfg)
                    c["data"]["decode"] = mode
                    c["data"]["experiment_name"] = f"e_{mode}_{w}_{rep}"
                    res["export_img_per_s"].setdefault(f"{mode}_workers{w}", []).append(export_rate(c, model, w))
        dd = DeviceDecoder(files[:256], 256, _upload_stream(torch.device("cuda", 0)))

        def run_async(i):
            host, offsets, coef, out, st, _ = dd.batches[i]
            plan = N.jpeg_plan(host.numpy(), offsets)[0]
            with torch.cuda.stream(dd.stream):
                dd.ctx.jpeg_decode_gray(torch.from_numpy(plan).pin_memory().to(dd.dev, non_blocking=True),
                                        host.to(dd.dev, non_blocking=True), len(offsets) - 1, coef, out, st)
        dd.run_async = run_async
        res["export_step_ms"] = {"alone": step_time(model, cfg, dd, False), "with_decode_batch256": step_time(model, cfg, dd, True),
                                 "alone_again": step_time(model, cfg, dd, False)}
        res["gpu_after"] = gpu_info()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
