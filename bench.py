#!/usr/bin/env python
"""bench.py - pseudo-label images/s of the homography-adaptation export (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--precision fp32|f16|bf16]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload = BASELINE.json configs[1]: MagicPoint homography-adaptation export, 240x320 synthetic images, 100
homographies (1 identity + 99 warps), aggregation 'sum', valid_border_margin 3, nms 4, det_thresh 0.015, top_k 0,
random-init weights.  One "step" = one pass of the hot path over `--images-per-step` images per GPU
(warp -> encoder/head over all (image, homography) pairs -> aggregate -> NMS/threshold/compaction).

Prints ONE JSON line (rank 0).  `value` = images/s with the images already resident in HBM; `e2e` = the same through
the public API (HomographyAdaptation.__call__, i.e. what ExportDetections runs) from pinned HOST images to HOST
keypoint arrays, copies inside the timed region.  `roofline` = the dominant kernel (block_2 convolution) timed with
CUDA events inside the library during the timed region; `kernels` lists the same for the other kernels.
`cpu_baseline` (N=1, rank 0) = the oracle port of the reference timed on the host cores on a bounded sample (1 image x
25 of 100 homographies); `gpu_reference` = the same port with device="cuda" (stock cuDNN with torch's TF32 default,
torchvision's CUDA nms, 100 sequential batch-1 steps) - the honest GPU bar next to the CPU figure.

`--impl reference` times the reference's CPU path (oracle port, the reference is pure Python) on the host cores: exactly
--steps timed steps after --warmup untimed ones, each a bounded sample (1 image x h of the 100 homographies, h sized so
the run takes about --ref-budget-s seconds), same `config` object as the native arm.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

H, W, NUM_H = 240, 320, 100
WORKLOAD = "MagicPoint HA pseudo-label export, 240x320, 100 homographies (configs[1])"
MODEL_CFG = {"script": "SuperPoint", "class_name": "SuperPoint", "model_name": "magicpoint",
             "vgg_cn": [64, 64, 64, 64, 128, 128, 128, 128],
             "detector_head": {"detector_dim": [128, 256], "grid_size": 8, "nms": 4, "det_thresh": 0.015, "top_k": 0}}
HA_CFG = {"num": NUM_H, "aggregation": "sum", "filter_counts": 0, "valid_border_margin": 3,
          "params": {"translation": True, "rotation": True, "scaling": True, "perspective": True, "scaling_amplitude": 0.2,
                     "perspective_amplitude_x": 0.2, "perspective_amplitude_y": 0.2, "allow_artifacts": True,
                     "patch_ratio": 0.85, "max_angle": 1.57}}
# exact FLOPs (2*MACs) of one MagicPoint forward at 240x320, per layer (SURVEY.md section 8a)
# in the tensor-core modes block_1 is fused into block_2's kernel (front_tc.cu): its 0.088 GFLOP are then timed (and
# counted) under "backbone.block_2"
LAYER_FLOPS = {"backbone.block_1": 0.088e9, "backbone.block_2": 5.662e9, "backbone.block_3": 1.416e9,
               "backbone.block_4": 1.416e9, "backbone.block_5": 0.708e9, "backbone.block_6": 1.416e9,
               "backbone.block_7": 0.354e9, "backbone.block_8": 0.354e9, "detector_head.convPa": 0.708e9,
               "detector_head.convPb": 0.040e9}
FLOPS_PER_IMAGE = 1.2161e12
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def ncu_block2_traffic_per_forward(fused=True):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel's launch in the committed `ncu --set full`
    capture (latest profiles/r*_kernels_final.json, 100 forwards per launch) -> bytes per forward, or None."""
    for name in ("r2_kernels_final.json", "r1_kernels_final.json"):
        try:
            ks = json.loads((ROOT / "profiles" / name).read_text())
            pat = "front_tc_kernel" if fused else "conv_tc_kernel<9>"
            k = max((k for k in ks if pat in k["kernel"]), key=lambda k: k["time_us"])
            return (k["dram_read_MB"] + k["dram_write_MB"]) * 1e6 / float(k.get("forwards_per_launch", 100))
        except Exception:
            continue
    return None


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return json.loads(f.read_text()), "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_config(args, world):
    """`config` of BOTH arms' JSON lines - the reference arm runs on the native arm's config, so the two lines carry the
    identical object: the workload, how the native arm runs it, and (labelled) how the reference arm samples it."""
    ips = args.images_per_step
    return {"workload": WORKLOAD, "images_per_step_per_gpu": ips, "forwards_per_step_per_gpu": ips * NUM_H,
            "precision": args.precision, "weights": "random-init", "sampler": "device", "streams": args.streams,
            "parallelism": f"image-sharded x{world}",
            "kernel_timing": "per-kernel durations (roofline, kernels[]) come from a second pass over the same K steps "
                             "with a CUDA event pair around every launch; value/ms_per_step are the uninstrumented pass",
            "l2_policy": "no explicit flush: each step streams > 1 GB of fresh activations per GPU (>> 126 MB L2) "
                         "and uses images not seen before",
            "reference_arm": "bench.py --impl reference runs the same workload through the CPU oracle port of the reference "
                             "(torch-CPU fp32, all host threads, incl. the in-model NMS the reference pays for): every step is a "
                             "bounded sample, 1 image x h of the 100 homographies, extrapolated linearly; images_per_step / "
                             "precision / sampler / streams describe the native arm"}


def random_init_state_dict():
    """torch default init under torch.manual_seed(0) of the reference architecture (parameter holder only)."""
    import torch

    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    torch.manual_seed(0)
    return {k: v.detach().cpu() for k, v in get_model(copy.deepcopy(MODEL_CFG), "cpu").state_dict().items()}


def cpu_reference_sample(n_hom: int, threads: int | None = None, device: str | None = None):
    """Time the oracle port of ExportDetections (full forward incl. the in-model NMS the reference pays for and discards)
    on the host cores - or, with ``device="cuda"``, the same code on the GPU the way the reference would run there
    (cuDNN, TF32 default, torchvision CUDA nms): ONE 240x320 image with `n_hom` homographies; extrapolate linearly to 100."""
    import numpy as np
    import torch

    from oracle import spn_oracle as O

    if threads is None:
        # every host core this process may use (torchrun exports OMP_NUM_THREADS=1, which would make it a 1-thread run)
        try:
            threads = len(os.sched_getaffinity(0))
        except AttributeError:
            threads = os.cpu_count() or 1
    torch.set_num_threads(max(1, threads))
    cfg = {"homography_adaptation": dict(copy.deepcopy(HA_CFG), num=n_hom), "model": copy.deepcopy(MODEL_CFG)}
    sd = random_init_state_dict()  # the same random-init weights the native arm runs (flat ~1/65 heatmap)
    g = torch.Generator().manual_seed(0)
    img = torch.rand((1, 1, H, W), generator=g)
    np.random.seed(0)
    if device is not None:   # warm-up: cuDNN autotuning, torchvision op loading, allocator
        O.homography_adaptation(sd, img, {**cfg, "homography_adaptation": dict(cfg["homography_adaptation"], num=3)},
                                full_forward=True, device=device)
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    O.homography_adaptation(sd, img, cfg, full_forward=True, device=device)
    if device is not None:
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    per_forward = dt / n_hom
    where = "host cores" if device is None else f"{device} (cuDNN, allow_tf32={torch.backends.cudnn.allow_tf32}, torchvision CUDA nms)"
    return {"seconds": dt, "img_per_s": 1.0 / (per_forward * NUM_H), "cores": torch.get_num_threads(),
            "sample": f"1 image x {n_hom} of {NUM_H} homographies (240x320, full model forward incl. in-model NMS, "
                      f"kornia-shim warps) on {where}, linearly extrapolated to {NUM_H}"}


def run_reference(args):
    """The reference arm: exactly `--steps` timed steps after `--warmup` untimed ones, each step one bounded sample of
    the workload (1 image x h of the 100 homographies through the CPU oracle port, all host threads).  h is fixed for
    the run, chosen from a two-homography calibration so that warm-up + timed steps take about `--ref-budget-s` seconds
    (2 <= h <= --ref-homographies).  value = images' worth of work done in the timed steps / their wall time."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", 1))
    steps, warmup = args.steps, args.warmup
    calib = cpu_reference_sample(2)
    per_h = calib["seconds"] / 2
    h = int(min(max(2, args.ref_budget_s / ((steps + warmup) * per_h)), max(2, args.ref_homographies)))
    timed = []
    for i in range(warmup + steps):
        r = cpu_reference_sample(h)
        if i >= warmup:
            timed.append(r["seconds"])
    total = sum(timed)
    v = steps * (h / NUM_H) / total
    sample = (f"{steps} timed steps (+{warmup} warm-up), each 1 image x {h} of {NUM_H} homographies (240x320, full model forward "
              f"incl. in-model NMS, kornia-shim warps) on host cores, linearly extrapolated to {NUM_H}")
    line = {"impl": "reference", "metric": "pseudo-label img/s (240x320, 100 H)", "value": v, "unit": "img/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * total / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "cpu_baseline": {"value": v, "unit": "img/s", "cores": calib["cores"], "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


DUMP_MAX_IMAGES = 128   # 128 heatmaps (39 MB) + at most 128 x 16384 keypoints (17 MB) stay under 64 MB
DUMP_MAX_BYTES = 64 * 2**20


def dump_outputs(out_dir, step, max_kp):
    """Write what the timed path returned in its last step, as float32 DIR/<name>.npy:
    heatmap (n,H,W) aggregated heatmaps, homographies (n,NUM_H-1,3,3) the warps they aggregate, keypoints (N,2) the (row,
    col) box_nms kept, concatenated in image order, keypoint_counts (n,) keypoints per image.  A step of more than
    DUMP_MAX_IMAGES images is represented by a fixed seeded sample of DUMP_MAX_IMAGES of them, in image order."""
    import numpy as np

    n = step["heat"].shape[0]
    idx = np.arange(n) if n <= DUMP_MAX_IMAGES else np.sort(np.random.RandomState(0).choice(n, DUMP_MAX_IMAGES, replace=False))
    counts = step["kp_count"].cpu().numpy()[idx]
    kp = step["kp"].cpu().numpy()[idx]
    arrays = {"heatmap": step["heat"].cpu().numpy()[idx],
              "homographies": step["homographies"].cpu().numpy()[idx],
              "keypoints": np.concatenate([kp[j, :min(int(c), max_kp)] for j, c in enumerate(counts)]),
              "keypoint_counts": counts}
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    out_dir.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", a)


def run_native(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from superpoint_nerf_pytorch_b200.engine_solvers.export import HomographyAdaptation
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    from superpoint_nerf_pytorch_b200.utils.sharding import gather_export_counts, shard_indices

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    mcfg = dict(copy.deepcopy(MODEL_CFG), precision=args.precision)
    model = get_model(mcfg, dev).eval()
    model.load_state_dict(random_init_state_dict())  # random-init weights (no checkpoints ship with the reference)
    ha = dict(copy.deepcopy(HA_CFG), sampler="device", seed=1234, max_forwards=args.max_forwards, streams=args.streams)
    cfg = {"homography_adaptation": ha, "model": mcfg}
    eng = HomographyAdaptation(cfg, model, dev)
    ctx = model.native()

    ips = args.images_per_step
    n_steps = args.warmup + args.steps
    total_images = world * ips * n_steps
    my_ids = list(shard_indices(total_images, rank, world))   # image id = global id, rank r takes ids = r mod world
    g = torch.Generator().manual_seed(1000 + rank)
    host_pool = torch.rand((len(my_ids), 1, H, W), generator=g).pin_memory()      # synthetic COCO-shaped images in [0,1]
    dev_pool = host_pool.to(dev)
    max_kp = min(H * W, 16384)
    dh = mcfg["detector_head"]

    def device_step(i):
        imgs = dev_pool[i * ips:(i + 1) * ips]
        heat, hom = eng.heatmaps(imgs, first_index=my_ids[i * ips])
        r = ctx.box_nms(heat, float(dh["nms"]), 0.1, float(dh["det_thresh"]), int(dh["top_k"]),
                        det_thresh=float(dh["det_thresh"]), want_map=False, max_kp=max_kp)
        r.update(heat=heat, homographies=hom)
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput -----------------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for i in range(args.warmup):
        device_step(i)
    barrier()
    if sampler:
        sampler.rows.clear()   # keep only samples taken during the timed region
    ctxs = list(model._ctxs.values())     # one context per concurrent stream

    def prof_read_all():
        tot = {}
        for c in ctxs:
            for k, (t, n) in c.profile_read().items():
                a = tot.get(k, (0.0, 0))
                tot[k] = (a[0] + t, a[1] + n)
        return tot

    # Pass 1 (the reported value): K steps, nothing but the path's own launches on the stream.
    l0 = sum(c.launches for c in ctxs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.warmup, n_steps):
        last = device_step(i)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = sum(c.launches for c in ctxs) - l0
    clocks = sampler.stop() if sampler else None
    # Pass 2 (per-kernel durations for the roofline): the same K steps again with a CUDA event pair around every
    # launch (spn_profile_enable); kept out of pass 1 because the event records sit between the kernels.
    for c in ctxs:
        c.profile_enable(True)
    prof_read_all()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for i in range(args.warmup, n_steps):
        r = device_step(i)
    i1.record()
    barrier()
    ms_instr = max_over_ranks(i0.elapsed_time(i1))
    prof = prof_read_all()
    for c in ctxs:
        c.profile_enable(False)
    kept = int(r["kp_count"].sum().item())
    value = world * ips * args.steps / (ms / 1e3)

    # ---- end to end through the public API: pinned host images -> host keypoint arrays ----------------------------
    # The public calls ExportDetections makes, software-pipelined the way its loop is: step i+1 is enqueued (pinned host
    # images -> device, whole GPU pass, keypoints -> pinned host) before the host collects step i's keypoint arrays.
    def e2e_launch(i):
        imgs = host_pool[i * ips:(i + 1) * ips].to(dev, non_blocking=True)
        heat, _ = eng.heatmaps(imgs, first_index=my_ids[i * ips])
        return eng.keypoints_async(heat)                    # handle; keypoints_wait -> list of (N,2) int64 numpy arrays

    eng.keypoints_wait(e2e_launch(0))
    barrier()
    t0 = time.perf_counter()
    e0.record()
    nk = 0
    pending = None
    for i in range(args.warmup, n_steps):
        cur = e2e_launch(i)
        if pending is not None:
            nk += sum(len(k) for k in eng.keypoints_wait(pending))
        pending = cur
    nk += sum(len(k) for k in eng.keypoints_wait(pending))
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
    e2e_value = world * ips * args.steps / (ms_e2e / 1e3)
    allc, _ = gather_export_counts(ips * args.steps, nk, device=dev)   # the one collective of the path (16 B / rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    forwards = ips * NUM_H * args.steps   # forwards per rank in the timed region

    def tensor_entry(name):
        t, n = prof.get(name, (0.0, 0))
        if not n:
            return None
        fl = LAYER_FLOPS[name] * forwards
        if name == "backbone.block_2" and "backbone.block_1" not in prof:
            fl += LAYER_FLOPS["backbone.block_1"] * forwards   # fused front end
        ach = fl / (t / 1e3) / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["bf16_tflops_sustained"], "ms_per_launch": t / n, "launches": n}

    def hbm_entry(name, bytes_per_rank):
        t, n = prof.get(name, (0.0, 0))
        if not n:
            return None
        ach = bytes_per_rank / (t / 1e3) / 1e9
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                "ms_per_launch": t / n, "launches": n}

    imgs_rank = ips * args.steps
    kernels = [tensor_entry(n) for n in LAYER_FLOPS]
    # fast modes: the image warp is fused into front_tc_kernel, warp_batch only writes the 1-byte validity masks;
    # strict fp32 mode: it also reads the image and writes the warped copy (614.4 KB / homography)
    fused_warp = args.precision in ("f16", "bf16")
    warp_bytes = NUM_H * H * W if fused_warp else (NUM_H - 1) * 4 * H * W * 2 + NUM_H * H * W
    kernels += [hbm_entry("warp_batch", imgs_rank * warp_bytes),
                hbm_entry("ha_aggregate", imgs_rank * (NUM_H * 4 * H * W + 4 * H * W)),              # 30.7 MB read + 307 KB written / image
                hbm_entry("softmax_d2s", imgs_rank * NUM_H * (65 * (H // 8) * (W // 8) * 4 + 4 * H * W)),
                hbm_entry("box_nms", imgs_rank * 4 * H * W * 2)]
    kernels = [k for k in kernels if k]
    dom = next((k for k in kernels if k["kernel"] == "backbone.block_2"), None)
    total_kernel_ms = sum(t for t, _ in prof.values())
    roof = None
    if dom:
        tpf = ncu_block2_traffic_per_forward() if fused_warp else None
        fwd_per_launch = forwards / max(dom["launches"], 1)
        roof = {"bound": "tensor", "achieved": dom["achieved"], "peak": dom["peak"], "unit": "TFLOP/s", "frac": dom["frac"],
                "traffic": (tpf * fwd_per_launch) if tpf else None, "traffic_unit": "bytes per launch (ncu dram read+write)",
                "algorithmic_flops_per_launch": (LAYER_FLOPS["backbone.block_2"] + (LAYER_FLOPS["backbone.block_1"]
                                                 if "backbone.block_1" not in prof else 0.0)) * fwd_per_launch,
                "ms_per_launch": dom["ms_per_launch"], "kernel": ("front_tc_kernel = homography warp + block_1 (1->64) + block_2 (64->64, ReLU, 2x2 pool) fused; implicit GEMM "
                           "M=pixels N=64 K=576 (+K=16 for block_1) @240x320") if fused_warp else
                          ("conv_split_fold_kernel<64> block_2 (fp16 hi/lo split: 3 MMAs per product, so the useful-FLOP rate tops out at a third of the tensor peak)"
                           if args.precision == "f16x3" else "conv_fp32_kernel block_2 (strict FFMA path; tensor peak shown for scale only)"),
                "peak_source": f"{pk_kind} bf16_tflops_sustained", "share_of_step": (prof["backbone.block_2"][0] / total_kernel_ms)
                if total_kernel_ms else None}
    line = {"metric": "pseudo-label img/s (240x320, 100 H)", "value": value, "unit": "img/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "ms_per_step_instrumented": ms_instr / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "f16": "f16", "bf16": "bf16", "f16x3": "f16x3 (fp16 hi/lo split, fp32-grade)"}[args.precision], "data": "synthetic",
            "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": ips * H * W * 4,
                    "d2h_bytes_per_step": ips * (max_kp * 2 * 4 + 4), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "roofline": roof, "kernels": kernels,
            "tensor_frac_whole_step": (value / world * FLOPS_PER_IMAGE / 1e12) / pk["bf16_tflops_sustained"],
            "clocks": clocks, "keypoints_last_step": kept, "export_counts": allc.tolist()}
    if world == 1 and not args.no_cpu_baseline:
        c = cpu_reference_sample(args.ref_homographies)
        line["cpu_baseline"] = {"value": c["img_per_s"], "unit": "img/s", "cores": c["cores"], "kind": "port", "sample": c["sample"]}
        try:    # the reference's own code path with device="cuda": the honest GPU bar (SURVEY.md section 8d, BASELINE.md section 4)
            gr = cpu_reference_sample(args.ref_homographies, device=str(dev))
            line["gpu_reference"] = {"value": gr["img_per_s"], "unit": "img/s", "kind": "port", "device": "B200", "sample": gr["sample"],
                                     "note": "not comparable bit for bit: TF32 cuDNN convolutions; 100 sequential batch-1 "
                                             "steps, each with the in-model NMS that export.py:69 discards"}
        except Exception as e:   # e.g. torchvision built without CUDA ops
            line["gpu_reference"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), last, max_kp)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default=os.environ.get("SPN_B200_PRECISION", "f16"), choices=["fp32", "f16", "bf16", "f16x3"],
                    help="f16 (default): tcgen05 convolutions, fp16 operands / fp32 accumulate, 5e-3 parity gate; "
                         "fp32: strict FFMA convolutions, 1e-4 parity gate")
    ap.add_argument("--images-per-step", type=int, default=128,
                    help="images per GPU per step; 128 makes a step ~170 ms so the timed region of the default run is > 3 s "
                         "(the sustained, power-capped regime rather than a burst)")
    ap.add_argument("--max-forwards", type=int, default=400)
    ap.add_argument("--streams", type=int, default=1)
    ap.add_argument("--ref-homographies", type=int, default=25, help="homographies in the bounded CPU sample (of 100)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="--impl reference: target wall time of warm-up + timed steps; sets the homographies per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's heatmaps, homographies and keypoints as float32 "
                         "DIR/<name>.npy (rank 0's images; inputs are seeded, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
