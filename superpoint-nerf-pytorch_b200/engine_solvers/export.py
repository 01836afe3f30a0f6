"""Export tasks with the reference's class API (engine_solvers/export.py:17-222): the constructor runs the task.

ExportDetections              homography-adaptation pseudo-labels -> <EXPER_PATH>/outputs/<experiment>/<split>/<name>.npy
Export_Hpatches_Repeatability two forwards per pair               -> <EXPER_PATH>/repeatability/<experiment>/<name>.npz
Export_Hpatches_Descriptors   + dense descriptors (H,W,256)       -> <EXPER_PATH>/descriptors/<experiment>/<name>.npz

Optional on-disk formats (extension keys under ``data``; the defaults are the reference's layouts):
  ``packed: true``   ExportDetections additionally writes ONE file per rank, ``<split>/packed_rank<r>.npz`` with
                     ``names`` (n,), ``keypoints`` (N,2) int32 (row, col), ``offsets`` (n+1,) into ``keypoints`` and
                     ``global_offset`` = this rank's base in the concatenation over ranks (the all_gather of per-rank
                     counts, utils/sharding.gather_export_counts); ``per_image_files: false`` then skips the .npy files.
                     ``load_packed_labels`` reads the shards back as {name: (N,2) int64}.
  ``sparse: true``   Export_Hpatches_Descriptors stores ``keypoints`` (k,2) int32 / ``desc_sparse`` (k,256) (and the
                     ``warped_`` twins) - the descriptors AT the post-NMS keypoints, which is all that
                     descriptor_evaluation.compute_homography reads - instead of two dense (H,W,256) maps
                     (2 x 315 MB per 480x640 pair -> ~2 MB).  evaluations/descriptor_evaluation.py consumes both layouts.

What changes underneath: the 99 sequential batch-1 steps of the reference (export.py:103-104) become ONE batched
pass per group of images - warp_batch -> encoder/head over all (image, homography) pairs -> fused inverse-warp
aggregation -> NMS/threshold/compaction - every stage a kernel behind include/spn_b200.h.  The in-model box_nms
whose result export.py:69 discards is not computed.

Extension keys under ``homography_adaptation`` (optional): ``sampler`` 'device' (default, spn_sample_homographies)
or 'numpy' (the reference's host sampler and RNG order), ``seed``, ``images_per_launch`` (default 1),
``max_forwards`` (forwards per encoder launch, default 400), ``streams`` (concurrent CUDA streams, default 1).

Geometry: homographies that come from the host (the numpy sampler, or matrices passed in) go through
``utils.kornia_geometry.sampling_matrices`` - the reference's own torch calls - and the kernels then follow kornia's
fp32 coordinate chain operation for operation, so validity masks, counts and warped samples are bit-identical to the
reference's CPU run.  Device-sampled homographies use ``spn_kornia_matrices`` (same algebra, device arithmetic).
The device sampler is keyed by (seed, global image index * (num-1) + j): the homographies of an image depend only on
its index in the dataset order (``first_index``), not on batching, resume state or rank.
"""
import os
from pathlib import Path

import numpy as np
import torch

from .. import settings
from ..data.data_utils.homographic_augmentation import Homographic_aug
from ..utils.kornia_geometry import sampling_matrices
from ..utils.train_utils import move_to_device

try:
    from tqdm import tqdm
except ImportError:  # pragma: no cover
    def tqdm(it, **kw):
        return it


class HomographyAdaptation:
    """Batched ExportDetections.step/homography_adaptation (export.py:42-125) for a group of images."""

    def __init__(self, config, model, device="cuda"):
        self.config = config
        self.ha = config["homography_adaptation"]
        self.dh = config["model"]["detector_head"]
        self.model = model.eval()
        self.device = device
        self.sampler = Homographic_aug(self.ha, device)
        self.max_forwards = int(self.ha.get("max_forwards", 400))
        self.seed = int(self.ha.get("seed", 0))
        self.n_streams = max(1, int(self.ha.get("streams", 1)))
        self.index_stride = max(1, int(self.ha.get("index_stride", 1)))   # rank sharding: image k of a group has index first + k*stride
        self._streams = None
        if not self.ha["valid_border_margin"]:
            # the reference's margin-0 path is shape-broken (mask stays 4-D, SURVEY.md section 8 a2)
            raise ValueError("homography_adaptation.valid_border_margin must be >= 1")

    def _homographies(self, NI, n_h, H, W, first_index):
        """-> (NI,n_h,3,3) homographies: HOST tensors from the numpy sampler (the reference's RNG order, export.py:47),
        DEVICE tensors from the device sampler."""
        if self.ha.get("sampler", "device") == "numpy":
            hs = [self.sampler.sample_homography_host((H, W), **self.ha["params"]) for _ in range(NI * n_h)]
            return torch.cat(hs).view(NI, n_h, 3, 3).contiguous()
        if self.index_stride == 1 or NI == 1:
            h, _ = self.sampler.sample_homographies_device((H, W), NI * n_h, seed=self.seed, first_index=first_index * n_h)
        else:
            h = torch.cat([self.sampler.sample_homographies_device((H, W), n_h, seed=self.seed,
                                                                   first_index=(first_index + k * self.index_stride) * n_h)[0]
                           for k in range(NI)])
        return h.view(NI, n_h, 3, 3)

    def _sampling_matrices(self, ctx, homographies, NI, n_h, H, W, dev):
        """-> (h, h_inv, fwd, bwd) on the device: H, its pixel-space inverse (export.py:49) and kornia's normalised
        sampling matrices for H and H^-1 (the grids of the warps at export.py:51-55,72)."""
        if homographies.is_cuda and self.ha.get("geometry", "auto") != "host":
            h = homographies.to(dev, torch.float32).contiguous().view(NI, n_h, 3, 3)
            fwd, bwd = ctx.kornia_matrices(h, H, W)
            return h, ctx.invert3x3(h), fwd, bwd
        hc = homographies.detach().to("cpu", torch.float32).reshape(-1, 3, 3)
        fwd, bwd = sampling_matrices(hc, (H, W))                      # the reference's torch calls on the host
        pack = torch.stack([hc, torch.inverse(hc), fwd, bwd]).to(dev)
        return tuple(t.view(NI, n_h, 3, 3) for t in pack)

    @torch.no_grad()
    def heatmaps(self, images, homographies=None, enable_HA=True, first_index=0):
        """images (NI,1,H,W) CUDA fp32 -> (aggregated heatmap (NI,H,W), homographies used (NI,n_h,3,3) or None).
        With ``streams`` > 1 the images are split into groups that run on separate CUDA streams (each with its own
        context/workspace) so the bandwidth-bound kernels of one group overlap the tensor-core kernels of another."""
        NI = images.shape[0]
        n_h = int(self.ha["num"]) - 1
        if self.n_streams == 1 or NI < 2 or not enable_HA or n_h == 0:
            return self._heatmaps_group(images, homographies, enable_HA, first_index, 0)
        if self._streams is None:
            self._streams = [torch.cuda.Stream(device=images.device) for _ in range(self.n_streams)]
        cur = torch.cuda.current_stream(images.device)
        groups = [g for g in torch.chunk(torch.arange(NI), self.n_streams) if len(g)]
        heats, hs = [], []
        for k, idx in enumerate(groups):
            st = self._streams[k]
            st.wait_stream(cur)
            lo, hi = int(idx[0]), int(idx[-1]) + 1
            with torch.cuda.stream(st):
                hg = None if homographies is None else homographies[lo:hi]
                heat, h = self._heatmaps_group(images[lo:hi], hg, enable_HA, first_index + lo * self.index_stride, k)
            heat.record_stream(cur)
            h.record_stream(cur)
            heats.append(heat)
            hs.append(h)
        for k in range(len(groups)):
            cur.wait_stream(self._streams[k])
        return torch.cat(heats), torch.cat(hs)

    def _heatmaps_group(self, images, homographies, enable_HA, first_index, slot):
        NI, _, H, W = images.shape
        ctx = self.model.native(slot)
        imgs = images.detach().to(torch.float32).contiguous().view(NI, H, W)
        if not enable_HA:
            return self.model.prob_heatmap(imgs, slot=slot), None
        n_h = int(self.ha["num"]) - 1
        if n_h == 0:
            return self.model.prob_heatmap(imgs, slot=slot), None
        if homographies is None:
            homographies = self._homographies(NI, n_h, H, W, first_index)
        h, hinv, fwd, hback = self._sampling_matrices(ctx, homographies, NI, n_h, H, W, imgs.device)   # export.py:49 + kornia
        fused = self.model.mode in (1, 2) and self.ha.get("fused_warp", True)    # 16-bit modes: warp inside the first conv kernel
        warped, mask = ctx.warp_batch(imgs, fwd, self.ha["valid_border_margin"], want_warped=not fused)  # export.py:51-66
        B = NI * (n_h + 1)
        probs = torch.empty((B, H, W), dtype=torch.float32, device=imgs.device)
        for s in range(0, B, self.max_forwards):                                 # export.py:69-70
            e = min(B, s + self.max_forwards)
            if fused:
                self.model.prob_heatmap_ha(imgs, hinv, s, e - s, mask=mask[s:e], out=probs[s:e], slot=slot)
            else:
                self.model.prob_heatmap(warped[s:e], mask=mask[s:e], out=probs[s:e], slot=slot)
        agg = ctx.ha_aggregate(probs.view(NI, n_h + 1, H, W), hback, self.ha["valid_border_margin"],
                               self.ha["aggregation"])                           # export.py:72-77,106-114
        return agg, h

    @torch.no_grad()
    def keypoints_async(self, heat):
        """box_nms + threshold + nonzero (export.py:116-125) enqueued on the current stream; the keypoint lists are
        copied to pinned host memory asynchronously.  Returns a handle for ``keypoints_wait``."""
        ctx = self.model.native()
        NI, H, W = heat.shape
        max_kp = min(H * W, 16384)
        with torch.cuda.device(heat.device):      # copies and the completion event go on the heatmap's device
            r = ctx.box_nms(heat, float(self.dh["nms"]), 0.1, float(self.dh["det_thresh"]), int(self.dh["top_k"]),
                            det_thresh=float(self.dh["det_thresh"]), want_map=False, max_kp=max_kp)
            kp_h = torch.empty(r["kp"].shape, dtype=torch.int32, pin_memory=True)
            cnt_h = torch.empty(r["kp_count"].shape, dtype=torch.int32, pin_memory=True)
            kp_h.copy_(r["kp"], non_blocking=True)
            cnt_h.copy_(r["kp_count"], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(heat.device))
        return {"heat": heat, "kp": kp_h, "count": cnt_h, "event": ev, "max_kp": max_kp, "dev": r}

    def keypoints_wait(self, handle):
        """-> list of (N,2) int64 numpy arrays (row, col), row-major order like torch.nonzero."""
        handle["event"].synchronize()
        counts = handle["count"].numpy()
        if counts.max(initial=0) > handle["max_kp"]:      # rare: more keypoints than the buffer, redo with the true size
            ctx = self.model.native()
            r = ctx.box_nms(handle["heat"], float(self.dh["nms"]), 0.1, float(self.dh["det_thresh"]), int(self.dh["top_k"]),
                            det_thresh=float(self.dh["det_thresh"]), want_map=False, max_kp=int(counts.max()))
            kp = r["kp"].cpu().numpy()
        else:
            kp = handle["kp"].numpy()
        return [kp[i, :counts[i]].astype(np.int64) for i in range(len(counts))]

    @torch.no_grad()
    def keypoints(self, heat):
        return self.keypoints_wait(self.keypoints_async(heat))

    def __call__(self, images, homographies=None, enable_HA=True, first_index=0):
        heat, _ = self.heatmaps(images, homographies, enable_HA, first_index)
        return self.keypoints(heat)


class ExportDetections:
    def __init__(self, config, model, dataloader, split, enable_HA, device):
        self.config = config
        self.model = model.eval()
        self.dataloader = dataloader
        self.split = split
        self.enable_HA = enable_HA
        if self.enable_HA:
            print("\033[92m✅ Homography Adaptation enabled \033[0m")
        self.device = device
        self.output_dir = self._init_output_dir()
        self.engine = HomographyAdaptation(config, model, device)
        self.one_homography = self.engine.sampler
        self._stage_slots, self._stage_next = [{}, {}, {}], 0
        self.packed = bool(config["data"].get("packed", False))
        self.per_image_files = bool(config["data"].get("per_image_files", True)) or not self.packed
        self._packed_names, self._packed_kp = [], []
        self.homography_adaptation()
        if self.packed:
            self._write_packed()

    def _init_output_dir(self):
        out = Path(settings.EXPER_PATH, "outputs", self.config["data"]["experiment_name"], self.split)
        os.makedirs(out, exist_ok=True)
        return out

    def _stage(self, group):
        """Images of a group -> one device tensor.  Host images go through a rotating pinned staging buffer and one
        non-blocking copy, so the host never waits for the GPU here (a plain ``.to(device)`` of pageable memory is
        stream-ordered behind the previous group's kernels and blocks the loop until they finish)."""
        imgs = [g[1] for g in group]
        if all(i.is_cuda for i in imgs):
            return torch.cat(imgs, dim=0)
        shape = (len(imgs),) + tuple(imgs[0].shape[1:])
        slot = self._stage_slots[self._stage_next % len(self._stage_slots)]
        self._stage_next += 1
        if slot.get("buf") is None or tuple(slot["buf"].shape[1:]) != shape[1:] or slot["buf"].shape[0] < shape[0]:
            slot["buf"] = torch.empty(shape, dtype=torch.float32).pin_memory()
            slot["ev"] = None
        if slot["ev"] is not None:
            slot["ev"].synchronize()               # the copy that last read this buffer (two groups ago) is done
        buf = slot["buf"][:shape[0]]
        for k, im in enumerate(imgs):
            buf[k].copy_(im[0])
        dev = buf.to(self.device, non_blocking=True)
        with torch.cuda.device(dev.device):            # the event goes on the stream that carries the copy
            slot["ev"] = torch.cuda.Event()
            slot["ev"].record(torch.cuda.current_stream(dev.device))
        return dev

    def _launch(self, group, index):
        """Enqueue the whole GPU pass for a group of images; returns a handle (nothing is synchronised)."""
        images = self._stage(group)
        heat, _ = self.engine.heatmaps(images, enable_HA=self.enable_HA, first_index=index)
        return [g[0] for g in group], self.engine.keypoints_async(heat)

    def _finish(self, pending):
        paths, handle = pending
        for path, kp in zip(paths, self.engine.keypoints_wait(handle)):
            if self.per_image_files:
                np.save(path, kp)
            if self.packed:
                self._packed_names.append(Path(path).stem)
                self._packed_kp.append(kp.astype(np.int32))

    def _write_packed(self):
        """One packed shard per rank; global offsets from the all_gather of per-rank (images, keypoints) counts."""
        from ..utils.sharding import gather_export_counts
        import torch.distributed as dist
        counts = np.array([len(k) for k in self._packed_kp], np.int64)
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        dev = self.device if rank or (dist.is_available() and dist.is_initialized()) else "cpu"
        allc, offs = gather_export_counts(len(counts), int(counts.sum()), device=dev)
        kp = np.concatenate(self._packed_kp) if self._packed_kp else np.zeros((0, 2), np.int32)
        np.savez(Path(self.output_dir, f"packed_rank{rank:03d}.npz"), names=np.array(self._packed_names), keypoints=kp,
                 offsets=np.concatenate([[0], np.cumsum(counts)]), global_offset=np.array(int(offs[rank])),
                 counts_all_ranks=allc.cpu().numpy())

    @torch.no_grad()
    def homography_adaptation(self):
        """Same loop as export.py:82-129, software-pipelined: while the GPU works on group k the host saves group k-1."""
        ha = self.config["homography_adaptation"]
        per_launch = int(ha.get("images_per_launch", 1))
        # device-sampler key of an image = its index in the dataset order (x stride + offset under rank sharding), so
        # the homographies of an image do not depend on which files already existed, on batching or on the rank
        stride, offset = int(ha.get("index_stride", 1)), int(ha.get("index_offset", 0))
        group, pending = [], None

        def flush():
            nonlocal group, pending
            if not group:
                return
            cur = self._launch(group, group[0][2])
            if pending is not None:
                self._finish(pending)
            pending = cur
            group = []

        for seen, data in enumerate(tqdm(self.dataloader, desc="Exporting detections", colour="green")):
            name = data["name"][0]
            save_path = Path(self.output_dir, f"{name}.npy")
            if self.per_image_files and save_path.exists():   # resume by file existence (export.py:89-91)
                flush()                                # keeps the indices of a group consecutive
                continue
            image = data["raw"]["image"]              # moved to the device per group (see _stage), not per image
            if not torch.is_tensor(image) or image.dim() != 4 or image.shape[0] != 1:
                raise ValueError(f"expected one (1,1,H,W) image per batch, got {tuple(getattr(image, 'shape', ()))}")
            if image.dtype != torch.float32:
                image = image.float()
            if group and group[0][1].shape != image.shape:
                flush()
            group.append((save_path, image, seen * stride + offset))
            if len(group) >= per_launch:
                flush()
        flush()
        if pending is not None:
            self._finish(pending)


def _np(t):
    return t.squeeze().cpu().numpy()


class _NpzWriter:
    """np.savez_compressed on a small thread pool (zlib releases the GIL): the HPatches exports are bound by the
    host-side compression of ~5 MB (repeatability) to ~630 MB (dense descriptors) per pair, not by the GPU.  At most
    ``depth`` files are in flight, so host memory stays bounded; files are byte-identical to a synchronous save."""

    def __init__(self, workers=None, depth=None):
        import concurrent.futures as cf
        workers = workers or max(1, min(8, (os.cpu_count() or 2) - 1))
        self.pool = cf.ThreadPoolExecutor(max_workers=workers)
        self.depth = depth or 2 * workers
        self.pending = []

    def save(self, path, arrays):
        while len(self.pending) >= self.depth:
            self.pending.pop(0).result()           # re-raises a writer's exception here
        self.pending.append(self.pool.submit(np.savez_compressed, path, **arrays))

    def close(self):
        try:
            for f in self.pending:
                f.result()
        finally:
            self.pending = []
            self.pool.shutdown(wait=True)


class Export_Hpatches_Repeatability:
    def __init__(self, config, model, dataloader, device):
        self.config = config
        self.model = model.eval()
        self.dataloader = dataloader
        self.device = device
        self.output_dir = Path(settings.EXPER_PATH, "repeatability", config["data"]["experiment_name"])
        os.makedirs(self.output_dir, exist_ok=True)
        self.export_repeatability()

    @torch.no_grad()
    def export_repeatability(self):
        writer = _NpzWriter()
        try:
            for i, data in enumerate(tqdm(self.dataloader, desc="Exporting repeatability detections", colour="green")):
                data = move_to_device(data, self.device)
                both = torch.cat([data["image"], data["warped_image"]], dim=0)  # one batched forward for the pair
                probs = self.model(both)["detector_output"]["prob_heatmap_nms"]
                output = {"image": _np(data["image"]), "warped_image": _np(data["warped_image"]),
                          "prob": _np(probs[0]), "warped_prob": _np(probs[1]), "homography": _np(data["homography"])}
                filename = data["name"][0] if "name" in data else str(i)
                writer.save(Path(self.output_dir, f"{filename}.npz"), output)
        finally:
            writer.close()


class Export_Hpatches_Descriptors:
    def __init__(self, config, model, dataloader, device):
        self.config = config
        self.model = model.eval()
        self.dataloader = dataloader
        self.device = device
        self.output_dir = Path(settings.EXPER_PATH, "descriptors", config["data"]["experiment_name"])
        os.makedirs(self.output_dir, exist_ok=True)
        self.export_descriptors()

    @torch.no_grad()
    def export_descriptors(self):
        sparse = bool(self.config["data"].get("sparse", False))
        writer = _NpzWriter(workers=max(1, min(4, (os.cpu_count() or 2) - 1)), depth=4)   # ~630 MB per pair in flight
        try:
            for i, data in enumerate(tqdm(self.dataloader, desc="Exporting HPatches descriptors", colour="green")):
                data = move_to_device(data, self.device)
                both = torch.cat([data["image"], data["warped_image"]], dim=0)
                if sparse:                            # one C-ABI call: forward + NMS/top-k once + descriptors at keypoints
                    out = self.model(both, keypoints=True)
                    det, des = out["detector_output"], out["descriptor_output"]
                    n = det["keypoint_count"].cpu().numpy()
                    cap = det["keypoints"].shape[1]
                    if n.max() > cap:
                        raise RuntimeError(f"{int(n.max())} keypoints exceed the list capacity {cap}: set detector_head.top_k")
                    kp, ds = det["keypoints"].cpu().numpy(), des["desc_sparse"].cpu().numpy()
                    output = {"image": _np(data["image"]), "warped_image": _np(data["warped_image"]),
                              "prob": _np(det["prob_heatmap_nms"][0]), "warped_prob": _np(det["prob_heatmap_nms"][1]),
                              "keypoints": kp[0, :n[0]], "desc_sparse": ds[0, :n[0]],
                              "warped_keypoints": kp[1, :n[1]], "warped_desc_sparse": ds[1, :n[1]],
                              "homography": _np(data["homography"])}
                    filename = data["name"][0] if "name" in data else str(i)
                    writer.save(Path(self.output_dir, f"{filename}.npz"), output)
                    continue
                out = self.model(both)
                probs = out["detector_output"]["prob_heatmap_nms"]
                desc = out["descriptor_output"]["desc"]
                output = {"image": _np(data["image"]), "warped_image": _np(data["warped_image"]),
                          "prob": _np(probs[0]), "warped_prob": _np(probs[1]),
                          "desc": desc[0].cpu().numpy().transpose(1, 2, 0), "warped_desc": desc[1].cpu().numpy().transpose(1, 2, 0),
                          "homography": _np(data["homography"])}
                filename = data["name"][0] if "name" in data else str(i)
                writer.save(Path(self.output_dir, f"{filename}.npz"), output)
        finally:
            writer.close()


class ExportNeRFDetections:
    """NeRF multi-view pseudo-labels with the reference's class interface (engine_solvers/export.py:225-366): for every
    view j of a batch, the heatmap of j is averaged with the heatmaps of ~75 % of the other views k, re-projected into j
    through the depth maps and camera poses (3x3 patches around k's detections), then box_nms + threshold + nonzero ->
    ``<EXPER_PATH>/outputs/<experiment>/<split>/<name>.npy``.

    What changes underneath: the reference runs the model once per (j, k) pair; here every view is forwarded ONCE through
    the one-call path (heatmap + NMS + keypoint list, spn_detect_describe), the source views are drawn with python's
    ``random.choices`` exactly as in export.py:320-321, and then ONE spn_nerf_fuse call builds the averaged heatmaps of
    every target view of the batch (re-projection, border filter, ordered 3x3 patch copies and the running sum in two
    kernels), followed by one batched bit-exact box_nms and one copy to the host.  The pairing quirk of export.py:269-271
    (the border filter shortens ``unwarped_pts`` but the loop zips it with the unfiltered ``warped_pts``) is reproduced
    as is.  ``reproject`` is the per-pair composition (warp_points_NeRF -> filter_points -> spn_nerf_splat) that the
    fused kernel is tested against."""

    def __init__(self, config, model, dataloader, split, device):
        self.config = config
        self.model = model.eval()
        self.dataloader = dataloader
        self.split = split
        self.device = device
        self.output_dir = Path(settings.EXPER_PATH, "outputs", self.config["data"]["experiment_name"], self.split)
        os.makedirs(self.output_dir, exist_ok=True)
        self.export_NeRF()

    @torch.no_grad()
    def reproject(self, prob_k, pts_k, depth_k, intrinsics, rot_k, trans_k, rot_j, trans_j):
        """One ExportNeRFDetections.step without the model call: view k's detections splatted into view j's frame."""
        from ..data.data_utils.kp_utils import filter_points, warp_points_NeRF
        ctx = self.model.native()
        H, W = prob_k.shape
        if len(pts_k) == 0:
            return torch.zeros_like(prob_k)
        unwarped = warp_points_NeRF(pts_k.to(torch.float32), depth_k.unsqueeze(0), intrinsics.unsqueeze(0), rot_k.unsqueeze(0),
                                    trans_k.unsqueeze(0), rot_j.unsqueeze(0), trans_j.unsqueeze(0), self.device)
        unwarped = filter_points(unwarped.reshape(-1, 2), (H, W), self.device)
        n = len(unwarped)
        return ctx.nerf_splat(prob_k, unwarped.to(torch.float32).contiguous(), pts_k[:n].contiguous())

    @torch.no_grad()
    def fuse_per_pair(self, prob, kp, cnt, data, targets, offsets, sources):
        """What spn_nerf_fuse computes, one ``reproject`` per (target, source) pair as export.py:322-325 does:
        -> (n_targets,H,W) = stack([prob[j]] + splats).sum(0) / (1 + n) per target."""
        raw, K = data["raw"], data["camera_intrinsic_matrix"]
        out = []
        for t, j in enumerate(targets):
            maps = [prob[j]]
            for k in sources[offsets[t]:offsets[t + 1]]:
                maps.append(self.reproject(prob[k], kp[k, :cnt[k]], raw["input_depth"][k], K[j], raw["input_rotation"][k],
                                           raw["input_translation"][k], raw["input_rotation"][j], raw["input_translation"][j]))
            out.append(torch.stack(maps).sum(0) / float(len(maps)))
        return torch.stack(out)

    @torch.no_grad()
    def export_NeRF(self):
        import random
        dh = self.config["model"]["detector_head"]
        for _, data in enumerate(tqdm(self.dataloader, desc="Exporting NeRF Labels", colour="green")):
            data = move_to_device(data, self.device)
            names = data["name"]
            todo = [j for j in range(len(names)) if not Path(self.output_dir, f"{names[j]}.npy").exists()]
            if not todo:
                continue
            out = self.model(data["raw"]["image"], keypoints=True)["detector_output"]      # every view forwarded once
            prob, kp, cnt = out["prob_heatmap"], out["keypoints"], out["keypoint_count"].cpu().numpy()
            if cnt.max(initial=0) > kp.shape[1]:
                raise RuntimeError("keypoint list overflow: set detector_head.top_k")
            # the targets and their source views, drawn in the reference's order (export.py:316-321); a view whose file
            # exists - or that an earlier view of the batch with the same name will write - is skipped without a draw
            targets, offsets, sources, paths, planned = [], [0], [], [], set()
            for j in range(len(names)):
                save_path = Path(self.output_dir, f"{names[j]}.npy")
                if save_path.exists() or save_path in planned:
                    continue
                other_index = [k for k in range(len(names)) if k != j]
                other_index = random.choices(other_index, k=int(0.75 * len(other_index)))     # export.py:320-321, python's RNG
                targets.append(j)
                sources += other_index
                offsets.append(len(sources))
                paths.append(save_path)
                planned.add(save_path)
            raw = data["raw"]
            ctx = self.model.native()
            mean = ctx.nerf_fuse(prob, kp, out["keypoint_count"], raw["input_depth"].to(torch.float32),
                                 data["camera_intrinsic_matrix"].to(torch.float32), raw["input_rotation"].to(torch.float32),
                                 raw["input_translation"].to(torch.float32), targets, offsets, sources)
            for path, kp_t in zip(paths, self._keypoints(ctx, mean, dh)):
                np.save(path, kp_t)

    @staticmethod
    def _keypoints(ctx, heat, dh):
        """box_nms + threshold + nonzero of every fused heatmap (export.py:326-334): one batched call, one copy to the
        host (-> list of (N,2) int64 arrays)."""
        cap = min(heat[0].numel(), 16384)
        for _ in range(2):
            r = ctx.box_nms(heat, float(dh["nms"]), 0.1, float(dh["det_thresh"]), int(dh["top_k"]),
                            det_thresh=float(dh["det_thresh"]), want_map=False, max_kp=cap)
            kp_h = torch.empty(r["kp"].shape, dtype=torch.int32, pin_memory=True)
            cnt_h = torch.empty(r["kp_count"].shape, dtype=torch.int32, pin_memory=True)
            kp_h.copy_(r["kp"], non_blocking=True)
            cnt_h.copy_(r["kp_count"], non_blocking=True)
            torch.cuda.current_stream(heat.device).synchronize()
            counts = cnt_h.numpy()
            if counts.max(initial=0) <= cap:
                break
            cap = int(counts.max())                   # more keypoints than the list holds: redo with the true size
        kp = kp_h.numpy()
        return [kp[i, :counts[i]].astype(np.int64) for i in range(len(counts))]


def load_packed_labels(directory):
    """Read every ``packed_rank*.npz`` shard of an ExportDetections run -> {name: (N,2) int64 (row, col)} - the same
    arrays the per-image ``<name>.npy`` files hold (what data/COCO.py:100-102 of the reference loads as labels)."""
    out = {}
    for f in sorted(Path(directory).glob("packed_rank*.npz")):
        z = np.load(f)
        off = z["offsets"]
        for i, name in enumerate(z["names"]):
            out[str(name)] = z["keypoints"][off[i]:off[i + 1]].astype(np.int64)
    return out
