"""ctypes binding of include/spn_b200.h, include/spn_jpeg.h, include/spn_nerf.h, include/spn_posed.h, include/spn_match.h, include/spn_retrieval.h, include/spn_verify.h and include/spn_tracks.h.  PyTorch is used only for device memory and streams."""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

import torch

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libspn_b200.so"

MODE_FP32, MODE_F16, MODE_BF16, MODE_F16X3 = 0, 1, 2, 3
MODES = {"fp32": MODE_FP32, "f16": MODE_F16, "fp16": MODE_F16, "bf16": MODE_BF16, "f16x3": MODE_F16X3, "strict_tc": MODE_F16X3}

LAYER_PREFIXES = [
    "backbone.block_1", "backbone.block_2", "backbone.block_3", "backbone.block_4",
    "backbone.block_5", "backbone.block_6", "backbone.block_7", "backbone.block_8",
    "detector_head.convPa", "detector_head.convPb", "descriptor_head.convDa", "descriptor_head.convDb",
]


class NativeError(RuntimeError):
    pass


class HomographyParams(C.Structure):
    _fields_ = [("translation", C.c_int), ("rotation", C.c_int), ("scaling", C.c_int), ("perspective", C.c_int),
                ("scaling_amplitude", C.c_float), ("perspective_amplitude_x", C.c_float),
                ("perspective_amplitude_y", C.c_float), ("patch_ratio", C.c_float), ("max_angle", C.c_float),
                ("translation_overflow", C.c_float), ("n_scales", C.c_int), ("n_angles", C.c_int),
                ("allow_artifacts", C.c_int)]


_vp, _i, _f = C.c_void_p, C.c_int, C.c_float
# name -> (restype, argtypes); must list every symbol include/spn_b200.h declares
PROTOTYPES = {
    "spn_last_error": (C.c_char_p, []),
    "spn_version": (_i, []),
    "spn_create": (_i, [C.POINTER(_vp), _i]),
    "spn_destroy": (_i, [_vp]),
    "spn_set_option": (_i, [_vp, C.c_char_p, _i]),
    "spn_pack_weights": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _vp]),
    "spn_conv_layer": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "spn_encoder_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "spn_encoder_forward_ha": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "spn_detector_head_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "spn_descriptor_head_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "spn_dense_descriptors": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "spn_sample_descriptors": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "spn_detect_describe": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "spn_box_nms_topk": (_i, [_vp, _vp, _i, _i, _i, _f, _f, _f, _i, _f, _vp, _vp, _vp, _vp, _i, _vp]),
    "spn_nms_stats": (_i, [_vp, _i, _i, _i, _vp]),
    "spn_check_guards": (_i, [_vp, _vp]),
    "spn_warp_batch": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "spn_ha_aggregate": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "spn_sample_homographies": (_i, [_vp, C.POINTER(HomographyParams), C.c_uint64, C.c_uint64, _i, _i, _i, _vp, _vp, _vp]),
    "spn_resize_crop": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp]),
    "spn_invert3x3": (_i, [_vp, _vp, _i, _vp, _vp]),
    "spn_kornia_matrices": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "spn_select_keypoints": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "spn_repeatability_counts": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, C.c_double, _vp, _vp]),
    "spn_mutual_nn_match": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "spn_detector_labels": (_i, [_vp, _vp, _vp, _vp, C.c_uint64, _i, _i, _i, _vp, _vp, _vp]),
    "spn_nerf_splat": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "spn_launch_count": (C.c_int64, [_vp]),
    "spn_profile_enable": (_i, [_vp, _i]),
    "spn_profile_read": (_i, [_vp, _vp, _vp]),
}

# name -> (restype, argtypes); must list every symbol include/spn_jpeg.h declares
JPEG_PROTOTYPES = {
    "spn_jpeg_plan": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "spn_jpeg_decode_gray": (_i, [_vp, _vp, _vp, _i, _vp, C.c_int64, _vp, _vp, _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_nerf.h declares
NERF_PROTOTYPES = {
    "spn_nerf_fuse": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_posed.h declares
POSED_PROTOTYPES = {
    "spn_posed_reproject": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, C.c_double, _vp, _vp, _vp, _vp, _vp,
                                 _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_match.h declares
MATCH_PROTOTYPES = {
    "spn_match_pairs": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _f, _f, _vp, _vp, _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_retrieval.h declares
RETRIEVAL_PROTOTYPES = {
    "spn_knn": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "spn_residual_sums": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_verify.h declares
VERIFY_PROTOTYPES = {
    "spn_verify_pairs": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _vp, C.c_int64, _i, C.c_double, C.c_double, _i, C.c_uint64, _vp, _vp,
                              _vp, _vp, _vp, _vp]),
}
# name -> (restype, argtypes); must list every symbol include/spn_tracks.h declares
TRACKS_PROTOTYPES = {
    "spn_track_labels": (_i, [_vp, _vp, C.c_int64, C.c_int32, _i, _vp, _vp, _vp]),
    "spn_track_table": (_i, [_vp, _vp, C.c_int32, _vp, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}
JPEG_OK, JPEG_UNSUPPORTED, JPEG_MALFORMED = 0, 1, 2
JPEG_INFO_FIELDS = 5

_lib = None
_lock = threading.Lock()


def library_path() -> Path:
    return _LIB_PATH


def load_library():
    """dlopen libspn_b200.so and bind every prototype.  Fails loudly (no fallback) if it is missing."""
    global _lib
    with _lock:
        if _lib is None:
            if not _LIB_PATH.exists():
                # build on demand (nvcc, in-tree); still no fallback: without nvcc or on failure this raises
                try:
                    import importlib.util
                    spec = importlib.util.spec_from_file_location("spn_build", _HERE / "build.py")
                    mod = importlib.util.module_from_spec(spec)
                    spec.loader.exec_module(mod)
                    mod.build()
                except Exception as e:
                    raise NativeError(f"{_LIB_PATH} not found and building it failed ({e}); build it with "
                                      "`python superpoint-nerf-pytorch_b200/build.py` (there is no CPU/PyTorch fallback)")
            lib = C.CDLL(str(_LIB_PATH))
            for name, (res, args) in (PROTOTYPES | JPEG_PROTOTYPES | NERF_PROTOTYPES | POSED_PROTOTYPES | MATCH_PROTOTYPES |
                                       RETRIEVAL_PROTOTYPES | VERIFY_PROTOTYPES | TRACKS_PROTOTYPES).items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            _lib = lib
    return _lib


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device=None):
    """torch's current stream ON THE GIVEN DEVICE (not on torch's current device, which may be another GPU)."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _chk_dev(t: torch.Tensor, dtype, name, device=None):
    if not (torch.is_tensor(t) and t.is_cuda):
        raise NativeError(f"{name} must be a CUDA tensor (no CPU fallback)")
    if device is not None and t.device.index != device:
        raise NativeError(f"{name} lives on cuda:{t.device.index} but this context owns cuda:{device}")
    if t.dtype != dtype:
        raise NativeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise NativeError(f"{name} must be contiguous (strides {t.stride()} for shape {tuple(t.shape)})")


def _dense(t):
    """Row-major dense view of a tensor (copies only if needed) - the C ABI takes dense arrays."""
    return None if t is None else t.contiguous()


def jpeg_plan(data, offsets):
    """spn_jpeg_plan (host only, no GPU needed): data = the files back to back (contiguous uint8 numpy), offsets (n+1,)
    int64 -> (plan blob uint8 numpy, info (n, 5) int64 numpy {status, height, width, luma blocks, output offset},
    coef_bytes, out_bytes)."""
    import numpy as np
    lib = load_library()
    data = np.ascontiguousarray(data, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    info = np.zeros((n, JPEG_INFO_FIELDS), np.int64)
    totals = np.zeros(2, np.int64)
    size = C.c_int64(0)
    args = (C.c_void_p(data.ctypes.data) if data.size else None, C.c_void_p(offsets.ctypes.data), n)
    tail = (C.c_void_p(info.ctypes.data), C.c_void_p(totals.ctypes.data))
    for plan in (None, True):
        if plan is not None:
            plan = np.empty(size.value, np.uint8)
        rc = lib.spn_jpeg_plan(*args, None if plan is None else C.c_void_p(plan.ctypes.data), C.byref(size), *tail)
        if rc != 0:
            raise NativeError(f"spn_jpeg_plan failed ({rc}): {lib.spn_last_error().decode(errors='replace')}")
    return plan, info, int(totals[0]), int(totals[1])


class Context:
    """Owns one spn_ctx (device weights + workspace) on one GPU."""

    def __init__(self, device: int | None = None):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise NativeError("CUDA is not available: superpoint-nerf-pytorch_b200 has no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else int(device)
        h = C.c_void_p()
        self._call("spn_create", C.byref(h), self.device)
        self.handle = h
        self._weights_key = None

    def _s(self):
        return _stream(self.device)

    def _call(self, name, *args):
        rc = getattr(self.lib, name)(*args)
        if rc != 0:
            raise NativeError(f"{name} failed ({rc}): {self.lib.spn_last_error().decode(errors='replace')}")

    def close(self):
        if getattr(self, "handle", None):
            self.lib.spn_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: int):
        """Options of the tensor-core path: 'fuse_front', 'fuse_head' (default 1), 'ws_guard' (default 0)."""
        self._call("spn_set_option", self.handle, name.encode(), int(value))

    @property
    def launches(self) -> int:
        return int(self.lib.spn_launch_count(self.handle))

    PROF_SLOTS = 24
    PROF_NAMES = {i: n for i, n in enumerate(LAYER_PREFIXES)} | {12: "warp_batch", 13: "ha_aggregate", 14: "box_nms",
                                                                 15: "softmax_d2s", 16: "dense_desc", 17: "prep", 18: "sampler"}

    def profile_enable(self, on: bool):
        self._call("spn_profile_enable", self.handle, 1 if on else 0)

    def profile_read(self):
        """-> {kernel name: (total ms, launches)} since the last read (CUDA events recorded inside the library)."""
        ms = (C.c_float * self.PROF_SLOTS)()
        cnt = (C.c_int64 * self.PROF_SLOTS)()
        self._call("spn_profile_read", self.handle, C.cast(ms, C.c_void_p), C.cast(cnt, C.c_void_p))
        return {self.PROF_NAMES.get(i, f"slot{i}"): (float(ms[i]), int(cnt[i])) for i in range(self.PROF_SLOTS) if cnt[i]}

    # ---- weights -------------------------------------------------------------------------------
    def load_state_dict(self, sd: dict, eps: float = 1e-5):
        """Fold BN and upload every VGG_Block present in a reference-format state dict (engine.py:108-117)."""
        for lid, pre in enumerate(LAYER_PREFIXES):
            if f"{pre}.conv2d.weight" not in sd:
                continue
            get = lambda k: sd[f"{pre}.{k}"].detach().to("cpu", torch.float32).contiguous()  # noqa: E731
            w, b = get("conv2d.weight"), get("conv2d.bias")
            g, be, mu, var = get("norm.weight"), get("norm.bias"), get("norm.running_mean"), get("norm.running_var")
            cout, cin, k, _ = w.shape
            self._call("spn_pack_weights", self.handle, lid, _ptr(w), _ptr(b), _ptr(g), _ptr(be), _ptr(mu), _ptr(var),
                       C.c_float(eps), cout, cin, k, self._s())

    def conv_layer(self, layer: int, x: torch.Tensor, mode: int, relu=True, pool=False, cout=None):
        """One VGG_Block (conv + folded BN [+ ReLU] [+ 2x2 max-pool]) on NCHW fp32 tensors."""
        x = _dense(x)
        _chk_dev(x, torch.float32, "x", self.device)
        B, _, H, W = x.shape
        out = torch.empty((B, cout, H // 2 if pool else H, W // 2 if pool else W), dtype=torch.float32, device=x.device)
        self._call("spn_conv_layer", self.handle, layer, mode, _ptr(x), B, H, W, int(relu), int(pool), _ptr(out), self._s())
        return out

    # ---- forward -------------------------------------------------------------------------------
    def encoder_forward(self, images: torch.Tensor, mode: int):
        images = _dense(images)
        _chk_dev(images, torch.float32, "images", self.device)
        B, H, W = images.shape
        self._call("spn_encoder_forward", self.handle, _ptr(images), B, H, W, mode, self._s())

    def encoder_forward_ha(self, images: torch.Tensor, hinv, slot_begin: int, n_slots: int, mode: int):
        """Fused warp + encoder for slots [slot_begin, slot_begin+n_slots) of (images (NI,H,W), hinv (NI,n_h,3,3))."""
        images, hinv = _dense(images), _dense(hinv)
        _chk_dev(images, torch.float32, "images", self.device)
        NI, H, W = images.shape
        n_h = 0 if hinv is None else hinv.shape[1]
        if n_h:
            _chk_dev(hinv, torch.float32, "hinv", self.device)
        self._call("spn_encoder_forward_ha", self.handle, _ptr(images), NI, _ptr(hinv) if n_h else None, n_h, int(slot_begin),
                   int(n_slots), H, W, mode, self._s())

    def detector_head_forward(self, B, H, W, mode, mask=None, want_logits=False, out=None):
        dev = torch.device("cuda", self.device)
        if out is None:
            prob = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        else:
            _chk_dev(out, torch.float32, "out", self.device)
            if tuple(out.shape) != (B, H, W):
                raise NativeError(f"out must be {(B, H, W)}, got {tuple(out.shape)}")
            prob = out
        logits = torch.empty((B, 65, H // 8, W // 8), dtype=torch.float32, device=dev) if want_logits else None
        if mask is not None:
            mask = _dense(mask)
            _chk_dev(mask, torch.uint8, "mask", self.device)
        self._call("spn_detector_head_forward", self.handle, B, H, W, mode, _ptr(mask), _ptr(logits), _ptr(prob), self._s())
        return prob, logits

    def descriptor_head_forward(self, B, H, W, mode):
        raw = torch.empty((B, 256, H // 8, W // 8), dtype=torch.float32, device=torch.device("cuda", self.device))
        self._call("spn_descriptor_head_forward", self.handle, B, H, W, mode, _ptr(raw), self._s())
        return raw

    def dense_descriptors(self, raw: torch.Tensor, grid: int):
        raw = _dense(raw)
        _chk_dev(raw, torch.float32, "desc_raw", self.device)
        B, Cc, Hc, Wc = raw.shape
        out = torch.empty((B, Cc, Hc * grid, Wc * grid), dtype=torch.float32, device=raw.device)
        self._call("spn_dense_descriptors", self.handle, _ptr(raw), B, Cc, Hc, Wc, grid, _ptr(out), self._s())
        return out

    def sample_descriptors(self, raw, grid, kp, kp_count, interp="bicubic"):
        raw, kp, kp_count = _dense(raw), _dense(kp), _dense(kp_count)
        _chk_dev(raw, torch.float32, "desc_raw", self.device)
        _chk_dev(kp, torch.int32, "kp", self.device)
        _chk_dev(kp_count, torch.int32, "kp_count", self.device)
        B, Cc, Hc, Wc = raw.shape
        max_kp = kp.shape[1]
        out = torch.empty((B, max_kp, Cc), dtype=torch.float32, device=raw.device)   # the kernel zeroes rows >= count
        self._call("spn_sample_descriptors", self.handle, _ptr(raw), B, Cc, Hc, Wc, grid, _ptr(kp), _ptr(kp_count), max_kp,
                   0 if interp == "bicubic" else 1, _ptr(out), self._s())
        return out

    def detect_describe(self, images, mode, nms_size, det_thresh, top_k=0, iou=0.1, max_kp=None, descriptors=True,
                        interp="bicubic", want_logits=True, want_map=True, want_pred=True):
        """One-call forward + keypoints (+ sparse descriptors): images (B,H,W) fp32 CUDA -> dict with logits, prob, nms,
        pred, kp (B,max_kp,2) int32 (row, col), kp_count (B,), desc_raw, desc_sparse (B,max_kp,256)."""
        images = _dense(images)
        _chk_dev(images, torch.float32, "images", self.device)
        B, H, W = images.shape
        dev = images.device
        if max_kp is None:
            max_kp = int(top_k) if top_k else min(H * W, 16384)
        f32 = dict(dtype=torch.float32, device=dev)
        out = {"logits": torch.empty((B, 65, H // 8, W // 8), **f32) if want_logits else None,
               "prob": torch.empty((B, H, W), **f32),
               "nms": torch.empty((B, H, W), **f32) if want_map else None,
               "pred": torch.empty((B, H, W), dtype=torch.int32, device=dev) if want_pred else None,
               "kp": torch.empty((B, max_kp, 2), dtype=torch.int32, device=dev),
               "kp_count": torch.empty((B,), dtype=torch.int32, device=dev),
               "desc_raw": torch.empty((B, 256, H // 8, W // 8), **f32) if descriptors else None,
               "desc_sparse": torch.empty((B, max_kp, 256), **f32) if descriptors else None}
        self._call("spn_detect_describe", self.handle, _ptr(images), B, H, W, mode, C.c_float(nms_size), C.c_float(iou),
                   C.c_float(det_thresh), int(top_k), 0 if interp == "bicubic" else 1, _ptr(out["logits"]), _ptr(out["prob"]),
                   _ptr(out["nms"]), _ptr(out["pred"]), _ptr(out["kp"]), _ptr(out["kp_count"]), int(max_kp), _ptr(out["desc_raw"]),
                   _ptr(out["desc_sparse"]), self._s())
        return out

    def box_nms(self, prob, size, iou=0.1, min_prob=0.01, top_k=0, det_thresh=None, want_map=True, want_pred=False,
                max_kp=0):
        """prob (B,H,W).  Returns dict(nms, pred, kp, kp_count) with the requested members."""
        prob = _dense(prob)
        _chk_dev(prob, torch.float32, "prob", self.device)
        B, H, W = prob.shape
        dev = prob.device
        det = float(min_prob if det_thresh is None else det_thresh)
        out = {"nms": torch.empty_like(prob) if want_map else None,
               "pred": torch.empty((B, H, W), dtype=torch.int32, device=dev) if want_pred else None,
               "kp": torch.zeros((B, max_kp, 2), dtype=torch.int32, device=dev) if max_kp else None,
               "kp_count": torch.zeros((B,), dtype=torch.int32, device=dev) if max_kp else None}
        self._call("spn_box_nms_topk", self.handle, _ptr(prob), B, H, W, C.c_float(size), C.c_float(iou), C.c_float(min_prob),
                   int(top_k), C.c_float(det), _ptr(out["nms"]), _ptr(out["pred"]), _ptr(out["kp"]), _ptr(out["kp_count"]),
                   int(max_kp), self._s())
        return out

    def check_guards(self):
        """Number of guard bytes (bands around the workspace / scratch buffer, gaps between the carved regions when
        option ``ws_guard`` is on) that a kernel overwrote; 0 = none.  Synchronises the device."""
        out = (C.c_int64 * 1)()
        self._call("spn_check_guards", self.handle, C.cast(out, C.c_void_p))
        return int(out[0])

    def nms_stats(self, B, H, W):
        out = (C.c_int64 * 4)()
        self._call("spn_nms_stats", self.handle, B, H, W, C.cast(out, C.c_void_p))
        return {"global_rounds": int(out[0]), "local_iterations": int(out[1]), "tile_visits": int(out[2])}

    # ---- homography adaptation -------------------------------------------------------------------
    def warp_batch(self, images, hinv, margin, want_warped=True):
        """images (NI,H,W), hinv (NI,n_h,3,3) = kornia sampling matrices (``kornia_matrices`` / utils.kornia_geometry
        ``fwd``) -> warped (NI*(n_h+1),H,W) fp32 (None if not wanted), mask u8 (same shape)."""
        images, hinv = _dense(images), _dense(hinv)
        _chk_dev(images, torch.float32, "images", self.device)
        NI, H, W = images.shape
        n_h = 0 if hinv is None else hinv.shape[1]
        if n_h:
            _chk_dev(hinv, torch.float32, "hinv", self.device)
        warped = torch.empty((NI * (n_h + 1), H, W), dtype=torch.float32, device=images.device) if want_warped else None
        mask = torch.empty((NI * (n_h + 1), H, W), dtype=torch.uint8, device=images.device)
        self._call("spn_warp_batch", self.handle, _ptr(images), NI, _ptr(hinv) if n_h else None, n_h, H, W, int(margin),
                   _ptr(warped), _ptr(mask), self._s())
        return warped, mask

    def ha_aggregate(self, probs, h, margin, aggregation="sum"):
        """probs (NI,n_h+1,H,W) masked heatmaps, h (NI,n_h,3,3) = kornia sampling matrices of the inverse homographies
        (``bwd``) -> (NI,H,W)."""
        probs, h = _dense(probs), _dense(h)
        _chk_dev(probs, torch.float32, "probs", self.device)
        NI, n1, H, W = probs.shape
        n_h = n1 - 1
        if n_h:
            _chk_dev(h, torch.float32, "h", self.device)
        out = torch.empty((NI, H, W), dtype=torch.float32, device=probs.device)
        self._call("spn_ha_aggregate", self.handle, _ptr(probs), _ptr(h) if n_h else None, NI, n_h, H, W, int(margin),
                   1 if aggregation == "max" else 0, _ptr(out), self._s())
        return out

    def sample_homographies(self, params: dict, seed: int, first_index: int, count: int, H: int, W: int):
        p = HomographyParams(
            int(params.get("translation", True)), int(params.get("rotation", True)), int(params.get("scaling", True)),
            int(params.get("perspective", True)), float(params.get("scaling_amplitude", 0.1)),
            float(params.get("perspective_amplitude_x", 0.1)), float(params.get("perspective_amplitude_y", 0.1)),
            float(params.get("patch_ratio", 0.5)), float(params.get("max_angle", 1.57)),
            float(params.get("translation_overflow", 0.0)), int(params.get("n_scales", 5)), int(params.get("n_angles", 25)),
            int(params.get("allow_artifacts", False)))
        dev = torch.device("cuda", self.device)
        h = torch.empty((count, 3, 3), dtype=torch.float32, device=dev)
        hinv = torch.empty((count, 3, 3), dtype=torch.float32, device=dev)
        self._call("spn_sample_homographies", self.handle, C.byref(p), C.c_uint64(seed), C.c_uint64(first_index), count, H, W,
                   _ptr(h), _ptr(hinv), self._s())
        return h, hinv

    def kornia_matrices(self, h, H, W):
        """h (...,3,3) fp32 CUDA pixel-space homographies -> (fwd, bwd) kornia sampling matrices, device arithmetic
        (spn_kornia_matrices).  Host homographies: utils.kornia_geometry.sampling_matrices (the reference's bits)."""
        h = _dense(h)
        _chk_dev(h, torch.float32, "h", self.device)
        fwd, bwd = torch.empty_like(h), torch.empty_like(h)
        self._call("spn_kornia_matrices", self.handle, _ptr(h), h.numel() // 9, int(H), int(W), _ptr(fwd), _ptr(bwd), self._s())
        return fwd, bwd

    def detector_labels(self, kpts_heatmap, valid_mask=None, noise=None, seed=0):
        """utils/losses.py:13-27 label building: kpts_heatmap (B,H,W) int32, valid_mask (B,H,W) int32 or None, noise
        (B,65,H/8,W/8) fp32 or None -> (labels (B,H/8,W/8) int64, valid cells (B,H/8,W/8) fp32)."""
        kpts_heatmap = _dense(kpts_heatmap)
        _chk_dev(kpts_heatmap, torch.int32, "kpts_heatmap", self.device)
        B, H, W = kpts_heatmap.shape
        if valid_mask is not None:
            valid_mask = _dense(valid_mask)
            _chk_dev(valid_mask, torch.int32, "valid_mask", self.device)
        if noise is not None:
            noise = _dense(noise)
            _chk_dev(noise, torch.float32, "noise", self.device)
        labels = torch.empty((B, H // 8, W // 8), dtype=torch.int64, device=kpts_heatmap.device)
        cells = torch.empty((B, H // 8, W // 8), dtype=torch.float32, device=kpts_heatmap.device)
        self._call("spn_detector_labels", self.handle, _ptr(kpts_heatmap), _ptr(valid_mask), _ptr(noise), C.c_uint64(seed), B, H, W,
                   _ptr(labels), _ptr(cells), self._s())
        return labels, cells

    def nerf_splat(self, prob_src, dst_pts, src_pts):
        """ExportNeRFDetections.step splat: prob_src (H,W) fp32, dst_pts (n,2) fp32, src_pts (n,2) int32 -> (H,W) fp32."""
        prob_src = _dense(prob_src)
        _chk_dev(prob_src, torch.float32, "prob_src", self.device)
        H, W = prob_src.shape
        n = int(dst_pts.shape[0])
        if n:
            dst_pts, src_pts = _dense(dst_pts), _dense(src_pts)
            _chk_dev(dst_pts, torch.float32, "dst_pts", self.device)
            _chk_dev(src_pts, torch.int32, "src_pts", self.device)
        out = torch.empty((H, W), dtype=torch.float32, device=prob_src.device)
        self._call("spn_nerf_splat", self.handle, _ptr(prob_src), _ptr(dst_pts) if n else None, _ptr(src_pts) if n else None, n, H, W,
                   _ptr(out), self._s())
        return out

    def nerf_fuse(self, prob, kp, kp_count, depth, K, R, t, targets, offsets, sources):
        """Fused NeRF label heatmaps of one batch (spn_nerf_fuse): prob (V,H,W) fp32, kp (V,max_kp,2) int32 (row, col),
        kp_count (V,) int32, depth (V,H,W) fp32, K / R (V,3,3) fp32, t (V,3,1) or (V,3) fp32, all CUDA; targets (n,)
        view indices, offsets (n+1,) and sources (offsets[n],) the CSR list of each target's source views (host
        sequences).  -> (n,H,W): out[i] = (prob[targets[i]] + sum of the source splats, in order) / (1 + n_sources)."""
        import numpy as np
        prob, kp, kp_count, depth = _dense(prob), _dense(kp), _dense(kp_count), _dense(depth)
        for x, dt, name in ((prob, torch.float32, "prob"), (kp, torch.int32, "kp"), (kp_count, torch.int32, "kp_count"),
                            (depth, torch.float32, "depth")):
            _chk_dev(x, dt, name, self.device)
        V, H, W = prob.shape
        if kp.dim() != 3 or kp.shape[0] != V or kp.shape[2] != 2 or tuple(kp_count.shape) != (V,) or tuple(depth.shape) != (V, H, W):
            raise NativeError(f"nerf_fuse: kp {tuple(kp.shape)}, kp_count {tuple(kp_count.shape)}, depth {tuple(depth.shape)} "
                              f"do not match prob {(V, H, W)}")
        mats = []
        for x, n, name in ((K, 9, "K"), (R, 9, "R"), (t, 3, "t")):
            x = _dense(x)
            _chk_dev(x, torch.float32, name, self.device)
            if x.numel() != V * n:
                raise NativeError(f"nerf_fuse: {name} has shape {tuple(x.shape)}, expected {V} x {n} values")
            mats.append(x)
        tg = np.ascontiguousarray(np.asarray(targets, dtype=np.int64).reshape(-1).astype(np.int32))
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1).astype(np.int32))
        src = np.ascontiguousarray(np.asarray(sources, dtype=np.int64).reshape(-1).astype(np.int32))
        if len(off) != len(tg) + 1 or (len(off) and int(off[-1]) != len(src)):
            raise NativeError(f"nerf_fuse: {len(tg)} targets need {len(tg) + 1} offsets ending at len(sources) = {len(src)}, "
                              f"got {off.tolist()[:8]}{'...' if len(off) > 8 else ''}")
        out = torch.empty((len(tg), H, W), dtype=torch.float32, device=prob.device)
        hp = lambda a: C.c_void_p(a.ctypes.data) if a.size else None  # noqa: E731
        self._call("spn_nerf_fuse", self.handle, _ptr(prob), _ptr(kp), _ptr(kp_count), int(kp.shape[1]), _ptr(depth), *map(_ptr, mats),
                   V, H, W, len(tg), hp(tg), hp(off), hp(src), _ptr(out), self._s())
        return out

    # ---- on-GPU evaluation (evaluations/*.py of the reference) -----------------------------------
    def posed_reproject(self, kp, kp_count, depth, K, R, t, pairs, depth_tol):
        """Keypoints of view a reprojected into view b for every pair (spn_posed_reproject): kp (V,max_kp,2) int32 (row,
        col), kp_count (V,) int32, depth (V,H,W) fp32 ray depth, K / R (V,3,3) fp32, t (V,3,1) or (V,3) fp32, all CUDA;
        pairs (P,2) host (a, b) view indices.  -> dict with proj (P,max_kp,2) float64 (a's keypoints in b, NaN where
        undefined), vis (P,2,max_kp) int32 (a visible in b, b visible in a), set1 / set2 (P,max_kp,2) float64 (the
        compacted visible points, both in b's frame) and set_count (P,2) int32."""
        import numpy as np
        kp, kp_count, depth = _dense(kp), _dense(kp_count), _dense(depth)
        for x, dt, name in ((kp, torch.int32, "kp"), (kp_count, torch.int32, "kp_count"), (depth, torch.float32, "depth")):
            _chk_dev(x, dt, name, self.device)
        if depth.dim() != 3 or kp.dim() != 3 or kp.shape[0] != depth.shape[0] or kp.shape[2] != 2 or \
                tuple(kp_count.shape) != (depth.shape[0],):
            raise NativeError(f"posed_reproject: kp {tuple(kp.shape)}, kp_count {tuple(kp_count.shape)} do not match depth "
                              f"{tuple(depth.shape)} (V,H,W)")
        V, H, W = depth.shape
        mats = []
        for x, n, name in ((K, 9, "K"), (R, 9, "R"), (t, 3, "t")):
            x = _dense(x)
            _chk_dev(x, torch.float32, name, self.device)
            if x.numel() != V * n:
                raise NativeError(f"posed_reproject: {name} has shape {tuple(x.shape)}, expected {V} x {n} values")
            mats.append(x)
        pr = np.asarray(pairs, dtype=np.int64)
        if pr.size == 0:
            pr = pr.reshape(0, 2)
        if pr.ndim != 2 or pr.shape[1] != 2:
            raise NativeError(f"posed_reproject: pairs must be (P, 2), got shape {pr.shape}")
        pr = np.ascontiguousarray(pr.astype(np.int32))
        P, max_kp = len(pr), int(kp.shape[1])
        f64 = dict(dtype=torch.float64, device=depth.device)
        out = {"proj": torch.empty((P, max_kp, 2), **f64), "vis": torch.empty((P, 2, max_kp), dtype=torch.int32, device=depth.device),
               "set1": torch.empty((P, max_kp, 2), **f64), "set2": torch.empty((P, max_kp, 2), **f64),
               "set_count": torch.empty((P, 2), dtype=torch.int32, device=depth.device)}
        self._call("spn_posed_reproject", self.handle, _ptr(kp), _ptr(kp_count), max_kp, _ptr(depth), *map(_ptr, mats), V, H, W, P,
                   C.c_void_p(pr.ctypes.data) if P else None, C.c_double(float(depth_tol)),
                   *[_ptr(out[k]) if P else None for k in ("proj", "vis", "set1", "set2", "set_count")], self._s())
        return out

    SELECT_CAP = 16384

    def select_keypoints(self, prob, warp=None, bounds=None, emit_warped=False, keep_k=300):
        """prob (B,H,W) fp32 CUDA NMS'd heatmaps; warp: (B,3,3) float64 numpy / tensor on the HOST or None.
        -> (pts (B,keep_k,2) float64 (row, col), score (B,keep_k), count (B,) int32): select_k_best order (ascending)."""
        import numpy as np
        prob = _dense(prob)
        _chk_dev(prob, torch.float32, "prob", self.device)
        B, H, W = prob.shape
        bh, bw = (H, W) if bounds is None else (int(bounds[0]), int(bounds[1]))
        wptr = None
        if warp is not None:
            w = np.ascontiguousarray(np.asarray(warp, dtype=np.float64).reshape(B, 9))
            wptr = C.c_void_p(w.ctypes.data)
        dev = prob.device
        pts = torch.zeros((B, keep_k, 2), dtype=torch.float64, device=dev)
        score = torch.zeros((B, keep_k), dtype=torch.float32, device=dev)
        count = torch.zeros((2 * B,), dtype=torch.int32, device=dev)
        self._call("spn_select_keypoints", self.handle, _ptr(prob), B, H, W, wptr, bh, bw, int(bool(emit_warped)), int(keep_k),
                   _ptr(pts), _ptr(score), _ptr(count), self._s())
        return pts, score, count

    def repeatability_counts(self, pts1, n1, pts2, n2, thresh):
        """-> (B,4) int32 {N1, N2, count1, count2}."""
        pts1, pts2 = _dense(pts1), _dense(pts2)
        _chk_dev(pts1, torch.float64, "pts1", self.device)
        _chk_dev(pts2, torch.float64, "pts2", self.device)
        B, cap, _ = pts1.shape
        if pts2.shape[1] != cap:
            raise NativeError("repeatability_counts: both point sets must have the same capacity")
        out = torch.zeros((B, 4), dtype=torch.int32, device=pts1.device)
        self._call("spn_repeatability_counts", self.handle, _ptr(pts1), _ptr(_dense(n1)), _ptr(pts2), _ptr(_dense(n2)), B, cap,
                   C.c_double(float(thresh)), _ptr(out), self._s())
        return out

    def mutual_nn_match(self, desc1, n1, desc2, n2):
        """desc1 (B,cap1,C), desc2 (B,cap2,C) fp32 CUDA -> (match (B,cap1) int32 train index or -1, dist (B,cap1))."""
        desc1, desc2 = _dense(desc1), _dense(desc2)
        _chk_dev(desc1, torch.float32, "desc1", self.device)
        _chk_dev(desc2, torch.float32, "desc2", self.device)
        B, c1, Cc = desc1.shape
        c2 = desc2.shape[1]
        match = torch.empty((B, c1), dtype=torch.int32, device=desc1.device)
        dist = torch.empty((B, c1), dtype=torch.float32, device=desc1.device)
        self._call("spn_mutual_nn_match", self.handle, _ptr(desc1), _ptr(_dense(n1)), _ptr(desc2), _ptr(_dense(n2)), B, c1, c2, Cc,
                   _ptr(match), _ptr(dist), self._s())
        return match, dist

    MATCH_MAX_PAIRS = 65535

    def match_pairs(self, desc, count, pairs, mutual=True, ratio=0.0, max_dist=float("inf")):
        """Matches of pairs of a descriptor pool (spn_match_pairs, include/spn_match.h): desc (N,cap,C) fp32 and count
        (N,) int32 CUDA (detect_describe's desc_sparse / kp_count), pairs (P,2) host (a, b) set indices, at most
        MATCH_MAX_PAIRS.  -> (match (P,cap) int32 index into b or -1, dist (P,cap) fp32, 0 where there is no match)."""
        import numpy as np
        desc, count = _dense(desc), _dense(count)
        _chk_dev(desc, torch.float32, "desc", self.device)
        _chk_dev(count, torch.int32, "count", self.device)
        if desc.dim() != 3 or tuple(count.shape) != (desc.shape[0],):
            raise NativeError(f"match_pairs: desc {tuple(desc.shape)} must be (N,cap,C) and count {tuple(count.shape)} (N,)")
        pr = np.asarray(pairs, dtype=np.int64)
        if pr.size == 0:
            pr = pr.reshape(0, 2)
        if pr.ndim != 2 or pr.shape[1] != 2:
            raise NativeError(f"match_pairs: pairs must be (P, 2), got shape {pr.shape}")
        if pr.size and (pr.min() < np.iinfo(np.int32).min or pr.max() > np.iinfo(np.int32).max):
            raise NativeError("match_pairs: a pair index does not fit int32")
        pr = np.ascontiguousarray(pr.astype(np.int32))
        N, cap, Cc = desc.shape
        P = len(pr)
        match = torch.empty((P, cap), dtype=torch.int32, device=desc.device)
        dist = torch.empty((P, cap), dtype=torch.float32, device=desc.device)
        self._call("spn_match_pairs", self.handle, _ptr(desc), _ptr(count), N, cap, Cc, C.c_void_p(pr.ctypes.data) if P else None, P,
                   int(bool(mutual)), C.c_float(ratio), C.c_float(max_dist), _ptr(match) if P else None, _ptr(dist) if P else None,
                   self._s())
        return match, dist

    VERIFY_MAX_PAIRS = 65535
    VERIFY_MODELS = {"fundamental": 0, "homography": 1}

    def verify_pairs(self, kp, offsets, matches, pairs, model="fundamental", threshold=3.0, confidence=0.999, max_iters=10000,
                     seed=0):
        """RANSAC per pair (spn_verify_pairs, include/spn_verify.h): kp (N,cap,2) int32 (row, col) keypoint pool, offsets
        (P+1,) int64 and matches (M,2) int32 CUDA (matching.match_pairs' output), pairs (P,2) host (a, b), at most
        VERIFY_MAX_PAIRS; model 'fundamental' or 'homography'.  -> (models (P,3,3) fp64, num_inliers (P,) int32 (-1: the
        pair's offsets or indices are out of range), hypotheses (P,) int32, best (P,) int32, inliers (M,) uint8); inlier
        rows of pairs with out-of-range offsets stay 0."""
        import numpy as np
        if model not in self.VERIFY_MODELS:
            raise NativeError(f"verify_pairs: model must be one of {', '.join(self.VERIFY_MODELS)}, got {model!r}")
        kp, offsets, matches = _dense(kp), _dense(offsets), _dense(matches)
        for x, dt, name in ((kp, torch.int32, "kp"), (offsets, torch.int64, "offsets"), (matches, torch.int32, "matches")):
            _chk_dev(x, dt, name, self.device)
        if kp.dim() != 3 or kp.shape[2] != 2 or matches.dim() != 2 or matches.shape[1] != 2 or offsets.dim() != 1:
            raise NativeError(f"verify_pairs: kp {tuple(kp.shape)} must be (N,cap,2), matches {tuple(matches.shape)} (M,2) and "
                              f"offsets {tuple(offsets.shape)} (P+1,)")
        pr = np.asarray(pairs, dtype=np.int64)
        if pr.size == 0:
            pr = pr.reshape(0, 2)
        if pr.ndim != 2 or pr.shape[1] != 2:
            raise NativeError(f"verify_pairs: pairs must be (P, 2), got shape {pr.shape}")
        if pr.size and (pr.min() < np.iinfo(np.int32).min or pr.max() > np.iinfo(np.int32).max):
            raise NativeError("verify_pairs: a pair index does not fit int32")
        pr = np.ascontiguousarray(pr.astype(np.int32))
        P, M = len(pr), int(matches.shape[0])
        if offsets.shape[0] != P + 1:
            raise NativeError(f"verify_pairs: {P} pairs need {P + 1} offsets, got {offsets.shape[0]}")
        N, cap, _ = kp.shape
        dev = kp.device
        models = torch.zeros((P, 3, 3), dtype=torch.float64, device=dev)
        num, hyp, best = (torch.zeros((P,), dtype=torch.int32, device=dev) for _ in range(3))
        inliers = torch.zeros((M,), dtype=torch.uint8, device=dev)
        self._call("spn_verify_pairs", self.handle, _ptr(kp), N, cap, C.c_void_p(pr.ctypes.data) if P else None, P, _ptr(offsets),
                   _ptr(matches) if M else None, M, self.VERIFY_MODELS[model], C.c_double(threshold), C.c_double(confidence),
                   int(max_iters), C.c_uint64(seed), *[_ptr(x) if P else None for x in (models, num, hyp, best)],
                   _ptr(inliers) if M else None, self._s())
        return models, num, hyp, best, inliers

    TRACKS_MAX_ROWS = 2 ** 31 - 1

    def track_labels(self, edges, K, labels=None):
        """Connected components of a match graph (spn_track_labels, include/spn_tracks.h): edges (E,2) int32 CUDA, rows
        in [0, K).  -> (labels (K,) int32, the smallest row of every row's component; bad (1,) int64, the edges with an
        endpoint outside [0, K), which are not applied).  ``labels``: the labels of an earlier call with the same K; the
        edges are joined into its components in place, so an edge list split over several calls gives the labels of one
        call."""
        edges = _dense(edges)
        _chk_dev(edges, torch.int32, "edges", self.device)
        if edges.dim() != 2 or edges.shape[1] != 2:
            raise NativeError(f"track_labels: edges must be (E, 2), got shape {tuple(edges.shape)}")
        if isinstance(K, bool) or not 1 <= int(K) <= self.TRACKS_MAX_ROWS:
            raise NativeError(f"track_labels: K = {K!r} rows outside [1, {self.TRACKS_MAX_ROWS}]")
        K, E = int(K), int(edges.shape[0])
        resume = labels is not None
        if not resume:
            labels = torch.empty((K,), dtype=torch.int32, device=edges.device)
        else:
            _chk_dev(labels, torch.int32, "labels", self.device)
            if tuple(labels.shape) != (K,):
                raise NativeError(f"track_labels: labels must be ({K},), got shape {tuple(labels.shape)}")
        bad = torch.empty((1,), dtype=torch.int64, device=edges.device)
        self._call("spn_track_labels", self.handle, _ptr(edges) if E else None, C.c_int64(E), K, int(resume), _ptr(labels),
                   _ptr(bad), self._s())
        return labels, bad

    def track_table(self, labels, img_offsets, min_length=2):
        """The track table of component labels (spn_track_table, include/spn_tracks.h): labels (K,) int32 (track_labels),
        img_offsets (N+1,) int64 (image n's rows are img_offsets[n]:img_offsets[n+1]), both CUDA.  -> (track_offsets
        (K//2+1,) int64, obs (K,2) int32 (image, keypoint), consistent (K//2,) uint8, track_of (K,) int32, totals (2,) int64
        (T, O), bad (1,) int64), at their upper bounds: only the first T (+1) / O entries are written."""
        labels, img_offsets = _dense(labels), _dense(img_offsets)
        _chk_dev(labels, torch.int32, "labels", self.device)
        _chk_dev(img_offsets, torch.int64, "img_offsets", self.device)
        if labels.dim() != 1 or img_offsets.dim() != 1 or img_offsets.shape[0] < 2:
            raise NativeError(f"track_table: labels {tuple(labels.shape)} must be (K,) and img_offsets "
                              f"{tuple(img_offsets.shape)} (N+1,) with N >= 1")
        K, N = int(labels.shape[0]), int(img_offsets.shape[0]) - 1
        if not 1 <= K <= self.TRACKS_MAX_ROWS or N >= 2 ** 31 - 1:
            raise NativeError(f"track_table: K = {K} rows outside [1, {self.TRACKS_MAX_ROWS}] or N = {N} images too many")
        if isinstance(min_length, bool) or not isinstance(min_length, int) or min_length < 2:
            raise NativeError(f"track_table: min_length must be an integer >= 2, got {min_length!r}")
        dev = labels.device
        out = (torch.empty((K // 2 + 1,), dtype=torch.int64, device=dev), torch.empty((K, 2), dtype=torch.int32, device=dev),
               torch.empty((K // 2,), dtype=torch.uint8, device=dev), torch.empty((K,), dtype=torch.int32, device=dev),
               torch.empty((2,), dtype=torch.int64, device=dev), torch.empty((1,), dtype=torch.int64, device=dev))
        self._call("spn_track_table", self.handle, _ptr(labels), K, _ptr(img_offsets), N, min(min_length, 2 ** 31 - 1),
                   *[_ptr(x) if x.numel() else None for x in out], self._s())
        return out

    def knn(self, query, train, k, exclude_self=False):
        """The k nearest train rows of every query row (spn_knn, include/spn_retrieval.h): query (nq,C) and train (nt,C)
        fp32 CUDA.  -> (index (nq,k) int32, ascending distance, -1 in slots past the usable train rows; dist2 (nq,k)
        fp32, +inf there).  exclude_self: query and train are the same set and row i is not its own neighbour."""
        query, train = _dense(query), _dense(train)
        _chk_dev(query, torch.float32, "query", self.device)
        _chk_dev(train, torch.float32, "train", self.device)
        if query.dim() != 2 or train.dim() != 2 or query.shape[1] != train.shape[1]:
            raise NativeError(f"knn: query {tuple(query.shape)} and train {tuple(train.shape)} must be (n, C) with the same C")
        nq, Cc = query.shape
        nt = train.shape[0]
        index = torch.empty((nq, k), dtype=torch.int32, device=query.device)
        dist2 = torch.empty((nq, k), dtype=torch.float32, device=query.device)
        self._call("spn_knn", self.handle, _ptr(query) if nq else None, nq, _ptr(train) if nt else None, nt, Cc, int(k),
                   int(bool(exclude_self)), _ptr(index) if nq else None, _ptr(dist2) if nq else None, self._s())
        return index, dist2

    def residual_sums(self, desc, count, assign, words):
        """Per-image, per-word residual sums (spn_residual_sums, include/spn_retrieval.h): desc (N,cap,C) fp32 and count
        (N,) int32 (detect_describe's desc_sparse / kp_count), assign (N,cap) int32 word per row, words (K,C) fp32, all
        CUDA.  -> (sums (N,K,C) fp32: sum of x_i - c_w over the rows assigned to w, in row order; n (N,K) int32)."""
        desc, count, assign, words = _dense(desc), _dense(count), _dense(assign), _dense(words)
        for x, dt, name in ((desc, torch.float32, "desc"), (count, torch.int32, "count"), (assign, torch.int32, "assign"),
                            (words, torch.float32, "words")):
            _chk_dev(x, dt, name, self.device)
        if desc.dim() != 3 or tuple(count.shape) != (desc.shape[0],) or tuple(assign.shape) != tuple(desc.shape[:2]) or \
                words.dim() != 2 or words.shape[1] != desc.shape[2]:
            raise NativeError(f"residual_sums: desc {tuple(desc.shape)} (N,cap,C), count {tuple(count.shape)} (N,), assign "
                              f"{tuple(assign.shape)} (N,cap) and words {tuple(words.shape)} (K,C) do not fit together")
        N, cap, Cc = desc.shape
        K = words.shape[0]
        sums = torch.empty((N, K, Cc), dtype=torch.float32, device=desc.device)
        n = torch.empty((N, K), dtype=torch.int32, device=desc.device)
        self._call("spn_residual_sums", self.handle, *[_ptr(x) if N else None for x in (desc, count, assign, words)], N, cap, Cc, K,
                   _ptr(sums) if N else None, _ptr(n) if N else None, self._s())
        return sums, n

    def resize_crop(self, src: torch.Tensor, new_h, new_w, crop_top, crop_left, H, W, divisor=255.0):
        """src (H0,W0) uint8 or fp32 CUDA -> (H,W) fp32: bilinear resize + centre crop + /divisor (loader pre-processing)."""
        src = _dense(src)
        if not (src.is_cuda and src.dim() == 2 and src.dtype in (torch.uint8, torch.float32)):
            raise NativeError("resize_crop: src must be a 2-D uint8/float32 CUDA tensor")
        out = torch.empty((H, W), dtype=torch.float32, device=src.device)
        self._call("spn_resize_crop", self.handle, _ptr(src), int(src.dtype == torch.uint8), src.shape[0], src.shape[1], int(new_h),
                   int(new_w), int(crop_top), int(crop_left), int(H), int(W), C.c_float(divisor), _ptr(out), self._s())
        return out

    def jpeg_decode_gray(self, plan, data, n, coef, out, status):
        """Enqueue spn_jpeg_decode_gray on the current stream: plan (uint8), data (uint8 file bytes), coef (int16 scratch of
        at least the plan's coef_bytes), out (uint8 planes of at least out_bytes), status (int32, n) - all CUDA tensors
        of this context's device.  Images whose status ends up non-zero must be decoded on the host."""
        for t, dt, name in ((plan, torch.uint8, "plan"), (data, torch.uint8, "data"), (coef, torch.int16, "coef"),
                            (out, torch.uint8, "out"), (status, torch.int32, "status")):
            _chk_dev(t, dt, name, self.device)
        if status.numel() < n:
            raise NativeError(f"status holds {status.numel()} entries, {n} needed")
        self._call("spn_jpeg_decode_gray", self.handle, _ptr(plan), _ptr(data), int(n), _ptr(coef), C.c_int64(coef.numel() * 2),
                   _ptr(out), _ptr(status), self._s())

    def invert3x3(self, m):
        m = _dense(m)
        _chk_dev(m, torch.float32, "m", self.device)
        out = torch.empty_like(m)
        self._call("spn_invert3x3", self.handle, _ptr(m), m.numel() // 9, _ptr(out), self._s())
        return out


_contexts: dict[int, Context] = {}


def get_context(device=None) -> Context:
    """Process-wide context per GPU (weights are per-model: models create their own Context)."""
    if not torch.cuda.is_available():
        raise NativeError("CUDA is not available: superpoint-nerf-pytorch_b200 has no CPU fallback")
    idx = None if device is None else torch.device(device).index
    if idx is None:                      # 'cuda' without an index means torch's CURRENT device, not GPU 0
        idx = torch.cuda.current_device()
    if idx not in _contexts:
        _contexts[idx] = Context(idx)
    return _contexts[idx]
