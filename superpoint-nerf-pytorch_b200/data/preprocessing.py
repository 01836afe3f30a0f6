"""Loader pre-processing that feeds the hot path (SURVEY.md section 8f-1), mirroring the reference's dataset methods:

    ratio_preserving_resize      <- data/COCO.py:66-76, data/HPatches.py:64-72 (+ the "/= 255." of COCO.py:135)
    adapt_homography_to_resize   <- data/HPatches.py:74-100

Image decoding runs with torchvision on the host (as in the reference), or, with ``data.decode: device``, for a batch
of baseline JPEG files on the GPU (``launch_jpeg_decode`` / ``finish_jpeg_decode``, bit-identical to the host decode); everything after
the decode is one kernel (spn_resize_crop) that takes the decoded uint8 image, so the host->device copy is 1
byte/pixel (or the compressed file).
"""
import numpy as np
import torch

from .._native import get_context, jpeg_plan


def resize_geometry(src_shape, target):
    """(new_h, new_w, crop_top, crop_left) exactly as the reference computes them: fp32 scale arithmetic truncated to
    int32 (COCO.py:70-73), torchvision centre-crop offsets int(round((size - crop) / 2))."""
    target_t = torch.as_tensor(list(target), dtype=torch.int32)
    shape_f = torch.as_tensor(list(src_shape), dtype=torch.float32)
    scales = torch.divide(target_t, shape_f)
    new = (shape_f * torch.max(scales)).to(torch.int32)
    nh, nw = int(new[0]), int(new[1])
    H, W = int(target[0]), int(target[1])
    # torchvision.transforms.functional.center_crop pads a too-small image symmetrically ((c - s) // 2 first) then crops
    pad_top = (H - nh) // 2 if nh < H else 0
    pad_left = (W - nw) // 2 if nw < W else 0
    ph, pw = max(nh, H), max(nw, W)
    top = int(round((ph - H) / 2.0)) - pad_top
    left = int(round((pw - W) / 2.0)) - pad_left
    return nh, nw, top, left


_upload_streams = {}


def pin_host(image, device=None):
    """Decoded host image -> page-locked copy (torch's caching pinned allocator; called on the decode threads) so that the
    upload is a real asynchronous DMA instead of a staged copy the issuing thread has to wait for.  ``device``: the GPU
    the loader feeds - a new thread's current device is 0, and pinning there would create a context on GPU 0 in every
    rank of a multi-GPU export."""
    if not torch.cuda.is_available() or image.is_cuda:
        return image
    try:
        dev = torch.device(device) if device is not None else torch.device("cuda")
        with torch.cuda.device(dev if dev.index is not None else torch.cuda.current_device()):
            return image.pin_memory()
    except RuntimeError:
        return image


def _upload_stream(device):
    """One side stream per GPU for the loader's uploads."""
    key = torch.device(device).index
    if key not in _upload_streams:
        _upload_streams[key] = torch.cuda.Stream(device=device)
    return _upload_streams[key]


def ratio_preserving_resize(image, target, normalize=True, device=None):
    """image (H0,W0) uint8 or fp32 (CUDA, or CPU - it is uploaded) -> (H,W) fp32 CUDA, /255 when ``normalize``.

    A host image is uploaded and resized on a side stream: a copy from pageable memory blocks the calling thread until
    the stream it was issued on reaches it, and on the consumer's stream that is after every kernel of the export group
    already in flight (the loader then runs in lock step with the GPU instead of ahead of it).  The consumer's stream
    only waits for the side stream's event.  Pinned host images (the datasets pin them on their decode threads) make
    the upload truly asynchronous."""
    if image.dim() == 3 and image.shape[0] == 1:
        image = image[0]
    nh, nw, top, left = resize_geometry(image.shape, target)
    scale = 255.0 if normalize else 1.0
    if image.is_cuda:
        return get_context(image.device).resize_crop(image, nh, nw, top, left, int(target[0]), int(target[1]), scale)
    dev = torch.device(device) if device is not None else torch.device("cuda")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    cur, side = torch.cuda.current_stream(dev), _upload_stream(dev)
    with torch.cuda.stream(side):
        image = image.to(dev, non_blocking=True)
        out = get_context(dev).resize_crop(image, nh, nw, top, left, int(target[0]), int(target[1]), scale)
    out.record_stream(cur)
    cur.wait_stream(side)
    return out


def _resolve(device):
    dev = torch.device(device) if device is not None else torch.device("cuda")
    return torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev


_decode_streams = {}


def launch_jpeg_decode(files, device=None):
    """Start the device decode of JPEG files (uint8 numpy arrays of the file bytes) -> handle for finish_jpeg_decode.

    One plan (host header parse), one pinned upload of the concatenated files, one spn_jpeg_decode_gray and one status
    read-back on a decode stream of its own, so a decode in flight never delays the resizes the loader's side stream
    runs for the consumer.  Nothing here waits for the GPU."""
    dev = _resolve(device)
    offsets = np.zeros(len(files) + 1, np.int64)
    np.cumsum([len(f) for f in files], out=offsets[1:])
    host = torch.empty(int(offsets[-1]), dtype=torch.uint8, pin_memory=True)
    np.concatenate(files, out=host.numpy())
    plan, info, coef_bytes, out_bytes = jpeg_plan(host.numpy(), offsets)
    n = len(files)
    ctx = get_context(dev)
    if dev.index not in _decode_streams:
        _decode_streams[dev.index] = torch.cuda.Stream(device=dev)
    stream = _decode_streams[dev.index]
    with torch.cuda.stream(stream):
        d_data = host.to(dev, non_blocking=True)
        d_plan = torch.from_numpy(plan).pin_memory().to(dev, non_blocking=True)
        coef = torch.empty(coef_bytes // 2, dtype=torch.int16, device=dev)
        planes = torch.empty(max(out_bytes, 1), dtype=torch.uint8, device=dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        ctx.jpeg_decode_gray(d_plan, d_data, n, coef, planes, status)
        status_host = torch.empty(n, dtype=torch.int32, pin_memory=True)
        status_host.copy_(status, non_blocking=True)
        done = torch.cuda.Event()
        done.record(stream)
    return {"dev": dev, "ctx": ctx, "info": info, "planes": planes, "status": status_host, "done": done, "stream": stream}


def finish_jpeg_decode(handle, target, normalize=True):
    """-> list of (H,W) fp32 CUDA images (ratio_preserving_resize of the grayscale decode), None where the device decoder
    did not decode the file (the caller decodes it on the host).  Waits for the decode's event only (never for the
    consumer's stream); the resizes run on the loader's side stream after that event, and the consumer's stream waits
    for the side stream."""
    dev, ctx, info, planes = handle["dev"], handle["ctx"], handle["info"], handle["planes"]
    handle["done"].synchronize()
    status = handle["status"].numpy()
    cur, side = torch.cuda.current_stream(dev), _upload_stream(dev)
    side.wait_event(handle["done"])
    planes.record_stream(side)
    scale = 255.0 if normalize else 1.0
    out = []
    with torch.cuda.stream(side):
        for i in range(len(status)):
            if status[i] != 0:
                out.append(None)
                continue
            h, w, off = int(info[i, 1]), int(info[i, 2]), int(info[i, 4])
            nh, nw, top, left = resize_geometry((h, w), target)
            img = ctx.resize_crop(planes[off:off + h * w].view(h, w), nh, nw, top, left, int(target[0]), int(target[1]), scale)
            img.record_stream(cur)
            out.append(img)
    cur.wait_stream(side)
    return out


def adapt_homography_to_resize(homography, image_shape, warped_image_shape, target):
    """HPatches ground-truth homography expressed between the resized + centre-cropped images (HPatches.py:74-100).
    3x3 host arithmetic in fp32, in the reference's operation order."""
    source_size = torch.as_tensor(image_shape, dtype=torch.float32)
    source_warped_size = torch.as_tensor(warped_image_shape, dtype=torch.float32)
    target_size = torch.as_tensor(list(target), dtype=torch.float32)
    s = torch.max(torch.divide(target_size, source_size))
    up_scale = torch.diag(torch.stack([1.0 / s, 1.0 / s, torch.tensor(1.0)]))
    warped_s = torch.max(torch.divide(target_size, source_warped_size))
    down_scale = torch.diag(torch.stack([warped_s, warped_s, torch.tensor(1.0)]))

    def shift(size, scale, sign):
        t = torch.eye(3, dtype=torch.float32)
        t[0, -1] = sign * ((size[1] * scale - target_size[1]) / torch.tensor(2.0)).to(torch.int32)
        t[1, -1] = sign * ((size[0] * scale - target_size[0]) / torch.tensor(2.0)).to(torch.int32)
        return t

    return shift(source_warped_size, warped_s, -1.0) @ down_scale @ torch.as_tensor(homography, dtype=torch.float32) @ up_scale \
        @ shift(source_size, s, 1.0)
