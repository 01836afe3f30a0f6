"""Seeded JPEG files for the decoder tests: cv2 / Pillow encodes and a small baseline writer for streams no encoder
produces (coefficients chosen directly, fill bytes, 16-bit quantisation tables, odd sampling declarations)."""
import io

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7,
                   14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39,
                   46, 53, 60, 61, 54, 47, 55, 62, 63])            # zigzag index -> natural index


def _lengths_to_table(symbols, lengths):
    """Canonical Huffman table (JPEG DHT order) -> (bits[1..16], values, {symbol: (code, length)})."""
    order = sorted(range(len(symbols)), key=lambda i: (lengths[i], i))
    bits = [0] * 17
    codes, code, prev = {}, 0, None
    for i in order:
        l = lengths[i]
        if prev is not None:
            code = (code + 1) << (l - prev)
        codes[symbols[i]] = (code, l)
        bits[l] += 1
        prev = l
    return bits[1:], [symbols[i] for i in order], codes


def _tables():
    dc_syms = list(range(16))
    dc_len = [3] * 6 + [5] * 7 + [7] * 3                  # Kraft sum < 1: no all-ones code
    ac_syms = [0x00, 0x01, 0x02, 0x11, 0x03, 0x21, 0x04, 0x12, 0x31, 0x05, 0xF0]
    ac_syms += [(r << 4) | s for r in range(16) for s in range(1, 11) if (r << 4) | s not in ac_syms]
    ac_len = [2] * 2 + [4] * 4 + [6] * 8 + [8] * 16 + [10] * 32
    ac_len += [12] * (len(ac_syms) - len(ac_len) - 2) + [16, 16]     # codes longer than 9 bits exercise the slow path
    return _lengths_to_table(dc_syms, dc_len), _lengths_to_table(ac_syms, ac_len)


(DC_BITS, DC_VALS, DC_CODES), (AC_BITS, AC_VALS, AC_CODES) = _tables()


class _Bits:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, v, l):
        for k in range(l - 1, -1, -1):
            self.acc = (self.acc << 1) | ((v >> k) & 1)
            self.n += 1
            if self.n == 8:
                self.out.append(self.acc)
                if self.acc == 0xFF:
                    self.out.append(0)
                self.acc, self.n = 0, 0

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def _category(v):
    return 0 if v == 0 else int(abs(int(v))).bit_length()


def _put_value(bw, v, s):
    if s:
        bw.put(v if v >= 0 else v + (1 << s) - 1, s)


def _encode_block(bw, blk, pred):
    """blk: 64 ints in natural order; returns the new DC predictor."""
    zz = [int(blk[ZIGZAG[k]]) for k in range(64)]
    diff = zz[0] - pred
    s = _category(diff)
    bw.put(*DC_CODES[s])
    _put_value(bw, diff, s)
    run = 0
    for k in range(1, 64):
        v = zz[k]
        if v == 0:
            run += 1
            continue
        while run > 15:
            bw.put(*AC_CODES[0xF0])
            run -= 16
        s = _category(v)
        assert s <= 10, "AC values are limited to +-1023"
        bw.put(*AC_CODES[(run << 4) | s])
        _put_value(bw, v, s)
        run = 0
    if run:
        bw.put(*AC_CODES[0x00])
    return zz[0]


def _segment(marker, payload):
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)


def write_baseline(luma, height, width, quant, sampling=(1, 1), ncomp=1, restart=0, fill_bytes=0, sof=0xC0, q16=False,
                   chroma_seed=None, jfif=True):
    """Baseline (or SOF1) Huffman JPEG from luma blocks.

    luma: int array (blocks_y, blocks_x, 64) in natural order covering the MCU-padded luma plane; quant: 64 ints in
    natural order (luma table; chroma uses the same); sampling: luma (h, v) for ncomp == 3 (chroma 1x1), or the factors a
    1-component frame declares; restart: MCUs per interval; fill_bytes: extra 0xFF bytes before every marker inside and
    after the entropy data; q16: write the table with 16-bit entries; chroma_seed: random chroma coefficients."""
    h, v = sampling
    out = bytearray(b"\xff\xd8")
    if jfif:
        out += _segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    qz = [int(quant[ZIGZAG[k]]) for k in range(64)]
    out += _segment(0xDB, bytes([0x10 if q16 else 0x00]) + (b"".join(x.to_bytes(2, "big") for x in qz) if q16 else bytes(qz)))
    comps = [(1, h, v)] + [(2 + c, 1, 1) for c in range(ncomp - 1)]
    out += _segment(sof, bytes([8]) + height.to_bytes(2, "big") + width.to_bytes(2, "big") + bytes([ncomp]) +
                    b"".join(bytes([cid, (ch << 4) | cv, 0]) for cid, ch, cv in comps))
    for tc, tid, bits, vals in ((0, 0, DC_BITS, DC_VALS), (1, 0, AC_BITS, AC_VALS), (0, 1, DC_BITS, DC_VALS), (1, 1, AC_BITS, AC_VALS)):
        out += _segment(0xC4, bytes([(tc << 4) | tid]) + bytes(bits) + bytes(vals))
    if restart:
        out += _segment(0xDD, restart.to_bytes(2, "big"))
    out += _segment(0xDA, bytes([ncomp]) + b"".join(bytes([cid, 0x00 if cid == 1 else 0x11]) for cid, _, _ in comps) + bytes([0, 63, 0]))
    bw = _Bits()
    rng = np.random.RandomState(chroma_seed) if chroma_seed is not None else None
    if ncomp == 1:
        mcus_y, mcus_x, mh, mv = (height + 7) // 8, (width + 7) // 8, 1, 1
    else:
        mcus_y, mcus_x, mh, mv = -(-height // (8 * v)), -(-width // (8 * h)), h, v
    assert luma.shape[:2] == (mcus_y * mv, mcus_x * mh), (luma.shape, mcus_y * mv, mcus_x * mh)
    preds = [0] * ncomp
    n_mcu = mcus_x * mcus_y
    for m in range(n_mcu):
        if restart and m and m % restart == 0:
            bw.flush()
            bw.out += b"\xff" * fill_bytes + bytes([0xFF, 0xD0 + (m // restart - 1) % 8])
            preds = [0] * ncomp
        my, mx = divmod(m, mcus_x)
        for by in range(mv):
            for bx in range(mh):
                preds[0] = _encode_block(bw, luma[my * mv + by, mx * mh + bx], preds[0])
        for c in range(1, ncomp):
            blk = np.zeros(64, np.int64)
            if rng is not None:
                blk[0] = rng.randint(-200, 200)
                blk[1:6] = rng.randint(-20, 20, 5)
            preds[c] = _encode_block(bw, blk, preds[c])
    bw.flush()
    out += bw.out + b"\xff" * fill_bytes + b"\xff\xd9"
    return bytes(out)


def blocks_for(height, width, sampling=(1, 1), ncomp=1):
    """Shape (blocks_y, blocks_x) of the luma array write_baseline expects."""
    h, v = sampling
    if ncomp == 1:
        return (height + 7) // 8, (width + 7) // 8
    return -(-height // (8 * v)) * v, -(-width // (8 * h)) * h


def make_image(kind, height, width, seed, channels=3):
    """'flat', 'smooth' or 'noise' uint8 image (H, W, channels)."""
    rng = np.random.RandomState(seed)
    if kind == "flat":
        img = np.full((height, width, channels), rng.randint(0, 256), np.uint8)
    elif kind == "noise":
        img = rng.randint(0, 256, (height, width, channels)).astype(np.uint8)
    else:
        y, x = np.mgrid[0:height, 0:width].astype(np.float64)
        base = 128 + 90 * np.sin(x / (7 + 13 * rng.rand())) * np.cos(y / (5 + 11 * rng.rand()))
        img = np.stack([np.clip(base + 25 * c, 0, 255) for c in range(channels)], -1).astype(np.uint8)
    return img


SAMPLINGS = {"411": "IMWRITE_JPEG_SAMPLING_FACTOR_411", "420": "IMWRITE_JPEG_SAMPLING_FACTOR_420",
             "422": "IMWRITE_JPEG_SAMPLING_FACTOR_422", "440": "IMWRITE_JPEG_SAMPLING_FACTOR_440",
             "444": "IMWRITE_JPEG_SAMPLING_FACTOR_444"}


def cv2_jpeg(img, quality=90, sampling="420", restart=0, optimize=False, progressive=False):
    import cv2
    params = [cv2.IMWRITE_JPEG_QUALITY, int(quality), cv2.IMWRITE_JPEG_RST_INTERVAL, int(restart),
              cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize), cv2.IMWRITE_JPEG_PROGRESSIVE, int(progressive)]
    if img.ndim == 3 and img.shape[2] == 3:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, getattr(cv2, SAMPLINGS[sampling])]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return buf.tobytes()


def pil_jpeg(img, mode, quality=90):
    """Pillow encode in `mode` ('CMYK', 'RGB' stored as RGB components, ...)."""
    from PIL import Image
    im = Image.fromarray(img[..., :3] if img.ndim == 3 else img)
    b = io.BytesIO()
    if mode == "CMYK":
        im.convert("CMYK").save(b, "JPEG", quality=quality)
    elif mode == "RGB":
        im.save(b, "JPEG", quality=quality, keep_rgb=True)
    else:
        im.convert(mode).save(b, "JPEG", quality=quality)
    return b.getvalue()


def host_gray(data):
    """The host decoder the device must match: torchvision decode_image(..., GRAY) -> (H, W) uint8 numpy."""
    import torch
    import torchvision
    t = torch.frombuffer(bytearray(data), dtype=torch.uint8)
    return torchvision.io.decode_image(t, torchvision.io.ImageReadMode.GRAY)[0].numpy()


def crafted_streams():
    """{name: (jpeg bytes, expected plan status)} for the corner cases no encoder produces."""
    rng = np.random.RandomState(7)
    q8 = np.clip(rng.randint(1, 40, 64), 1, 255)
    out = {}
    # IDCT outputs far outside +-384 (both signs), in 16-bit range and beyond it, incl. DC-only blocks (the SIMD shortcut)
    by, bx = blocks_for(24, 40)
    blk = rng.randint(-1023, 1024, (by, bx, 64))
    blk[0, 0, 1:] = 0
    blk[0, 0, 0] = 1000
    blk[0, 1, 1:] = 0
    blk[0, 1, 0] = -1000
    blk[1, 0, 8:] = 0
    out["idct_range"] = (write_baseline(blk, 24, 40, np.full(64, 60)), 0)
    big = np.zeros((by, bx, 64), np.int64)
    big[..., 0] = rng.randint(-900, 900, (by, bx))
    big[..., 1:4] = rng.randint(-300, 300, (by, bx, 3))
    out["idct_saturate_16bit_dq"] = (write_baseline(big, 24, 40, np.full(64, 255)), 0)
    # DC predictor far beyond int16: +2047 per block
    by, bx = blocks_for(8, 8 * 40)
    dcs = np.zeros((by, bx, 64), np.int64)
    dcs[0, :, 0] = np.cumsum(np.full(bx, 2047))
    out["dc_beyond_int16"] = (write_baseline(dcs, 8, 8 * 40, np.full(64, 3)), 0)
    # SOF1 with a 16-bit DQT
    by, bx = blocks_for(20, 30)
    q16 = rng.randint(1, 3000, 64)
    b = rng.randint(-3, 4, (by, bx, 64))
    out["sof1_q16"] = (write_baseline(b, 20, 30, q16, sof=0xC1, q16=True), 0)
    # 1-component frame that declares 2x2 sampling (decoded non-interleaved, block = MCU)
    by, bx = blocks_for(27, 35)
    b = rng.randint(-20, 21, (by, bx, 64))
    out["gray_2x2"] = (write_baseline(b, 27, 35, q8, sampling=(2, 2)), 0)
    # fill bytes before the RST and EOI markers, 3-component interleaved 2x1 luma
    by, bx = blocks_for(33, 50, (2, 1), 3)
    b = rng.randint(-30, 31, (by, bx, 64))
    out["fill_bytes_rst"] = (write_baseline(b, 33, 50, q8, sampling=(2, 1), ncomp=3, restart=2, fill_bytes=3, chroma_seed=1), 0)
    # 3x3 luma with chroma: 11 blocks per MCU, libjpeg rejects it
    by, bx = blocks_for(30, 30, (3, 3), 3)
    b = np.zeros((by, bx, 64), np.int64)
    out["mcu_too_large"] = (write_baseline(b, 30, 30, q8, sampling=(3, 3), ncomp=3), 2)
    # 16-bit DQT entries above 32767
    by, bx = blocks_for(8, 8)
    out["q16_too_large"] = (write_baseline(np.zeros((by, bx, 64), np.int64), 8, 8, np.full(64, 40000), q16=True), 1)
    return out
