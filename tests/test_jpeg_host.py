"""spn_jpeg_plan (host header parser of the device JPEG decoder, include/spn_jpeg.h): per-image status and geometry for
every supported and unsupported kind of file, robustness against malformed headers, and the error convention of the
new entry points.  No GPU needed."""
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
import jpeg_streams as J

OK, UNSUPPORTED, MALFORMED = 0, 1, 2


def plan(files):
    from superpoint_nerf_pytorch_b200 import _native as N
    offsets = np.zeros(len(files) + 1, np.int64)
    np.cumsum([len(f) for f in files], out=offsets[1:])
    data = np.frombuffer(b"".join(files), np.uint8) if sum(map(len, files)) else np.zeros(0, np.uint8)
    return N.jpeg_plan(data, offsets)


def blocks(h, w, mh=1, mv=1):
    return -(-h // (8 * mv)) * mv * (-(-w // (8 * mh)) * mh)


KINDS = {   # name -> (file, status, (h, w), luma blocks)
    "420": (J.cv2_jpeg(J.make_image("noise", 37, 51, 1), 90, "420"), OK, (37, 51), blocks(37, 51, 2, 2)),
    "422": (J.cv2_jpeg(J.make_image("noise", 37, 51, 1), 90, "422"), OK, (37, 51), blocks(37, 51, 2, 1)),
    "440": (J.cv2_jpeg(J.make_image("noise", 37, 51, 1), 90, "440"), OK, (37, 51), blocks(37, 51, 1, 2)),
    "444": (J.cv2_jpeg(J.make_image("noise", 37, 51, 1), 90, "444"), OK, (37, 51), blocks(37, 51)),
    "411": (J.cv2_jpeg(J.make_image("noise", 37, 51, 1), 90, "411"), OK, (37, 51), blocks(37, 51, 4, 1)),
    "gray": (J.cv2_jpeg(J.make_image("smooth", 9, 17, 1, 1)[..., 0], 90), OK, (9, 17), blocks(9, 17)),
    "restart": (J.cv2_jpeg(J.make_image("smooth", 64, 64, 1), 90, "420", restart=3), OK, (64, 64), blocks(64, 64, 2, 2)),
    "optimized": (J.cv2_jpeg(J.make_image("smooth", 16, 24, 1), 90, "420", optimize=True), OK, (16, 24), blocks(16, 24, 2, 2)),
    "progressive": (J.cv2_jpeg(J.make_image("noise", 20, 20, 1), 90, progressive=True), UNSUPPORTED, (20, 20), 0),
    "cmyk": (J.pil_jpeg(J.make_image("noise", 20, 20, 1), "CMYK"), UNSUPPORTED, (20, 20), 0),
    "rgb": (J.pil_jpeg(J.make_image("noise", 20, 20, 1), "RGB"), UNSUPPORTED, (20, 20), 0),
}


@pytest.mark.parametrize("name", sorted(KINDS))
def test_plan_reports_status_and_geometry(name):
    f, status, hw, nblk = KINDS[name]
    _, info, coef_bytes, out_bytes = plan([f])
    assert int(info[0, 0]) == status
    assert tuple(int(x) for x in info[0, 1:3]) == hw
    assert int(info[0, 3]) == nblk
    assert (coef_bytes, out_bytes) == ((nblk * 128, hw[0] * hw[1]) if status == OK else (0, 0))
    assert int(info[0, 4]) == (0 if status == OK else -1)


def test_plan_crafted_streams():
    for name, (f, status) in J.crafted_streams().items():
        assert int(plan([f])[1][0, 0]) == status, name


@pytest.mark.parametrize("cut", [1, 2])
@pytest.mark.parametrize("kind", ["420", "gray"])
def test_plan_sends_files_without_eoi_to_the_host(kind, cut):
    """A file cut in or before its EOI: torchvision raises on it, so the device must not decode it either."""
    f = KINDS[kind][0][:-cut]
    assert int(plan([f])[1][0, 0]) == UNSUPPORTED
    with pytest.raises(RuntimeError):
        J.host_gray(f)


def test_prefetch_stage_yields_items_before_a_failure_in_order():
    """The batched stage yields the same items in the same order as the per-item path, and the items before a failing
    one (in a worker or in the stage) before the exception."""
    from superpoint_nerf_pytorch_b200.utils.data_loaders import PrefetchLoader

    class Items:
        def __init__(self, bad_decode=None, bad_finish=None):
            self.bad_decode, self.bad_finish = bad_decode, bad_finish

        def __len__(self):
            return 41

        def decode(self, i):
            if i == self.bad_decode:
                raise ValueError(i)
            return i

        def finish(self, i):
            if i == self.bad_finish:
                raise KeyError(i)
            return i

        def batch_collator(self, b):
            return b

    class Batched(Items):
        def finish_batch(self, items):
            return (self.finish(i) for i in items)

    def run(ds):
        out = []
        try:
            for b in PrefetchLoader(ds, batch_size=1, workers=3, device_batch=6, rank=1, world=2):
                out += b
        except Exception as e:  # noqa: BLE001
            out.append(type(e).__name__)
        return out

    for kw in ({}, {"bad_decode": 23}, {"bad_finish": 17}):
        want = run(Items(**kw))
        assert run(Batched(**kw)) == want, kw
    assert run(Items(bad_finish=17)) == list(range(1, 17, 2)) + ["KeyError"]


def test_plan_packs_output_planes_in_order():
    files = [KINDS["420"][0], KINDS["progressive"][0], KINDS["gray"][0], b"not a jpeg", KINDS["444"][0]]
    _, info, coef_bytes, out_bytes = plan(files)
    assert list(info[:, 0]) == [OK, UNSUPPORTED, OK, MALFORMED, OK]
    assert list(info[:, 4]) == [0, -1, 37 * 51, -1, 37 * 51 + 9 * 17]
    assert out_bytes == 2 * 37 * 51 + 9 * 17
    assert coef_bytes == 128 * (blocks(37, 51, 2, 2) + blocks(9, 17) + blocks(37, 51))


def test_plan_survives_malformed_headers():
    """Truncations at every header byte, zero dimensions, over-subscribed Huffman tables, lengths past the end and random
    header corruption: an error status, never a crash or a read out of bounds.  Runs in a child process."""
    code = r'''
import sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np
import jpeg_streams as J
from superpoint_nerf_pytorch_b200 import _native as N
good = J.cv2_jpeg(J.make_image("smooth", 24, 32, 1), 90, "420", restart=2)
sos = good.index(b"\xff\xda")
cases = [good[:k] for k in range(0, sos + 14)]
def patched(marker, off, val):
    b = bytearray(good); p = b.index(marker) + off; b[p] = val; return bytes(b)
sof = good.index(b"\xff\xc0")
zero_h = bytearray(good); zero_h[sof + 5:sof + 7] = b"\x00\x00"; cases.append(bytes(zero_h))
zero_w = bytearray(good); zero_w[sof + 7:sof + 9] = b"\x00\x00"; cases.append(bytes(zero_w))
dht = good.index(b"\xff\xc4")
over = bytearray(good); over[dht + 5:dht + 21] = bytes([2, 2, 2, 2] + [0] * 12); cases.append(bytes(over))
longseg = bytearray(good); longseg[dht + 2:dht + 4] = b"\xff\xf0"; cases.append(bytes(longseg))
rng = np.random.RandomState(0)
for _ in range(400):
    b = bytearray(good)
    for p in rng.randint(2, sos + 14, rng.randint(1, 4)):
        b[p] = rng.randint(0, 256)
    cases.append(bytes(b))
statuses = []
for c in cases:
    data = np.frombuffer(c, np.uint8) if c else np.zeros(0, np.uint8)
    # each file alone, at the very end of an exactly sized buffer
    _, info, _, _ = N.jpeg_plan(np.ascontiguousarray(data), np.array([0, len(c)], np.int64))
    statuses.append(int(info[0, 0]))
assert all(s != 0 for s in statuses[:sos + 14]), statuses[:sos + 14]
assert all(s == 2 for s in statuses[sos + 14:sos + 18]), statuses[sos + 14:sos + 18]
print("planned", len(cases))
''' % (str(ROOT), str(ROOT / "tests"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "planned" in out.stdout


def test_jpeg_entry_points_reject_null_arguments():
    """Every symbol of include/spn_jpeg.h called with NULL and zero arguments returns a negative code and sets a message
    (child process, like the spn_b200.h check)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
n = 0
for name, (res, args) in N.JPEG_PROTOTYPES.items():
    vals = [None if a in (C.c_void_p, C.c_char_p) else a(0) for a in args]
    rc = getattr(lib, name)(*vals)
    msg = lib.spn_last_error().decode()
    assert rc < 0 and msg, (name, rc, msg)
    n += 1
print("checked", n)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "checked 2" in out.stdout


def test_header_declares_exactly_the_jpeg_prototypes():
    import re
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_jpeg.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.JPEG_PROTOTYPES)
    assert not set(N.JPEG_PROTOTYPES) & set(N.PROTOTYPES)
