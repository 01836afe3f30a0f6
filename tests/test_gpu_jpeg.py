"""Device JPEG decoder (spn_jpeg_decode_gray) against the host decoder (torchvision decode_image GRAY), bit for bit, and
the loader / export with ``data.decode: device`` against ``host``."""
import copy
import shutil
from pathlib import Path

import numpy as np
import pytest
import torch

import jpeg_streams as J

pytestmark = pytest.mark.gpu

GUARD = 4096


def device_decode(files):
    """-> (list of (H,W) uint8 numpy or None, statuses); paints guard bands around d_out and d_coef and checks them."""
    from superpoint_nerf_pytorch_b200 import _native as N
    offsets = np.zeros(len(files) + 1, np.int64)
    np.cumsum([len(f) for f in files], out=offsets[1:])
    data = np.frombuffer(b"".join(files), np.uint8).copy()
    plan, info, coef_bytes, out_bytes = N.jpeg_plan(data, offsets)
    ctx = N.get_context("cuda:0")
    dev = torch.device("cuda", 0)
    coef_full = torch.full((coef_bytes // 2 + 2 * GUARD,), 0x5A5A, dtype=torch.int16, device=dev)
    out_full = torch.full((out_bytes + 2 * GUARD,), 0xA5, dtype=torch.uint8, device=dev)
    coef, out = coef_full[GUARD:GUARD + coef_bytes // 2], out_full[GUARD:GUARD + out_bytes]
    status = torch.full((len(files),), -7, dtype=torch.int32, device=dev)
    ctx.jpeg_decode_gray(torch.from_numpy(plan).to(dev), torch.from_numpy(data).to(dev), len(files), coef, out, status)
    torch.cuda.synchronize()
    for band in (coef_full[:GUARD], coef_full[GUARD + coef_bytes // 2:]):
        assert bool((band == 0x5A5A).all()), "d_coef guard band overwritten"
    for band in (out_full[:GUARD], out_full[GUARD + out_bytes:]):
        assert bool((band == 0xA5).all()), "d_out guard band overwritten"
    st = status.cpu().numpy()
    o = out.cpu().numpy()
    imgs = []
    for i in range(len(files)):
        s, h, w, _, off = (int(x) for x in info[i])
        imgs.append(o[off:off + h * w].reshape(h, w) if st[i] == 0 else None)
    return imgs, st


def assert_exact(files, names):
    imgs, st = device_decode(files)
    for f, name, img, s in zip(files, names, imgs, st):
        assert s == 0, (name, s)
        ref = J.host_gray(f)
        assert img.shape == ref.shape and np.array_equal(img, ref), (name, int(np.abs(img.astype(int) - ref).max()))


@pytest.mark.parametrize("kind", ["flat", "smooth", "noise"])
def test_subsamplings(kind):
    files = [J.cv2_jpeg(J.make_image(kind, 121, 163, 5), 90, s) for s in J.SAMPLINGS]
    assert_exact(files, list(J.SAMPLINGS))


def test_qualities_and_optimized_tables():
    files, names = [], []
    for q in (5, 10, 25, 50, 75, 90, 95, 100):
        for opt in (False, True):
            files.append(J.cv2_jpeg(J.make_image("noise", 96, 128, q), q, "420", optimize=opt))
            names.append(f"q{q} opt{opt}")
    assert_exact(files, names)


@pytest.mark.parametrize("rst", [1, 7])
def test_restart_intervals(rst):
    files = [J.cv2_jpeg(J.make_image("smooth", 100, 140, 3), 85, s, restart=rst) for s in ("420", "444")]
    files.append(J.cv2_jpeg(J.make_image("noise", 100, 140, 3)[..., 0], 85, restart=rst))
    assert_exact(files, ["420", "444", "gray"])


@pytest.mark.parametrize("hw", [(1, 1), (7, 9), (17, 33), (1, 2000), (481, 643), (640, 480), (1080, 1920)])
def test_sizes(hw):
    h, w = hw
    files = [J.cv2_jpeg(J.make_image("noise", h, w, 11), 90, "420"), J.cv2_jpeg(J.make_image("smooth", h, w, 12, 1)[..., 0], 90)]
    assert_exact(files, ["420", "gray"])


def test_crafted_streams():
    streams = {k: f for k, (f, st) in J.crafted_streams().items() if st == 0}
    assert_exact(list(streams.values()), list(streams))


def test_mixed_batch_in_one_launch():
    rng = np.random.RandomState(3)
    files, names, unsupported = [], [], set()
    for i in range(64):
        h, w = int(rng.randint(1, 700)), int(rng.randint(1, 700))
        kind = ("flat", "smooth", "noise")[i % 3]
        if i % 16 == 5:
            files.append(J.cv2_jpeg(J.make_image(kind, h, w, i), 80, progressive=True))
            unsupported.add(i)
        elif i % 4 == 3:
            files.append(J.cv2_jpeg(J.make_image(kind, h, w, i, 1)[..., 0], int(rng.randint(5, 101)), restart=int(rng.randint(0, 9))))
        else:
            files.append(J.cv2_jpeg(J.make_image(kind, h, w, i), int(rng.randint(5, 101)), list(J.SAMPLINGS)[i % 5],
                                    restart=int(rng.randint(0, 9)), optimize=bool(i % 2)))
        names.append(f"#{i} {h}x{w}")
    imgs, st = device_decode(files)
    for i, (f, img, s) in enumerate(zip(files, imgs, st)):
        if i in unsupported:
            assert s == 1, names[i]
            continue
        assert s == 0, (names[i], s)
        assert np.array_equal(img, J.host_gray(f)), names[i]


def test_corrupt_entropy_data_never_differs_silently():
    """Truncated or bit-flipped entropy data: the host's pixels or a non-zero status, never a fault (guard bands are
    checked by device_decode)."""
    rng = np.random.RandomState(9)
    good = [J.cv2_jpeg(J.make_image("noise", 64, 80, 1), 90, "420", restart=r) for r in (0, 3)]
    files = []
    for g in good:
        sos = g.index(b"\xff\xda") + 14
        for cut in rng.randint(sos, len(g), 12):
            files.append(g[:cut])
        for _ in range(24):
            b = bytearray(g)
            for p in rng.randint(sos, len(g) - 2, rng.randint(1, 6)):
                b[p] ^= 1 << rng.randint(0, 8)
            files.append(bytes(b))
    imgs, st = device_decode(files)
    n_err = 0
    for f, img, s in zip(files, imgs, st):
        if s != 0:
            n_err += 1
            continue
        assert np.array_equal(img, J.host_gray(f))
    assert n_err > 0


# ---- loader and export -------------------------------------------------------------------------------------------------

def _write_dir(root):
    d = root / "data" / "COCO" / "images" / "training"
    d.mkdir(parents=True)
    rng = np.random.RandomState(0)
    for i in range(22):
        h, w = int(rng.randint(120, 500)), int(rng.randint(120, 500))
        img = J.make_image(("smooth", "noise", "flat")[i % 3], h, w, i)
        if i == 4:
            data = J.cv2_jpeg(img, 85, progressive=True)
        elif i == 9:
            data = J.pil_jpeg(img, "CMYK")
        elif i == 13:
            data = J.cv2_jpeg(img[..., 0], 70, restart=5)
        else:
            data = J.cv2_jpeg(img, int(rng.randint(30, 100)), list(J.SAMPLINGS)[i % 5], restart=int(rng.randint(0, 4)))
        (d / f"im{i:03d}.jpg").write_bytes(data)
    return d


def _data_cfg(decode, batch_size=1):
    return {"name": "COCO", "class_name": "COCO", "experiment_name": f"jpeg_{decode}", "preprocessing": {"resize": [240, 320]},
            "has_labels": False, "warped_pair": False, "batch_size": batch_size, "truncate": False, "decode": decode,
            "decode_batch": 8, "augmentation": {"photometric": {"enable": False}, "homographic": {"enable": False}}}


def _batches(decode, world=1, rank=0):
    from superpoint_nerf_pytorch_b200.utils.data_loaders import get_loader
    cfg = {"data": _data_cfg(decode, batch_size=3)}
    loader = get_loader(cfg, "export_pseudo_labels", device="cuda:0", export_split="training", rank=rank, world=world)
    return [(b["name"], b["raw"]["image"].cpu().numpy()) for b in loader]


@pytest.fixture()
def data_dir(tmp_path, monkeypatch):
    from superpoint_nerf_pytorch_b200 import settings
    d = _write_dir(tmp_path)
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    return d


@pytest.mark.parametrize("world", [1, 2])
def test_loader_device_decode_matches_host(data_dir, world):
    for rank in range(world):
        host, dev = _batches("host", world, rank), _batches("device", world, rank)
        assert [n for n, _ in host] == [n for n, _ in dev]
        for (_, a), (_, b) in zip(host, dev):
            assert a.dtype == np.float32 and a.shape[1:] == (1, 240, 320) and np.array_equal(a, b)


@pytest.mark.parametrize("corruption", ["entropy_third", "no_eoi_1", "no_eoi_2", "header"])
def test_loader_corrupt_file_same_in_both_modes(data_dir, corruption):
    good = (data_dir / "im010.jpg").read_bytes()
    sos = good.index(b"\xff\xda") + 20
    bad = {"entropy_third": good[:sos + (len(good) - sos) // 3], "no_eoi_1": good[:-1], "no_eoi_2": good[:-2],
           "header": b"\xff\xd8\xff\xe0\x00\x10garbage"}[corruption]
    (data_dir / "im010.jpg").write_bytes(bad)
    results = {}
    for mode in ("host", "device"):
        try:
            results[mode] = ("ok", _batches(mode))
        except Exception as e:   # noqa: BLE001 - the type is what both modes must agree on
            results[mode] = ("raise", type(e))
    assert results["host"][0] == results["device"][0]
    if results["host"][0] == "raise":
        assert results["host"][1] is results["device"][1]
    else:
        for (na, a), (nb, b) in zip(results["host"][1], results["device"][1]):
            assert na == nb and np.array_equal(a, b)


def test_export_writes_identical_files(data_dir, tmp_path):
    from conftest import HA_CFG, MP_MODEL
    from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportDetections
    from superpoint_nerf_pytorch_b200.utils.data_loaders import get_loader
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    from oracle import spn_oracle as O
    for p in sorted(data_dir.iterdir())[16:]:
        p.unlink()
    sd = O.make_state_dict("magicpoint", seed=1, logit_gain=10.0)
    outs = {}
    for mode in ("host", "device"):
        cfg = {"data": _data_cfg(mode), "model": dict(copy.deepcopy(MP_MODEL), precision="f16"),
               "homography_adaptation": dict(copy.deepcopy(HA_CFG), num=8, sampler="device", seed=1)}
        model = get_model(copy.deepcopy(cfg["model"]), "cuda:0").eval()
        model.load_state_dict(sd)
        loader = get_loader(cfg, "export_pseudo_labels", device="cuda:0", export_split="training")
        ExportDetections(cfg, model, loader, "training", True, "cuda:0")
        torch.cuda.synchronize()
        d = Path(tmp_path, "exper", "outputs", f"jpeg_{mode}", "training")
        outs[mode] = {p.name: np.load(p, allow_pickle=True) for p in sorted(d.glob("*.npy"))}
    assert len(outs["host"]) == 16 and outs["host"].keys() == outs["device"].keys()
    for k in outs["host"]:
        a, b = outs["host"][k], outs["device"][k]
        if a.dtype == object:
            a, b = a.item(), b.item()
            assert a.keys() == b.keys() and all(np.array_equal(np.asarray(a[x]), np.asarray(b[x])) for x in a), k
        else:
            assert np.array_equal(a, b), k
