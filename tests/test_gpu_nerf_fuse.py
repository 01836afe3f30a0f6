"""spn_nerf_fuse (include/spn_nerf.h) and the export_NeRF_labels task on the GPU: the fused heatmaps against the per-pair
composition ExportNeRFDetections.reproject -> stack -> sum -> / (n+1), the reference's step goldens replayed through the
fused kernel, the export's keypoints against the per-pair path, the CLI end to end, argument errors and guard bands.

Gate for heatmaps (the one of test_nerf_reproject_vs_reference_step_golden): the re-projection runs in fp32 with its
own 3x3 inverses, so a point within an ulp of an integer may truncate to the neighbouring pixel; at most 0.5 % of the
pixels may fail isclose(rtol=1e-6, atol=0).  Each test prints the fraction it measured."""
import copy
import random
import types

import numpy as np
import pytest
import torch

from conftest import MP_MODEL, keypoint_agreement, make_nerf_batch

pytestmark = pytest.mark.gpu

GATE = 5e-3


def _exporter(model_or_ctx):
    from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportNeRFDetections
    ex = object.__new__(ExportNeRFDetections)
    if hasattr(model_or_ctx, "native"):
        ex.model = model_or_ctx
    else:
        ex.model = types.SimpleNamespace(native=lambda slot=0: model_or_ctx)
    ex.device = "cuda"
    return ex


def _bad_fraction(got, want):
    got, want = got.cpu().numpy(), want.cpu().numpy()
    return float((~np.isclose(got, want, rtol=1e-6, atol=0)).mean())


def _views(seed, V, H, W):
    """A make_nerf_batch geometry of V views with sparse heatmaps and keypoint lists that include border points, a view
    without keypoints and points the border filter drops."""
    rng = np.random.RandomState(1000 + seed)
    bt = make_nerf_batch(seed, n_views=V, h=H, w=W)
    prob = (rng.rand(V, H, W) * 0.02).astype(np.float32)
    n_kp = max(8, H * W // 150)
    kp = np.zeros((V, n_kp + 16, 2), np.int32)
    cnt = np.zeros(V, np.int32)
    for v in range(V):
        if v == 1:
            continue                                       # a source without keypoints
        flat = rng.choice(H * W, n_kp, replace=False)
        pts = np.stack([flat // W, flat % W], 1)
        border = np.array([[0, rng.randint(W)], [1, rng.randint(W)], [H - 1, rng.randint(W)], [H - 2, rng.randint(W)],
                           [rng.randint(H), 0], [rng.randint(H), 1], [rng.randint(H), W - 1], [rng.randint(H), W - 2],
                           [2, 2], [H - 3, W - 3]])
        pts = np.unique(np.concatenate([pts, border]), axis=0)           # row-major order, like the NMS lists
        cnt[v] = len(pts)
        kp[v, :len(pts)] = pts
        prob[v, pts[:, 0], pts[:, 1]] = rng.uniform(0.05, 1.0, len(pts)).astype(np.float32)
    data = {"raw": {k: v.cuda() for k, v in bt["raw"].items()}, "camera_intrinsic_matrix": bt["camera_intrinsic_matrix"].cuda()}
    return torch.from_numpy(prob).cuda(), torch.from_numpy(kp).cuda(), torch.from_numpy(cnt).cuda(), cnt, data


def _pairs(V, rng):
    """Targets of every view (one twice), random.choices-style sources with repeats, explicit duplicates and a target
    without sources."""
    targets, offsets, sources = [], [0], []
    for j in list(range(V)) + [0]:
        others = [k for k in range(V) if k != j]
        src = [others[i] for i in rng.randint(0, len(others), int(0.75 * len(others)))]
        if j == 2 % V:
            src = src + src[:2]                            # duplicates, in summation order
        if j == V - 1:
            src = []                                       # out = prob[j]
        targets.append(j)
        sources += src
        offsets.append(len(sources))
    return targets, offsets, sources


def _fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources):
    raw = data["raw"]
    return ctx.nerf_fuse(prob, kp, kp_count, raw["input_depth"], data["camera_intrinsic_matrix"], raw["input_rotation"],
                         raw["input_translation"], targets, offsets, sources)


@pytest.mark.parametrize("H,W", [(64, 96), (240, 320), (480, 640)])
@pytest.mark.parametrize("V", [4, 5, 8, 16])
def test_nerf_fuse_matches_per_pair_composition(V, H, W):
    import superpoint_nerf_pytorch_b200 as P
    ctx = P.get_context("cuda:0")
    prob, kp, kp_count, cnt, data = _views(V + H, V, H, W)
    targets, offsets, sources = _pairs(V, np.random.RandomState(V * 7 + W))
    got = _fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources)
    want = _exporter(ctx).fuse_per_pair(prob, kp, cnt, data, targets, offsets, sources)
    assert got.shape == want.shape == (len(targets), H, W)
    bad = _bad_fraction(got, want)
    print(f"nerf_fuse V={V} {H}x{W}: {len(sources)} pairs, fraction of pixels off {bad:.2e}")
    assert bad <= GATE
    assert torch.equal(got[targets.index(V - 1)], prob[V - 1])      # no sources: the view's own heatmap, bit for bit
    again = _fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources)
    assert torch.equal(got, again)                                  # deterministic


def test_nerf_fuse_replays_the_reference_step_golden(golden):
    """nerf_step.npz holds ExportNeRFDetections.step of the unmodified reference for one (j, k) pair per case.  With a zero
    heatmap for j and that single pair, 2 * out is the reference's splat."""
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    g = golden("nerf_step.npz")
    ctx = get_model(dict(copy.deepcopy(MP_MODEL), precision="fp32"), "cuda").eval().native()
    det = float(g["det_thresh"])
    worst = 0.0
    for c in range(int(g["n"])):
        bseed, nv, j, k = (int(v) for v in g[f"case{c}"])
        bt = make_nerf_batch(bseed, n_views=nv)
        data = {"raw": {kk: v.cuda() for kk, v in bt["raw"].items()}, "camera_intrinsic_matrix": bt["camera_intrinsic_matrix"].cuda()}
        heat = torch.from_numpy(g[f"heat{c}"]).cuda()
        H, W = heat.shape
        r = ctx.box_nms(heat[None], float(g["nms"]), 0.1, det, int(g["top_k"]), det_thresh=det, want_map=False, max_kp=4096)
        prob = torch.zeros((nv, H, W), device="cuda")
        prob[k] = heat
        kp = torch.zeros((nv, 4096, 2), dtype=torch.int32, device="cuda")
        kp[k] = r["kp"][0]
        kp_count = torch.zeros(nv, dtype=torch.int32, device="cuda")
        kp_count[k] = r["kp_count"][0]
        out = _fuse(ctx, prob, kp, kp_count, data, [j], [0, 1], [k])
        bad = float((~np.isclose(2 * out[0].cpu().numpy(), g[f"splat{c}"], rtol=1e-6, atol=0)).mean())
        worst = max(worst, bad)
        assert bad <= GATE, (c, bad)
    print(f"nerf_fuse golden step replay: worst fraction of pixels off {worst:.2e}")


def _per_pair_export(ex, batch, dh):
    """The per-pair export loop (one reproject per pair, one box_nms per target) -> {name: keypoints}."""
    data = {"raw": {k: v.cuda() for k, v in batch["raw"].items()}, "camera_intrinsic_matrix": batch["camera_intrinsic_matrix"].cuda()}
    names = batch["name"]
    out = ex.model(data["raw"]["image"], keypoints=True)["detector_output"]
    prob, kp, cnt = out["prob_heatmap"], out["keypoints"], out["keypoint_count"].cpu().numpy()
    ctx = ex.model.native()
    res = {}
    for j in range(len(names)):
        others = [k for k in range(len(names)) if k != j]
        others = random.choices(others, k=int(0.75 * len(others)))
        mean = ex.fuse_per_pair(prob, kp, cnt, data, [j], [0, len(others)], others)
        r = ctx.box_nms(mean, float(dh["nms"]), 0.1, float(dh["det_thresh"]), int(dh["top_k"]), det_thresh=float(dh["det_thresh"]),
                        want_map=False, max_kp=16384)
        n = int(r["kp_count"][0])
        res[names[j]] = r["kp"][0, :n].cpu().numpy().astype(np.int64)
    return res


@pytest.mark.parametrize("V", [8, 16])
def test_export_keypoints_match_the_per_pair_path(V, golden, tmp_path, monkeypatch):
    from oracle import spn_oracle as O
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportNeRFDetections
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    g = golden("nerf_export.npz")
    mcfg = copy.deepcopy(MP_MODEL)
    mcfg["detector_head"]["top_k"] = 300
    mcfg["precision"] = "fp32"
    m = get_model(mcfg, "cuda").eval()
    m.load_state_dict(O.make_state_dict("magicpoint", seed=int(g["seed"]), logit_gain=float(g["gain"])))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path))
    batches = [make_nerf_batch(20 + V, n_views=V, h=120, w=160), make_nerf_batch(21 + V, n_views=V, h=120, w=160)]
    random.seed(int(g["py_seed"]))
    ExportNeRFDetections({"data": {"experiment_name": "fused"}, "model": mcfg}, m, batches, "training", "cuda")
    random.seed(int(g["py_seed"]))
    ex = _exporter(m)
    want = {}
    for bt in batches:
        want.update(_per_pair_export(ex, bt, mcfg["detector_head"]))
    worst, total = 1.0, 0
    for nm, kp_want in want.items():
        kp = np.load(tmp_path / "outputs" / "fused" / "training" / f"{nm}.npy")
        assert kp.dtype == np.int64 and kp.ndim == 2 and kp.shape[1] == 2
        a, b = keypoint_agreement(kp, kp_want)
        worst = min(worst, a, b)
        total += len(kp)
    print(f"NeRF export V={V}: {total} keypoints, worst agreement with the per-pair path {worst:.4f}")
    assert total > 0 and worst >= 0.995


def test_cli_export_nerf_labels_end_to_end(tmp_path, monkeypatch):
    """--task export_NeRF_labels on a scene tree: every file equals what ExportNeRFDetections writes when fed the same
    chunks with the same seeds; a second run writes nothing and changes no file."""
    import tyro
    import yaml
    from nerf_scenes import write_tree
    from superpoint_nerf_pytorch_b200 import engine, settings
    from superpoint_nerf_pytorch_b200.data.PosedViews import PosedViews
    from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportNeRFDetections
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    write_tree(tmp_path / "data", scenes=(("sceneA", 3, 6), ("sceneB", 4, 5)))
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(engine.Path(engine.__file__).parent / "configs" / "magicpoint_nerf_export.yaml"))
    cfg["data"].update(batch_size=4, preprocessing={"resize": [64, 96]}, experiment_name="cli")
    cfg["model"]["precision"] = "fp32"
    cfg_path = tmp_path / "nerf.yaml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    random.seed(11)                        # engine.main itself draws nothing before the export (tyro's parser does)
    engine.main(config_path=str(cfg_path), task="export_NeRF_labels", random_init=True)
    out_dir = tmp_path / "exper" / "outputs" / "cli" / "training"
    files = sorted(out_dir.glob("*.npy"))
    assert len(files) == 11

    ds = PosedViews(cfg["data"], task="training", device="cpu")
    random.seed(11)
    torch.manual_seed(0)
    model = get_model(copy.deepcopy(cfg["model"]), device="cuda:0")
    ExportNeRFDetections(dict(cfg, data=dict(cfg["data"], experiment_name="direct")), model, [ds[i] for i in range(len(ds))],
                         "training", "cuda:0")
    direct = tmp_path / "exper" / "outputs" / "direct" / "training"
    for f in files:
        a, b = np.load(f), np.load(direct / f.name)
        assert a.dtype == np.int64 and np.array_equal(a, b), f.name
    before = {f.name: (f.stat().st_mtime_ns, f.read_bytes()) for f in files}
    tyro.cli(engine.main, use_underscores=True, args=["--config_path", str(cfg_path), "--task", "export_NeRF_labels",
                                                      "--random_init", "True"])
    after = {f.name: (f.stat().st_mtime_ns, f.read_bytes()) for f in sorted(out_dir.iterdir())}
    assert after == before


def test_nerf_fuse_argument_errors_and_guard_bands():
    import superpoint_nerf_pytorch_b200 as P
    ctx = P.Context(0)
    ctx.set_option("ws_guard", 1)
    prob, kp, kp_count, cnt, data = _views(3, 5, 48, 72)
    targets, offsets, sources = _pairs(5, np.random.RandomState(3))
    want = _fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources)
    cases = [
        (([7], [0, 1], [0]), "view index 7"),                       # target outside [0, V)
        (([0], [0, 1], [-1]), "source view index -1"),              # source outside [0, V)
        (([0, 1], [0, 2, 1], [1]), "not monotone"),
        (([0], [1, 1], [2]), "must be 0"),
    ]
    for (tg, off, src), msg in cases:
        with pytest.raises(P.NativeError, match=msg):
            _fuse(ctx, prob, kp, kp_count, data, tg, off, src)
    import ctypes as C
    raw = data["raw"]
    arrays = [np.asarray(targets, np.int32), np.asarray(offsets, np.int32), np.asarray(sources, np.int32)]
    with pytest.raises(P.NativeError, match="max_kp"):                # max_kp = 0 with valid pointers
        ctx._call("spn_nerf_fuse", ctx.handle, *[C.c_void_p(x.data_ptr()) for x in (prob, kp, kp_count)], 0,
                  *[C.c_void_p(x.data_ptr()) for x in (raw["input_depth"], data["camera_intrinsic_matrix"], raw["input_rotation"],
                                                       raw["input_translation"])],
                  5, 48, 72, len(targets), *[C.c_void_p(a.ctypes.data) for a in arrays], C.c_void_p(want.data_ptr()), ctx._s())
    with pytest.raises(P.NativeError, match="bad shape"):
        small = {"raw": dict(data["raw"], input_depth=data["raw"]["input_depth"][:, :2, :2].contiguous()),
                 "camera_intrinsic_matrix": data["camera_intrinsic_matrix"]}
        _fuse(ctx, prob[:, :2, :2].contiguous(), kp, kp_count, small, targets, offsets, sources)
    assert torch.equal(_fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources), want)   # the context still works
    assert _fuse(ctx, prob, kp, kp_count, data, [], [0], []).shape == (0, 48, 72)
    for V, H, W in ((3, 37, 53), (6, 61, 90), (4, 29, 131), (2, 200, 17)):
        prob, kp, kp_count, cnt, data = _views(V * H, V, H, W)
        targets, offsets, sources = _pairs(V, np.random.RandomState(W))
        got = _fuse(ctx, prob, kp, kp_count, data, targets, offsets, sources)
        bad = _bad_fraction(got, _exporter(ctx).fuse_per_pair(prob, kp, cnt, data, targets, offsets, sources))
        assert bad <= GATE, (V, H, W, bad)
    assert ctx.check_guards() == 0
    ctx.close()
