"""spn_posed_reproject (include/spn_posed.h) and evaluations/posed_evaluation.py on the GPU: positions, flags, compacted
sets and counts bit-equal to the fp64 oracle (oracle/posed_oracle.py), repeatability and match correctness equal to the
oracle's on the same keypoints and matcher output, argument errors, guard bands, and the CLI end to end."""
import copy

import numpy as np
import pytest
import torch

from conftest import SP_MODEL, make_nerf_batch
from oracle import posed_oracle as O

pytestmark = pytest.mark.gpu

DEPTH_TOL = 0.05


def _model(top_k=300, precision="f16"):
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    cfg = copy.deepcopy(SP_MODEL)
    cfg["detector_head"]["top_k"] = top_k
    cfg["precision"] = precision
    torch.manual_seed(0)
    return get_model(cfg, "cuda").eval()


def _geometry(bt):
    raw = bt["raw"]
    return [x.cuda() for x in (raw["input_depth"], bt["camera_intrinsic_matrix"], raw["input_rotation"], raw["input_translation"])]


def _hand_made(kp, cnt, H, W, rng):
    """View 0: random points with some outside the image; view 1: no keypoints; view 2: a count above max_kp."""
    kp, cnt = kp.clone(), cnt.clone()
    max_kp = kp.shape[1]
    n = min(max_kp, 60)
    pts = np.stack([rng.randint(-3, H + 3, n), rng.randint(-3, W + 3, n)], 1).astype(np.int32)
    pts[:4] = [[-1, 0], [0, W], [H, W - 1], [H - 1, -2]]
    kp[0, :n] = torch.from_numpy(pts).cuda()
    cnt[0] = n
    cnt[1] = 0
    cnt[2] = max_kp + 7
    return kp, cnt


def _check_against_oracle(ctx, kp, cnt, depth, K, R, t, pairs):
    got = ctx.posed_reproject(kp, cnt, depth, K, R, t, pairs, DEPTH_TOL)
    want = O.posed_reproject(kp.cpu().numpy(), cnt.cpu().numpy(), depth.cpu().numpy(), K.cpu().numpy(), R.cpu().numpy(),
                             t.cpu().numpy(), pairs, DEPTH_TOL)
    g = {k: v.cpu().numpy() for k, v in got.items()}
    assert np.array_equal(g["proj"], want["proj"], equal_nan=True)
    assert np.array_equal(g["vis"], want["vis"])
    assert np.array_equal(g["set_count"], want["set_count"])
    assert np.array_equal(g["set1"], want["set1"], equal_nan=True) and np.array_equal(g["set2"], want["set2"], equal_nan=True)
    return got, want


@pytest.mark.parametrize("H,W", [(64, 96), (240, 320), (480, 640)])
@pytest.mark.parametrize("V", [4, 8, 16])
def test_posed_reproject_matches_oracle(V, H, W):
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import pair_list
    model = _model()
    bt = make_nerf_batch(V + H, n_views=V, h=H, w=W)
    depth, K, R, t = _geometry(bt)
    det = model(bt["raw"]["image"].cuda(), keypoints=True)["detector_output"]
    pairs = pair_list(V) + [(a, a) for a in range(V)]
    ctx = model.native()
    got, want = _check_against_oracle(ctx, det["keypoints"], det["keypoint_count"], depth, K, R, t, pairs)
    kp, cnt = _hand_made(det["keypoints"], det["keypoint_count"], H, W, np.random.RandomState(V * W))
    got, want = _check_against_oracle(ctx, kp, cnt, depth, K, R, t, pairs)
    # repeatability counts of the compacted sets equal the brute-force counts
    counts = ctx.repeatability_counts(got["set1"], got["set_count"][:, 0].contiguous(), got["set2"],
                                      got["set_count"][:, 1].contiguous(), 3.0).cpu().numpy()
    assert np.array_equal(counts, O.repeatability_counts(want["set1"], want["set_count"][:, 0], want["set2"], want["set_count"][:, 1], 3.0))
    again = ctx.posed_reproject(kp, cnt, depth, K, R, t, pairs, DEPTH_TOL)
    assert all(torch.equal(got[k].nan_to_num(-1), again[k].nan_to_num(-1)) for k in got)     # deterministic
    print(f"posed_reproject V={V} {H}x{W}: {len(pairs)} pairs, {int(want['set_count'].sum())} visible points")


def test_evaluate_chunk_matches_oracle_on_the_same_keypoints_and_matches():
    from superpoint_nerf_pytorch_b200.evaluations.posed_evaluation import evaluate_chunk, pair_list
    model = _model(top_k=400, precision="fp32")
    V, H, W = 6, 240, 320
    bt = make_nerf_batch(77, n_views=V, h=H, w=W)
    ev = {"distance_thresh": 3.0, "depth_tol": DEPTH_TOL, "max_gap": 0, "pose": False, "pose_thresh_px": 1.0}
    res = evaluate_chunk(model, bt, ev)
    out = model(bt["raw"]["image"].cuda(), keypoints=True)
    kp, cnt = out["detector_output"]["keypoints"], out["detector_output"]["keypoint_count"]
    desc = out["descriptor_output"]["desc_sparse"]
    depth, K, R, t = _geometry(bt)
    pairs = pair_list(V)
    want = O.posed_reproject(kp.cpu().numpy(), cnt.cpu().numpy(), depth.cpu().numpy(), K.cpu().numpy(), R.cpu().numpy(),
                             t.cpu().numpy(), pairs, DEPTH_TOL)
    counts = O.repeatability_counts(want["set1"], want["set_count"][:, 0], want["set2"], want["set_count"][:, 1], 3.0)
    assert np.array_equal(np.stack([res["N1"], res["N2"], res["count1"], res["count2"]], 1), counts)
    ctx = model.native()
    kp_h = kp.cpu().numpy()
    for q, (a, b) in enumerate(pairs):
        m, _ = ctx.mutual_nn_match(desc[a:a + 1], cnt[a:a + 1], desc[b:b + 1], cnt[b:b + 1])
        nm, nc = O.match_correct(want["proj"][q], want["vis"][q, 0], kp_h[b], m[0].cpu().numpy(), 3.0)
        assert (res["n_matches"][q], res["n_correct"][q]) == (nm, nc), (q, a, b)
    assert res["n_matches"].sum() > 0
    print(f"evaluate_chunk: {len(pairs)} pairs, repeatability {np.nanmean(res['repeatability']):.3f}, "
          f"{res['n_correct'].sum()} / {res['n_matches'].sum()} matches correct")


def test_posed_reproject_errors_and_guard_bands():
    import ctypes as C

    import superpoint_nerf_pytorch_b200 as P
    ctx = P.Context(0)
    ctx.set_option("ws_guard", 1)
    V, H, W = 4, 48, 72
    bt = make_nerf_batch(5, n_views=V, h=H, w=W)
    depth, K, R, t = _geometry(bt)
    rng = np.random.RandomState(0)
    kp = torch.from_numpy(np.stack([rng.randint(0, H, 50), rng.randint(0, W, 50)], 1).astype(np.int32)[None].repeat(V, 0)).cuda()
    cnt = torch.full((V,), 50, dtype=torch.int32, device="cuda")
    pairs = [(0, 1), (2, 3), (1, 1)]
    want = ctx.posed_reproject(kp, cnt, depth, K, R, t, pairs, DEPTH_TOL)
    with pytest.raises(P.NativeError, match=r"pair 1 = \(2, 4\) has a view index outside \[0, 4\)"):
        ctx.posed_reproject(kp, cnt, depth, K, R, t, [(0, 1), (2, 4)], DEPTH_TOL)
    with pytest.raises(P.NativeError, match="view index"):
        ctx.posed_reproject(kp, cnt, depth, K, R, t, [(-1, 0)], DEPTH_TOL)
    with pytest.raises(P.NativeError, match="depth_tol"):
        ctx.posed_reproject(kp, cnt, depth, K, R, t, pairs, -1.0)
    with pytest.raises(P.NativeError, match="do not match depth"):
        ctx.posed_reproject(kp[:3], cnt, depth, K, R, t, pairs, DEPTH_TOL)
    out = [torch.empty_like(want[k]) for k in ("proj", "vis", "set1", "set2", "set_count")]
    pr = np.asarray(pairs, np.int32)
    ptr = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
    for shape, msg in (((V, H, 40000), "bad shape"), ((0, H, W), "bad shape")):
        with pytest.raises(P.NativeError, match=msg):
            ctx._call("spn_posed_reproject", ctx.handle, ptr(kp), ptr(cnt), 50, ptr(depth), ptr(K), ptr(R), ptr(t), *shape, len(pairs),
                      C.c_void_p(pr.ctypes.data), C.c_double(DEPTH_TOL), *map(ptr, out), ctx._s())
    with pytest.raises(P.NativeError, match="max_kp"):
        ctx._call("spn_posed_reproject", ctx.handle, ptr(kp), ptr(cnt), 0, ptr(depth), ptr(K), ptr(R), ptr(t), V, H, W, len(pairs),
                  C.c_void_p(pr.ctypes.data), C.c_double(DEPTH_TOL), *map(ptr, out), ctx._s())
    again = ctx.posed_reproject(kp, cnt, depth, K, R, t, pairs, DEPTH_TOL)        # the context still works
    assert all(torch.equal(want[k].nan_to_num(-1), again[k].nan_to_num(-1)) for k in want)
    empty = ctx.posed_reproject(kp, cnt, depth, K, R, t, [], DEPTH_TOL)            # P = 0: a no-op
    assert empty["proj"].shape == (0, 50, 2) and empty["set_count"].shape == (0, 2)
    for V, H, W in ((3, 37, 53), (5, 61, 90), (2, 200, 17), (4, 9, 11)):
        bt = make_nerf_batch(V * H, n_views=V, h=H, w=W)
        depth, K, R, t = _geometry(bt)
        kp = torch.from_numpy(np.stack([rng.randint(-1, H + 1, (V, 333)), rng.randint(-1, W + 1, (V, 333))], -1).astype(np.int32)).cuda()
        cnt = torch.from_numpy(rng.randint(0, 340, V).astype(np.int32)).cuda()
        pairs = [(a, b) for a in range(V) for b in range(V)]
        _check_against_oracle(ctx, kp, cnt, depth, K, R, t, pairs)
    assert ctx.check_guards() == 0
    ctx.close()


def test_cli_posed_evaluation_end_to_end(tmp_path, monkeypatch):
    """The CLI on a scene tree writes the same pairs.npz as a direct evaluate_posed_views call; a second run gives
    byte-identical files."""
    import yaml
    from nerf_scenes import write_tree
    from superpoint_nerf_pytorch_b200 import settings
    from superpoint_nerf_pytorch_b200.data.PosedViews import PosedViews
    from superpoint_nerf_pytorch_b200.evaluations import posed_evaluation as PE
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    write_tree(tmp_path / "data", scenes=(("sceneA", 3, 6), ("sceneB", 4, 5)))
    monkeypatch.setattr(settings, "DATA_PATH", str(tmp_path / "data"))
    monkeypatch.setattr(settings, "EXPER_PATH", str(tmp_path / "exper"))
    cfg = yaml.safe_load(open(PE.Path(PE.__file__).parents[1] / "configs" / "superpoint_posed_eval.yaml"))
    cfg["data"].update(batch_size=4, preprocessing={"resize": [64, 96]}, experiment_name="cli")
    cfg["model"]["precision"] = "fp32"
    cfg["model"]["detector_head"].update(det_thresh=0.001, top_k=100)
    cfg_path = tmp_path / "eval.yaml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    PE.main(config_path=str(cfg_path), random_init=True)
    out_dir = tmp_path / "exper" / "posed_eval" / "cli" / "training"
    cli = np.load(out_dir / "pairs.npz")
    # chunks of 4, 2, 4 and 1 views: 6 + 1 + 6 + 0 pairs
    assert len(cli["a"]) == 13 and cli["name_a"][0] == "sceneA_f000" and cli["name_b"][-1] == "sceneB_f003"

    torch.manual_seed(0)
    model = get_model(copy.deepcopy(cfg["model"]), device="cuda:0")
    ds = PosedViews(cfg["data"], task="training", device="cpu")
    direct_cfg = dict(cfg, data=dict(cfg["data"], experiment_name="direct"))
    summary = PE.evaluate_posed_views(direct_cfg, model, [ds[i] for i in range(len(ds))], "training")
    direct = np.load(tmp_path / "exper" / "posed_eval" / "direct" / "training" / "pairs.npz")
    assert sorted(cli.files) == sorted(direct.files)
    for k in cli.files:
        assert np.array_equal(cli[k], direct[k], equal_nan=cli[k].dtype.kind == "f"), k
    assert summary["n_pairs"] == 13 and "pose_auc@5" in summary
    before = {f.name: f.read_bytes() for f in out_dir.iterdir()}
    PE.main(config_path=str(cfg_path), random_init=True)
    assert {f.name: f.read_bytes() for f in out_dir.iterdir()} == before
    print("posed evaluation summary:", summary)
