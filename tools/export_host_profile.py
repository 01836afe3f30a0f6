import os, copy, sys, tempfile, time, cProfile, pstats, io
from pathlib import Path
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from superpoint_nerf_pytorch_b200 import settings
from superpoint_nerf_pytorch_b200.engine import SyntheticLoader
from superpoint_nerf_pytorch_b200.engine_solvers.export import ExportDetections
from superpoint_nerf_pytorch_b200.utils.get_model import get_model
mcfg = dict(copy.deepcopy(bench.MODEL_CFG), precision="f16")
model = get_model(mcfg, "cuda").eval(); model.load_state_dict(bench.random_init_state_dict())
ha = dict(copy.deepcopy(bench.HA_CFG), sampler="device", images_per_launch=16, max_forwards=100, streams=1)
cfg = {"data": {"experiment_name": "task"}, "homography_adaptation": ha, "model": mcfg}
with tempfile.TemporaryDirectory() as tmp:
    settings.EXPER_PATH = tmp
    ExportDetections(cfg, model, SyntheticLoader(32, (240, 320), "export_pseudo_labels", seed=10**6), "warm", True, "cuda")
    torch.cuda.synchronize()
    pr = cProfile.Profile(); pr.enable(); t0 = time.perf_counter()
    ExportDetections(cfg, model, SyntheticLoader(1024, (240, 320), "export_pseudo_labels"), "training", True, "cuda")
    torch.cuda.synchronize(); dt = time.perf_counter() - t0; pr.disable()
print("img/s", 1024 / dt, "ms per 16-image group", dt / 64 * 1e3)
s = io.StringIO(); pstats.Stats(pr, stream=s).sort_stats("cumulative").print_stats(28); print(s.getvalue()[:6000])
