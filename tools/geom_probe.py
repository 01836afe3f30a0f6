"""Times (and, under ncu, exposes) the mask and aggregate kernels alone on the bench workload's geometry."""
import os, sys, copy, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from superpoint_nerf_pytorch_b200 import _native

dev = torch.device('cuda', 0)
ctx = _native.Context(0)
NI, NH, H, W = 16, 99, 240, 320
hp = dict(bench.HA_CFG["params"])
h, hinv = ctx.sample_homographies(hp, 1234, 0, NI * NH, H, W)
hinv, h = (t.view(NI, NH, 3, 3) for t in ctx.kornia_matrices(h, H, W))   # fwd (masks), bwd (aggregate)
imgs = torch.rand((NI, H, W), device=dev)
probs = torch.rand((NI, NH + 1, H, W), device=dev)
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
for name, fn in (("mask", lambda: ctx.warp_batch(imgs, hinv, 3, want_warped=False)),
                 ("aggregate", lambda: ctx.ha_aggregate(probs, h, 3))):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    print(name, "ms per call", e0.elapsed_time(e1) / reps)
