"""Per-kernel time of box_nms (+ top-k) for a single image and for a batch, from the context's CUDA-event profile."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from superpoint_nerf_pytorch_b200 import _native
ctx = _native.Context(0)
dev = torch.device('cuda', 0)
g = torch.Generator().manual_seed(7)
for (B, H, W, top_k) in ((1, 240, 320, 0), (1, 480, 640, 0), (1, 480, 640, 1000), (16, 240, 320, 0), (128, 240, 320, 0)):
    heat = (torch.rand((B, H, W), generator=g) ** 8 * 0.2).to(dev)      # sparse peaks, a few percent above the threshold
    for _ in range(3):
        r = ctx.box_nms(heat, 4.0, 0.1, 0.015, top_k, det_thresh=0.015, want_map=False, max_kp=16384)
    torch.cuda.synchronize()
    ctx.profile_enable(True); ctx.profile_read()
    n = 20
    for _ in range(n):
        r = ctx.box_nms(heat, 4.0, 0.1, 0.015, top_k, det_thresh=0.015, want_map=False, max_kp=16384)
    torch.cuda.synchronize()
    pr = ctx.profile_read(); ctx.profile_enable(False)
    t, c = pr["box_nms"]
    print(f"B {B:3d} {H}x{W} top_k {top_k:4d}: box_nms (rounds + ordered emission) {t / c * 1e3:.1f} us per call, "
          f"{int(r['kp_count'].float().mean())} keypoints per image, rounds {ctx.nms_stats(B, H, W)['global_rounds']}")
