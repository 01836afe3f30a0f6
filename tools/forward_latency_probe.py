import os, copy, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests'))
from conftest import SP_MODEL
from superpoint_nerf_pytorch_b200.utils.get_model import get_model
c = copy.deepcopy(SP_MODEL); c["precision"] = "f16"; c["detector_head"]["top_k"] = 1000
m = get_model(c, "cuda").eval()
x = torch.rand((1, 1, 480, 640), device="cuda")
for _ in range(3): m(x)
torch.cuda.synchronize()
ctx = m.native()
ctx.profile_enable(True); ctx.profile_read()
t0 = time.perf_counter()
for _ in range(10): out = m(x)
torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 10
pr = ctx.profile_read(); ctx.profile_enable(False)
print("wall ms per forward (with events)", dt * 1e3)
tot = 0
for k, (t, n) in sorted(pr.items(), key=lambda kv: -kv[1][0]):
    print(f"{k:28s} {t / 10:.4f} ms ({n // 10} launches)"); tot += t / 10
print("sum of kernels", tot)
import cProfile, pstats, io
pr2 = cProfile.Profile(); pr2.enable()
for _ in range(20): m(x)
torch.cuda.synchronize(); pr2.disable()
s = io.StringIO(); pstats.Stats(pr2, stream=s).sort_stats("tottime").print_stats(12); print(s.getvalue()[:2500])
