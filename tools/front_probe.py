"""Bottleneck experiments on front_tc_kernel: time it with parts of each role switched off (SPN_FRONT_DBG bits)."""
import os, sys, copy, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from superpoint_nerf_pytorch_b200.utils.get_model import get_model
dev = torch.device('cuda', 0)
mcfg = dict(copy.deepcopy(bench.MODEL_CFG), precision='f16')
model = get_model(mcfg, dev).eval(); model.load_state_dict(bench.random_init_state_dict())
ctx = model.native()
H, W, NH = 240, 320, 99
imgs = torch.rand((1, H, W), device=dev)
h, hinv = ctx.sample_homographies(bench.HA_CFG["params"], 1, 0, NH, H, W)
hinv = hinv.view(1, NH, 3, 3)
# needs a library built with SPN_FRONT_DBG_BUILD=1 (extra template instantiations)
names = {0: "baseline", 1: "P: no sampling", 2: "P: no A1 rows", 3: "P: nothing", 12: "E1: nothing", 16: "E2: no stores", 32: "E2: no ALU/stores", 96: "E2: nothing",
         128: "M: 4 of 36 MMA2", 111: "only MMAs", 15: "P+E1 off", 108: "E1+E2 off", 99: "P+E2 off", 0.5: "baseline again"}
if os.environ.get("SPN_PROBE_BASELINE_ONLY"):
    names = {0: "baseline"}
for dbg, name in names.items():
    if int(dbg) != 0 or not os.environ.get("SPN_PROBE_BASELINE_ONLY"):
        ctx.set_option("front_variant", int(dbg))
    for _ in range(2):
        ctx.encoder_forward_ha(imgs, hinv, 0, NH + 1, 1)
    torch.cuda.synchronize()
    ctx.profile_enable(True); ctx.profile_read()
    for _ in range(5):
        ctx.encoder_forward_ha(imgs, hinv, 0, NH + 1, 1)
    torch.cuda.synchronize()
    pr = ctx.profile_read(); ctx.profile_enable(False)
    t, n = pr["backbone.block_2"]
    print(f"dbg {int(dbg):3d} {name:22s}: front_tc {t / n:.4f} ms")
