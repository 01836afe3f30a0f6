import os, sys, copy, torch, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from superpoint_nerf_pytorch_b200.engine_solvers.export import HomographyAdaptation
from superpoint_nerf_pytorch_b200.utils.get_model import get_model
dev=torch.device('cuda',0)
mcfg=dict(copy.deepcopy(bench.MODEL_CFG), precision='f16')
model=get_model(mcfg,dev).eval(); model.load_state_dict(bench.random_init_state_dict())
ha=dict(copy.deepcopy(bench.HA_CFG), sampler='device', seed=1234, max_forwards=100)
eng=HomographyAdaptation({'homography_adaptation':ha,'model':mcfg}, model, dev)
ctx=model.native()
g=torch.Generator().manual_seed(1000)
NI=int(sys.argv[1]) if len(sys.argv)>1 else 4
imgs=torch.rand((NI,1,240,320),generator=g).to(dev)
heat,_=eng.heatmaps(imgs)
print('heat stats', heat.min().item(), heat.max().item(), (heat>=0.015).float().mean().item())
for it in range(3):
    torch.cuda.synchronize(); t=time.perf_counter()
    r=ctx.box_nms(heat,4.0,0.1,0.015,0,det_thresh=0.015,want_map=False,max_kp=16384*4)
    torch.cuda.synchronize(); print('nms ms', (time.perf_counter()-t)*1e3, ctx.nms_stats(NI,240,320), r['kp_count'].tolist())
flat=(1/65+0.0005*torch.randn((NI,240,320),device=dev)).contiguous()
for it in range(2):
    torch.cuda.synchronize(); t=time.perf_counter()
    r=ctx.box_nms(flat,4.0,0.1,0.015,0,det_thresh=0.015,want_map=False,max_kp=16384*4)
    torch.cuda.synchronize(); print('flat nms ms', (time.perf_counter()-t)*1e3, ctx.nms_stats(NI,240,320), r['kp_count'].tolist())
