"""Error behaviour at the drop-in boundary on a GPU box (include/spn_b200.h: negative SPN_E_* code + spn_last_error(),
surfaced by the binding as NativeError; the Python mirror raises ValueError for configurations the reference does not
support either).  After every rejected call the context must still work."""
import copy

import numpy as np
import pytest
import torch

from conftest import HA_CFG, MP_MODEL
from oracle import spn_oracle as O

pytestmark = pytest.mark.gpu


def test_cabi_argument_and_state_errors():
    import superpoint_nerf_pytorch_b200 as P
    from superpoint_nerf_pytorch_b200._native import MODE_F16, MODE_FP32
    ctx = P.Context(0)                                   # fresh context: no weights, no feature map
    x = torch.rand((1, 16, 24), device="cuda")
    with pytest.raises(P.NativeError, match="multiples of 8"):
        ctx.encoder_forward(torch.rand((1, 12, 20), device="cuda"), MODE_FP32)
    with pytest.raises(P.NativeError, match="no weights"):
        ctx.encoder_forward(x, MODE_FP32)
    with pytest.raises(P.NativeError, match="no feature map"):
        ctx.detector_head_forward(1, 16, 24, MODE_FP32)
    for name in ("no_such_switch", "fold", "fold_hybrid", "front_pair", "front_variant", "pdl"):
        with pytest.raises(P.NativeError, match="unknown option"):
            ctx.set_option(name, 1)
    with pytest.raises(P.NativeError, match="CUDA tensor"):
        ctx.encoder_forward(x.cpu(), MODE_FP32)
    with pytest.raises(P.NativeError, match="float32"):
        ctx.encoder_forward(x.double(), MODE_FP32)
    with pytest.raises(P.NativeError, match="CUDA tensor"):
        ctx.box_nms(torch.rand((1, 16, 24)), 4)
    ctx.load_state_dict(O.make_state_dict("magicpoint", seed=3))
    with pytest.raises(P.NativeError, match="tensor-core modes only"):
        ctx.encoder_forward_ha(x, None, 0, 1, MODE_FP32)
    with pytest.raises(P.NativeError, match="slot range"):
        ctx.encoder_forward_ha(x, None, 0, 2, MODE_F16)  # 1 image, no homographies: only slot 0 exists
    with pytest.raises(P.NativeError, match="no feature map"):
        ctx.encoder_forward(x, MODE_FP32)
        ctx.detector_head_forward(1, 16, 24, MODE_F16)   # feature map of another mode
    # the context survives all of the above: a valid pass still matches the oracle
    ctx.encoder_forward(x, MODE_FP32)
    prob, _ = ctx.detector_head_forward(1, 16, 24, MODE_FP32)
    want = O.model_forward(O.make_state_dict("magicpoint", seed=3), x.cpu().unsqueeze(1), dict(MP_MODEL, detector_head=dict(MP_MODEL["detector_head"], nms=0)))
    ref = want["detector_output"]["prob_heatmap"].numpy()
    assert np.abs(prob.cpu().numpy() - ref).max() / np.abs(ref).max() < 1e-4
    ctx.close()


def test_python_mirror_rejects_what_the_path_does_not_support():
    import superpoint_nerf_pytorch_b200 as P
    from superpoint_nerf_pytorch_b200.engine_solvers.export import HomographyAdaptation
    from superpoint_nerf_pytorch_b200.utils.get_model import get_model
    with pytest.raises(ValueError, match="precision"):
        get_model(dict(copy.deepcopy(MP_MODEL), precision="int8"), "cuda")
    with pytest.raises(ValueError, match="vgg_cn"):
        get_model(dict(copy.deepcopy(MP_MODEL), vgg_cn=[32] * 8), "cuda")
    m = get_model(copy.deepcopy(MP_MODEL), "cuda").eval()
    with pytest.raises(P.NativeError, match="inference-only"):
        m.train()
    with pytest.raises(P.NativeError, match="CUDA tensor"):
        m(torch.rand(1, 1, 16, 24))
    with pytest.raises(ValueError, match=r"\(B,1,H,W\)"):
        m(torch.rand(1, 3, 16, 24, device="cuda"))
    with pytest.raises(P.NativeError, match="multiples of 8"):
        m(torch.rand(1, 1, 20, 24, device="cuda"))
    with pytest.raises(ValueError, match="valid_border_margin"):
        HomographyAdaptation({"homography_adaptation": dict(copy.deepcopy(HA_CFG), valid_border_margin=0), "model": MP_MODEL}, m, "cuda")
    out = m(torch.rand(2, 1, 16, 24, device="cuda"))     # still usable
    assert bool(torch.isfinite(out["detector_output"]["prob_heatmap"]).all())
    with pytest.raises(P.NativeError, match="CUDA only"):
        get_model(copy.deepcopy(MP_MODEL), "cpu").eval().native()
