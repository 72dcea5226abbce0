"""-m gpu parity tests of the IoUNet row (SURVEY.md 8(f).1): the IoU feature branch of the network plan, `predict_iou` with its
analytic box gradient, and the on-device refinement loops -- against what the UNMODIFIED reference modules computed on PyTorch-CPU
(autograd, the oracle's independent PrRoIPool restatement) for the same seeded weights and inputs (tests/golden/iou.npz,
oracle/gen_iou_golden.py); and the plug-in's `predict_iou` seam inside the reference tracker's own autograd code when a pytracking
checkout is importable."""
import os

import numpy as np
import pytest
import torch

from oracle import gen_iou_golden as G

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "iou.npz")


def _setup():
    from baseline import ref_env
    if not ref_env.reference_available():
        pytest.skip("reference tree not staged (baseline/_ref)")
    from oracle import ref_shims
    ref_shims.install()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from baseline import ref_tracker
    net = ref_tracker.build_dimp_net("resnet50", seed=0)
    # non-trivial BN statistics in the IoUNet (the constructor leaves running_mean 0 / running_var 1)
    g = torch.Generator().manual_seed(5)
    for m in net.bb_regressor.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(0.05 * torch.randn(m.running_mean.shape, generator=g))
            m.running_var.copy_(0.7 + 0.6 * torch.rand(m.running_var.shape, generator=g))
            m.bias.data.copy_(0.05 * torch.randn(m.bias.shape, generator=g))
    with torch.no_grad():
        net.bb_regressor.iou_predictor.weight.mul_(20.0)      # box gradients of O(1e-2): the refinement loops move boxes by pixels
    return net


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _rel_elem(a, b, floor):
    """element-wise relative error, with the denominator floored at `floor` x the largest reference magnitude"""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float(((a - b).abs() / b.abs().clamp(min=floor * b.abs().max())).max())


def test_iou_feature_branch_matches_reference_get_iou_feat():
    from pytracking_b200.engine import BackboneEngine
    d = np.load(GOLDEN)
    sd = G.make_dimp_iou_state_dict()
    im = G.crop_input()
    eng = BackboneEngine(sd, arch="resnet50", max_batch=2, crop_size=288)
    eng.attach_iou_head(sd)
    out = eng.forward(im.cuda(), want=("layer2", "layer3", "iou3", "iou4"))
    again = eng.iou_features(2)                                   # the branch alone, from the arena
    assert torch.equal(again[0], out["iou3"]) and torch.equal(again[1], out["iou4"])
    for name in ("iou3", "iou4"):
        # the recorded sample of the reference map: entries at fixed flat indices and the map's largest magnitude
        mine = out[name].detach().double().cpu().reshape(-1)[torch.from_numpy(d[name + "_idx"]).long()]
        ref, ref_max = torch.from_numpy(d[name + "_val"]).double(), float(d[name + "_max"])
        err = float((mine - ref).abs().max() / ref_max)
        assert err < 1e-4, (name, err)
        # element-wise: entries above 1 % of the map's maximum to 2e-3 (two more 3x3 layers after layer2 / layer3)
        elem = float(((mine - ref).abs() / ref.abs().clamp(min=1e-2 * ref_max)).max())
        assert elem < 2e-3, (name, elem)
    eng.close()


def _inputs(net, seed, R):
    g = torch.Generator().manual_seed(seed)
    f3 = torch.relu(torch.randn(1, 256, 36, 36, generator=g))
    f4 = torch.relu(torch.randn(1, 256, 18, 18, generator=g))
    mod = [torch.randn(1, 256, 1, 1, generator=g).abs(), torch.randn(1, 256, 1, 1, generator=g).abs()]
    c = torch.tensor([120.0, 130.0]) + 30 * (torch.rand(R, 2, generator=g) - 0.5)
    sz = torch.tensor([70.0, 55.0]) * (0.6 + 0.8 * torch.rand(R, 2, generator=g))
    boxes = torch.cat([c - sz / 2, sz], 1).reshape(1, R, 4)
    return mod, [f3, f4], boxes


def _ref_iou_and_grad(net, mod, feat, boxes, device):
    netd = net.to(device)
    bb = boxes.clone().to(device).requires_grad_(True)
    iou = netd.bb_regressor.predict_iou([m.to(device) for m in mod], [f.to(device) for f in feat], bb)
    iou.backward(gradient=torch.ones_like(iou))
    return iou.detach().cpu(), bb.grad.detach().cpu()


def test_predict_iou_and_box_gradient_match_reference_autograd():
    from pytracking_b200.iou import IoUPredictor
    d = np.load(GOLDEN)
    pred = IoUPredictor(G.make_iou_state_dict())
    for seed, R in G.PREDICT:
        mod, feat, boxes = G.inputs(seed, R)
        iou, grad = pred.predict_iou([m.cuda() for m in mod], [f.cuda() for f in feat], boxes.cuda(), return_grad=True)
        ref_i, ref_g = torch.from_numpy(d["iou_%d" % seed]), torch.from_numpy(d["grad_%d" % seed])
        assert _rel(iou, ref_i) < 1e-4, (seed, _rel(iou, ref_i))
        assert _rel(grad, ref_g) < 1e-4, (seed, _rel(grad, ref_g))
        assert _rel_elem(iou, ref_i, 1e-3) < 1e-3
    pred.close()


@pytest.mark.parametrize("relative", [False, True])
def test_refinement_loop_matches_reference_optimize_boxes(relative):
    from pytracking_b200.iou import IoUPredictor
    d = np.load(GOLDEN)
    tag = "gpu_relative" if relative else "gpu_default"
    n_iter, step, _ = G.REFINE[tag]
    pred = IoUPredictor(G.make_iou_state_dict())
    mod, feat, boxes = G.inputs(G.REFINE_SEED, G.REFINE_R)
    ref_boxes, ref_iou = torch.from_numpy(d["boxes_" + tag]), torch.from_numpy(d["iou_" + tag])   # CPU reference loop (autograd)
    b, iou = pred.refine([m.cuda() for m in mod], [f.cuda() for f in feat], boxes.cuda(), n_iter, step, 1.0, relative)
    assert _rel(b, ref_boxes) < 1e-4, _rel(b, ref_boxes)
    assert float((b.cpu() - ref_boxes).abs().max()) < 2e-2            # pixels, after 5 / 10 ascent steps of O(1..10) px each
    assert _rel(iou, ref_iou) < 1e-3, _rel(iou, ref_iou)
    moved = float((ref_boxes - boxes.reshape(-1, 4)).abs().max())
    assert moved > 0.5, moved                                           # the loop really moved the boxes
    pred.close()


def test_plugin_predict_iou_seam_keeps_the_trackers_autograd_code_working():
    net = _setup()
    from pytracking_b200 import plugin
    mod, feat, boxes = _inputs(net, 11, 10)
    i_cpu, g_cpu = _ref_iou_and_grad(net, mod, feat, boxes, "cpu")
    plugin.install()
    plugin.stats.clear()
    try:
        i_eng, g_eng = _ref_iou_and_grad(net, mod, feat, boxes, "cuda")         # dimp.py:737-742 verbatim: predict_iou + backward
        assert plugin.stats.get("predict_iou", 0) == 1 and not plugin.stats.get("prroi_pooling_forward")
    finally:
        plugin.uninstall()
        net.cpu()
    assert _rel(i_eng, i_cpu) < 1e-4 and _rel(g_eng, g_cpu) < 1e-4, (_rel(i_eng, i_cpu), _rel(g_eng, g_cpu))
