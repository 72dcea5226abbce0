"""TEST INFRASTRUCTURE ONLY -- records what the UNMODIFIED reference IoUNet (`AtomIoUNet.get_iou_feat`, `predict_iou` with torch
autograd for the box gradient, ltr/models/bbreg/atom_iou_net.py) and the DiMP refinement loops (`DiMP.optimize_boxes` default /
relative, pytracking/tracker/dimp/dimp.py) compute on the CPU, PrRoIPool from the oracle's CPU restatement, for the seeded IoUNet
weights of `make_iou_state_dict()` and the seeded inputs of `inputs()`.  The IoU tests compare the library with these records.

    PYTRACKING_REFERENCE=<pytracking checkout> python -m oracle.gen_iou_golden

`tests/golden/iou.npz`:
  iou_<seed>, grad_<seed>          predict_iou and d(sum iou)/d(box) for the PREDICT cases
  boxes_<tag>, iou_<tag>           optimize_boxes output for the REFINE cases
  iou3_idx, iou3_val, iou3_max     get_iou_feat on synth.make_crop(3, 2, 288): a seeded sample of FEAT_SAMPLE entries of each map
  iou4_idx, iou4_val, iou4_max     (flat indices, values) and the map's largest magnitude
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

# DiMP-50's IoUNet: input_dim (512, 1024), pred_input_dim (256, 256), pred_inter_dim (256, 256)
CONV_BN = [("conv3_1r", 128, 512, 3), ("conv3_1t", 256, 512, 3), ("conv3_2t", 256, 256, 3), ("fc3_1r", 256, 128, 3),
           ("conv4_1r", 256, 1024, 3), ("conv4_1t", 256, 1024, 3), ("conv4_2t", 256, 256, 3), ("fc34_3r", 256, 512, 1),
           ("fc34_4r", 256, 512, 1)]
LINEAR_BN = [("fc3_rt", 256, 256 * 5 * 5), ("fc4_rt", 256, 256 * 3 * 3)]
PREDICT = ((0, 10), (1, 1), (2, 16))                 # (input seed, boxes)
REFINE = {"cpu_default": (3, 1.0, False), "cpu_relative": (4, 5e-3, True),        # (iterations, step length, relative)
          "gpu_default": (5, 1.0, False), "gpu_relative": (10, 2.5e-3, True)}
REFINE_SEED, REFINE_R = 7, 10
FEAT_SAMPLE = 4096


def make_iou_state_dict(seed=0):
    """bb_regressor.* of a DiMP-50 net: the reference constructor's initialisation (Kaiming-normal fan-in weights, zero biases,
    BatchNorm weights uniform in [0, 1)) drawn from a seeded generator, non-trivial BatchNorm statistics and biases, and the last
    layer scaled so that the box gradients are O(1e-2) and the refinement loops move boxes by pixels, as with a trained net."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def kaiming(*shape):
        fan_in = int(np.prod(shape[1:]))
        return torch.randn(*shape, generator=g) * (2.0 / fan_in) ** 0.5

    def bn(prefix, c):
        sd[prefix + ".weight"] = torch.rand(c, generator=g)
        sd[prefix + ".bias"] = 0.05 * torch.randn(c, generator=g)
        sd[prefix + ".running_mean"] = 0.05 * torch.randn(c, generator=g)
        sd[prefix + ".running_var"] = 0.7 + 0.6 * torch.rand(c, generator=g)

    for name, cout, cin, k in CONV_BN:
        sd["bb_regressor.%s.0.weight" % name] = kaiming(cout, cin, k, k)
        sd["bb_regressor.%s.0.bias" % name] = torch.zeros(cout)
        bn("bb_regressor.%s.1" % name, cout)
    for name, cout, cin in LINEAR_BN:
        sd["bb_regressor.%s.linear.weight" % name] = kaiming(cout, cin)
        sd["bb_regressor.%s.linear.bias" % name] = torch.zeros(cout)
        bn("bb_regressor.%s.bn" % name, cout)
    sd["bb_regressor.iou_predictor.weight"] = 0.4 * kaiming(1, 512)
    sd["bb_regressor.iou_predictor.bias"] = torch.zeros(1)
    return sd


def make_dimp_iou_state_dict():
    """The DiMP-50 state_dict of the IoU tests: the engine tests' seeded backbone / classifier plus make_iou_state_dict()."""
    from pytracking_b200 import synth
    sd = synth.make_dimp_state_dict("resnet50", seed=0, lut_seed=3)
    sd.update(make_iou_state_dict())
    return sd


def inputs(seed, R):
    """-> (modulation [2 x (1,256,1,1)], IoU features [(1,256,36,36), (1,256,18,18)], boxes (1,R,4) as x,y,w,h)"""
    g = torch.Generator().manual_seed(seed)
    f3 = torch.relu(torch.randn(1, 256, 36, 36, generator=g))
    f4 = torch.relu(torch.randn(1, 256, 18, 18, generator=g))
    mod = [torch.randn(1, 256, 1, 1, generator=g).abs(), torch.randn(1, 256, 1, 1, generator=g).abs()]
    c = torch.tensor([120.0, 130.0]) + 30 * (torch.rand(R, 2, generator=g) - 0.5)
    sz = torch.tensor([70.0, 55.0]) * (0.6 + 0.8 * torch.rand(R, 2, generator=g))
    return mod, [f3, f4], torch.cat([c - sz / 2, sz], 1).reshape(1, R, 4)


def crop_input():
    from pytracking_b200 import synth
    return synth.make_crop(3, 2, 288)


def record():
    from oracle import ref_shims
    ref_shims.install()
    from baseline import ref_tracker
    from pytracking.libs import TensorList
    from pytracking.tracker.dimp.dimp import DiMP
    from pytracking.utils import TrackerParams
    net = ref_tracker.build_dimp_net("resnet50", seed=0)
    missing, unexpected = net.load_state_dict(make_dimp_iou_state_dict(), strict=False)
    assert not unexpected and not [k for k in missing if k.startswith("bb_regressor.") and "num_batches" not in k], missing
    out = {}
    for seed, R in PREDICT:
        mod, feat, boxes = inputs(seed, R)
        bb = boxes.clone().requires_grad_(True)
        iou = net.bb_regressor.predict_iou(mod, feat, bb)                 # dimp.py:737-742: predict_iou + backward
        iou.backward(gradient=torch.ones_like(iou))
        out["iou_%d" % seed], out["grad_%d" % seed] = iou.detach().reshape(-1).numpy(), bb.grad.reshape(-1, 4).numpy()
    mod, feat, boxes = inputs(REFINE_SEED, REFINE_R)
    for tag, (n_iter, step, relative) in REFINE.items():
        p = TrackerParams()
        p.device = "cpu"
        p.box_refinement_iter, p.box_refinement_step_length, p.box_refinement_step_decay = n_iter, step, 1
        p.box_refinement_space = "relative" if relative else "default"
        trk = DiMP.__new__(DiMP)
        trk.params = p
        trk.net = type("N", (), {"bb_regressor": net.bb_regressor})()
        trk.iou_modulation = TensorList(mod)
        b, i = trk.optimize_boxes(TensorList(feat), boxes.reshape(-1, 4).clone())
        out["boxes_" + tag], out["iou_" + tag] = b.detach().numpy(), i.detach().numpy()
    im = crop_input()
    with torch.no_grad():
        x = (im / 255 - torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)) / torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
        bf = net.extract_backbone_features(x)
        c3, c4 = net.bb_regressor.get_iou_feat([bf["layer2"], bf["layer3"]])
    g = np.random.RandomState(0)
    for name, c in (("iou3", c3), ("iou4", c4)):
        flat = c.reshape(-1).numpy()
        idx = np.sort(g.choice(flat.size, FEAT_SAMPLE, replace=False)).astype(np.int32)
        out[name + "_idx"], out[name + "_val"], out[name + "_max"] = idx, flat[idx], np.float64(np.abs(flat).max())
    path = os.path.join(GOLDEN, "iou.npz")
    np.savez_compressed(path, **out)
    print(path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    record()
