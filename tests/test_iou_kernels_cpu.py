"""IoUNet box refinement (SURVEY 8 row f1) executed ON THE CPU: the kernels of csrc/iou_refine_kernels.cuh + csrc/prroi_kernels.cuh -- the
same source files the CUDA build compiles (`cuobjdump -sass` identical before and after they moved into headers) -- built as host code under
tests/cpu_emul/cuda_shim.h and run in the launch sequence of `b200trk_iou_predict` / `b200trk_iou_refine` (csrc/iou_refine.cu), against
what the UNMODIFIED reference computed for the same seeded weights and inputs (tests/golden/iou.npz, oracle/gen_iou_golden.py):
`AtomIoUNet.predict_iou` with torch autograd for the box gradient (ltr/models/bbreg/atom_iou_net.py:96-136) and
`DiMP.optimize_boxes_default / _relative` (pytracking/tracker/dimp/dimp.py:725-793), PrRoIPool from the oracle's CPU restatement.
CPU-tier counterparts of tests/test_iou_gpu.py."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import gen_iou_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    out = os.path.join(str(tmp_path_factory.mktemp("iou_emul")), "libiou_emul.so")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-pthread", "-shared", "-fPIC", "-ffp-contract=off", "-fno-gnu-unique", "-Wno-unknown-pragmas",
                    os.path.join(ROOT, "tests", "cpu_emul", "iou_emul.cpp"), "-o", out], check=True, capture_output=True)
    return C.CDLL(out)


@pytest.fixture(scope="module")
def sd():
    return G.make_iou_state_dict()


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "iou.npz"))


def _rel(a, b):
    a, b = torch.as_tensor(a).detach().double(), torch.as_tensor(b).detach().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _run(emul, sd, mod, feat, boxes, num_iter=0, step=1.0, decay=1.0, relative=False, want_grad=True):
    from pytracking_b200 import _lib
    keep = []

    def hp(key):
        t = sd["bb_regressor." + key].detach().float().contiguous()
        keep.append(t)
        return t

    def block(name):
        w = hp(name + ".linear.weight")
        return _lib.LinearBlock(w.data_ptr(), hp(name + ".linear.bias").data_ptr(), hp(name + ".bn.weight").data_ptr(), hp(name + ".bn.bias").data_ptr(),
                                hp(name + ".bn.running_mean").data_ptr(), hp(name + ".bn.running_var").data_ptr()), w.shape
    b3, s3 = block("fc3_rt")
    b4, s4 = block("fc4_rt")
    wp, bp = hp("iou_predictor.weight"), hp("iou_predictor.bias")
    C3 = C4 = 256
    P3, P4 = int(round((s3[1] // C3) ** 0.5)), int(round((s4[1] // C4) ** 0.5))
    p = lambda t: C.c_void_p(t.data_ptr())
    m3, m4 = mod[0].reshape(-1).contiguous(), mod[1].reshape(-1).contiguous()
    f3, f4 = feat[0].contiguous(), feat[1].contiguous()
    bx = boxes.reshape(-1, 4).clone().contiguous()
    R = bx.shape[0]
    iou, grad = torch.full((R,), float("nan")), torch.full((R, 4), float("nan"))
    rc = emul.iou_emul_run(C.byref(b3), C.byref(b4), p(wp), p(bp), C3, P3, C4, P4, int(s3[0]), int(s4[0]), p(m3), p(m4), p(f3), 36, 36, p(f4), 18, 18, p(bx), R,
                           num_iter, C.c_float(step), C.c_float(decay), int(relative), p(iou), p(grad) if (want_grad and num_iter == 0) else None)
    assert rc == 0
    return iou, grad, bx


@pytest.mark.parametrize("seed,R", G.PREDICT)
def test_predict_iou_and_box_gradient_kernel_sources_vs_reference_autograd(emul, sd, gold, seed, R):
    mod, feat, boxes = G.inputs(seed, R)
    ref_iou, ref_grad = torch.from_numpy(gold["iou_%d" % seed]), torch.from_numpy(gold["grad_%d" % seed])
    iou, grad, _ = _run(emul, sd, mod, feat, boxes)
    assert _rel(iou, ref_iou) < 1e-4 and _rel(grad, ref_grad) < 1e-4, (_rel(iou, ref_iou), _rel(grad, ref_grad))


@pytest.mark.parametrize("relative", [False, True])
def test_refinement_loop_kernel_sources_vs_reference_optimize_boxes(emul, sd, gold, relative):
    tag = "cpu_relative" if relative else "cpu_default"   # the tracker uses 10 / 5 iterations (tests/test_iou_gpu.py does too); fewer here for time
    n_iter, step, _ = G.REFINE[tag]
    mod, feat, boxes = G.inputs(G.REFINE_SEED, G.REFINE_R)
    ref_boxes, ref_iou = torch.from_numpy(gold["boxes_" + tag]), torch.from_numpy(gold["iou_" + tag])
    iou, _, b = _run(emul, sd, mod, feat, boxes, n_iter, step, 1.0, relative)
    assert _rel(b, ref_boxes) < 1e-4 and float((b - ref_boxes).abs().max()) < 2e-2, (_rel(b, ref_boxes), float((b - ref_boxes).abs().max()))
    assert _rel(iou, ref_iou) < 1e-3
    assert float((ref_boxes - boxes.reshape(-1, 4)).abs().max()) > 0.5                              # the loop really moved the boxes
