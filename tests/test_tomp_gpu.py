"""-m gpu parity tests of the ToMP row (SURVEY.md 8(a) T1) beyond `Transformer.forward` (tests/test_gpu_parity.py): the
`DenseBoxRegressor` tower and the token assembly on the engine against what the UNMODIFIED reference modules computed on PyTorch-CPU
for the same seeded weights and inputs (tests/golden/tomp_heads.npz, oracle/gen_tomp_golden.py), and the UNMODIFIED reference ToMP-101
tracker (pytracking/tracker/tomp/tomp.py) above the engine against the same tracker on stock PyTorch-CUDA (TF32 off) when a pytracking
checkout is importable."""
import os

import numpy as np
import pytest
import torch

from oracle import gen_tomp_golden as G

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "tomp_heads.npz")


def _ref():
    from baseline import ref_env
    if not ref_env.reference_available():
        pytest.skip("reference tree not staged (baseline/_ref)")
    from oracle import ref_shims
    ref_shims.install()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def test_box_regression_tower_matches_reference_module():
    from pytracking_b200.transformer_engine import BoxTower
    sd = G.make_tower_state_dict()
    feat, filt = G.tower_inputs()
    ref_cpu = torch.from_numpy(np.load(GOLDEN)["tower"])                      # [1,4,18,18]
    with torch.no_grad():
        fp = torch.nn.functional.linear(filt.cuda().reshape(-1, 256), sd["linear.weight"].cuda(), sd["linear.bias"].cuda()).reshape(1, 256, 1, 1)
        att = (feat.cuda()[0] * fp).sum(1)                                     # the 1x1 correlation
    tw = BoxTower(sd, 18, 18, max_batch=2)
    out = tw.forward(feat.cuda()[0], att)
    assert out.shape == (1, 4, 18, 18)
    assert _rel(out, ref_cpu) < 1e-4, _rel(out, ref_cpu)
    assert abs(tw.flops / 2 / 1e6 - (4 * 191.1 + 191.1 * 4 / 256)) < 2.0      # 9 * 256 * 256 * 324 = 191.1 MMAC per 256 -> 256 layer at 18x18
    two = tw.forward(torch.cat([feat.cuda()[0], feat.cuda()[0]]), torch.cat([att, att]))
    # the two samples of one launch are bitwise identical; a batch-1 launch may pick another split-K factor (different summation order)
    assert torch.equal(two[0], two[1]) and _rel(two[0], out[0]) < 1e-5
    tw.close()


def test_reference_tomp_tracker_above_engine():
    """ToMP-101 (parameter/tomp/tomp101.py, random-init tompnet101): every frame's backbone + head feature, transformer, classifier
    correlation and box-regression tower are served by the library; boxes (floating-point ltrb regression outputs) agree with the stock
    PyTorch-CUDA run to 1e-2 px while the trajectories coincide."""
    _ref()
    from baseline import ref_tracker
    from pytracking_b200 import plugin, synth
    n = 12
    frames, bb = synth.make_sequence(0, num_frames=n)
    plugin.install()
    plugin.stats.clear()
    try:
        eng = ref_tracker.run_sequence(ref_tracker.build_tomp("cuda"), frames, bb)
        stats = dict(plugin.stats)
    finally:
        plugin.uninstall()
    stock = ref_tracker.run_sequence(ref_tracker.build_tomp("cuda"), frames, bb)
    for seam in ("extract_backbone", "Head.extract_head_feat", "FilterPredictor.predict_cls_bbreg_filters_parallel", "Transformer.forward",
                 "apply_filter", "DenseBoxRegressor.forward", "max2d"):
        assert stats.get(seam, 0) >= n, (seam, stats)
    d = np.abs(eng["target_bbox"] - stock["target_bbox"]).max(axis=1)
    print("ToMP-101 above the engine vs stock PyTorch-CUDA, max abs box difference per frame [px]:", np.round(d, 5).tolist())
    assert d[:3].max() < 1e-2, d


def test_token_assembly_matches_reference_filter_predictor():
    """`b200trk_tomp_tokens` against the reference's own token construction (filter_predictor.py:92-135), intercepted at the
    transformer call, for 2 training frames + 1 test frame; with and without the test-frame embedding."""
    from pytracking_b200.transformer_engine import TokenBuilder
    d = np.load(GOLDEN)
    train_feat, test_feat, label, ltrb = G.token_inputs()
    for use_test in (False, True):
        tb = TokenBuilder(G.make_token_state_dict(use_test))
        out = tb.build(train_feat[:, 0].cuda(), test_feat[:, 0].cuda(), label[:, 0].cuda(), ltrb[:, 0].cuda(), B=2, use_test_token=use_test)
        assert tuple(out.shape) == G.TOKEN_SHAPE
        # the recorded sample of the reference tokens: entries at fixed flat indices and the tensor's largest magnitude
        k = "tokens%d" % use_test
        mine = out.detach().double().cpu().reshape(-1)[torch.from_numpy(d[k + "_idx"]).long()]
        err = float((mine - torch.from_numpy(d[k + "_val"]).double()).abs().max() / float(d[k + "_max"]))
        assert err < 1e-5, (use_test, err)
