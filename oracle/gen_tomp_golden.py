"""TEST INFRASTRUCTURE ONLY -- records what two UNMODIFIED reference ToMP modules compute on the CPU for seeded weights and inputs,
so that the library's box-regression tower and token assembly can be compared with them without the reference tree:
  * `DenseBoxRegressor.forward` (ltr/models/transformer/heads.py) with the weights of `make_tower_state_dict()`;
  * the token sequence `FilterPredictor.predict_cls_bbreg_filters_parallel` hands to its transformer (filter_predictor.py:92-135),
    intercepted at the transformer call, with the weights of `make_token_state_dict()`, 2 training frames + 1 test frame, with and
    without the test-frame embedding.

    PYTRACKING_REFERENCE=<pytracking checkout> python -m oracle.gen_tomp_golden

`tests/golden/tomp_heads.npz`: `tower` [1,4,18,18]; per `use_test` in (0, 1) a seeded sample of TOKEN_SAMPLE entries of the
[972, 2, 256] token tensor: `tokens<use_test>_idx` (flat indices), `tokens<use_test>_val`, `tokens<use_test>_max` (largest magnitude).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
TOKEN_SAMPLE = 4096
TOKEN_SHAPE = (972, 2, 256)


def _uniform(g, shape, fan_in):
    """torch's default Conv / Linear initialisation: U(-1/sqrt(fan_in), 1/sqrt(fan_in))"""
    b = fan_in ** -0.5
    return (2 * torch.rand(*shape, generator=g) - 1) * b


def make_tower_state_dict(seed=3):
    """DenseBoxRegressor(num_channels=256): default-initialised convolutions and projection, non-trivial GroupNorm affines and biases,
    the regression layer scaled by 0.3 (exp() of its output stays O(1))."""
    g = torch.Generator().manual_seed(seed)
    sd = {"linear.weight": _uniform(g, (256, 256), 256), "linear.bias": 0.1 * torch.randn(256, generator=g)}
    for i in (0, 3, 6, 9):
        sd["tower.%d.weight" % i] = _uniform(g, (256, 256, 3, 3), 256 * 9)
        sd["tower.%d.bias" % i] = 0.1 * torch.randn(256, generator=g)
        sd["tower.%d.weight" % (i + 1)] = 0.5 + torch.rand(256, generator=g)          # GroupNorm
        sd["tower.%d.bias" % (i + 1)] = 0.1 * torch.randn(256, generator=g)
    sd["bbreg_layer.weight"] = 0.3 * _uniform(g, (4, 256, 3, 3), 256 * 9)
    sd["bbreg_layer.bias"] = 0.1 * torch.randn(4, generator=g)
    return sd


def tower_inputs():
    """-> feat [1,1,256,18,18], filter [1,256,1,1]"""
    g = torch.Generator().manual_seed(4)
    return torch.randn(1, 1, 256, 18, 18, generator=g) * 0.3, torch.randn(1, 256, 1, 1, generator=g) * 0.2


def make_token_state_dict(use_test, seed=7):
    """FilterPredictor(feature_sz=18, use_test_frame_encoding=use_test): the box-encoding MLP (default-initialised 1x1 convolutions,
    non-trivial BatchNorm statistics and affines) and the query embeddings (standard normal, as nn.Embedding)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for i, (cout, cin) in ((0, (64, 4)), (3, (256, 64)), (6, (256, 256))):
        sd["box_encoding.%d.weight" % i] = _uniform(g, (cout, cin, 1), cin)
        sd["box_encoding.%d.bias" % i] = _uniform(g, (cout,), cin)
        if i < 6:
            sd["box_encoding.%d.running_mean" % (i + 1)] = 0.1 * torch.randn(cout, generator=g)
            sd["box_encoding.%d.running_var" % (i + 1)] = 0.6 + 0.8 * torch.rand(cout, generator=g)
            sd["box_encoding.%d.weight" % (i + 1)] = 0.8 + 0.4 * torch.rand(cout, generator=g)
            sd["box_encoding.%d.bias" % (i + 1)] = 0.1 * torch.randn(cout, generator=g)
    sd["query_embed_fg.weight"] = torch.randn(1, 256, generator=g)
    sd["query_embed_test.weight"] = torch.randn(1, 256, generator=g)
    sd["query_embed_fg_decoder.weight"] = sd["query_embed_fg.weight"]
    if not use_test:
        del sd["query_embed_test.weight"]
    return sd


def token_inputs():
    """-> train_feat [2,1,256,18,18], test_feat [1,1,256,18,18], label [2,1,18,18], ltrb [2,1,4,18,18]"""
    g = torch.Generator().manual_seed(8)
    return (torch.randn(2, 1, 256, 18, 18, generator=g), torch.randn(1, 1, 256, 18, 18, generator=g), torch.rand(2, 1, 18, 18, generator=g),
            torch.rand(2, 1, 4, 18, 18, generator=g))


def record():
    from oracle import ref_shims
    ref_shims.install()
    import ltr.models.transformer.filter_predictor as fp
    import ltr.models.transformer.heads as heads
    out = {}
    m = heads.DenseBoxRegressor(num_channels=256).eval()
    m.load_state_dict(make_tower_state_dict())
    feat, filt = tower_inputs()
    with torch.no_grad():
        out["tower"] = m(feat, filt)[0].numpy()                                      # [1,4,18,18]
    rng = np.random.RandomState(0)
    for use_test in (0, 1):
        captured = {}

        class FakeTransformer(torch.nn.Module):
            d_model = 256

            def forward(self, feat, mask=None, query_embed=None, pos_embed=None):
                captured["feat"], captured["mask"] = feat.clone(), mask
                return torch.zeros(1, 1, feat.shape[1], 256), torch.zeros_like(feat)
        m = fp.FilterPredictor(FakeTransformer(), feature_sz=18, use_test_frame_encoding=bool(use_test)).eval()
        missing, unexpected = m.load_state_dict(make_token_state_dict(use_test), strict=False)
        assert not unexpected and all("num_batches" in k for k in missing), (missing, unexpected)
        train_feat, test_feat, label, ltrb = token_inputs()
        with torch.no_grad():
            m.predict_cls_bbreg_filters_parallel(train_feat, test_feat, label, 1, ltrb)
        ref = captured["feat"].numpy()
        assert ref.shape == TOKEN_SHAPE, ref.shape
        # the mask layout the library's token builder assumes
        assert captured["mask"].shape == (2, 972) and int(captured["mask"][1].sum()) == 324 and int(captured["mask"][0].sum()) == 0
        flat = ref.reshape(-1)
        idx = np.sort(rng.choice(flat.size, TOKEN_SAMPLE, replace=False)).astype(np.int32)
        out["tokens%d_idx" % use_test], out["tokens%d_val" % use_test] = idx, flat[idx]
        out["tokens%d_max" % use_test] = np.float64(np.abs(flat).max())
    path = os.path.join(GOLDEN, "tomp_heads.npz")
    np.savez_compressed(path, **out)
    print(path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    record()
