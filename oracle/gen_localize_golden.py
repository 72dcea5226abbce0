"""TEST INFRASTRUCTURE ONLY -- records what the UNMODIFIED reference `DiMP.localize_target` (dimp.py, advanced and simple
localisation) returns on seeded random score maps that reach every branch of its decision tree, so that the localisation kernel
can be checked against it without the reference tree.

    PYTRACKING_REFERENCE=<pytracking checkout> python -m oracle.gen_localize_golden

`tests/golden/localize_random.npz`, one row per case of `cases()`: the translation vector `tv` [N,2], `scale_ind` [N] and the
flag code `flag` [N] (None 0, normal 1, hard_negative 2, uncertain 3, not_found 4, as in gen_host_logic_golden.py).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
FLAG = {None: 0, "normal": 1, "hard_negative": 2, "uncertain": 3, "not_found": 4}
N_CASES = 400


def cases(n=N_CASES):
    """Seeded localisation cases: (params overrides, scores [S,19,19], target_sz [2], sample_pos [S,2], sample_scales [S], pos [2])."""
    g = torch.Generator().manual_seed(0)
    for trial in range(n):
        adv = trial % 10 != 9
        S = 1 + trial % 3
        kw = dict(advanced_localization=adv, target_not_found_threshold=0.2, uncertain_threshold=0.25 if trial % 4 == 0 else -float("inf"),
                  hard_sample_threshold=0.3 if trial % 5 == 0 else -float("inf"), distractor_threshold=0.8, hard_negative_threshold=0.5,
                  dispalcement_scale=0.3 + 0.5 * (trial % 2))
        scores = 0.1 * torch.rand(S, 19, 19, generator=g)
        for s in range(S):
            for _ in range(1 + trial % 3):               # a few peaks of comparable height
                r, c = [int(v) for v in torch.randint(0, 19, (2,), generator=g)]
                scores[s, r, c] = 0.15 + 0.6 * float(torch.rand(1, generator=g))
        if trial % 7 == 0:                               # exact ties: the arg-max order must follow dcf.max2d
            scores[0, 3, 11] = scores[0, 12, 4] = scores.max() + 0.1
        target_sz = torch.Tensor([60, 80]) * (0.5 + float(torch.rand(1, generator=g)))
        sample_scales = 1.0 + 0.5 * torch.rand(S, generator=g)
        sample_pos = torch.Tensor([[240, 320]]).repeat(S, 1) + torch.rand(S, 2, generator=g)
        pos = sample_pos[0] + 40 * (torch.rand(2, generator=g) - 0.5)
        yield kw, scores, target_sz, sample_pos, sample_scales, pos


def record():
    from oracle import ref_shims
    ref_shims.install(prroi_cpu=False)
    from pytracking.tracker.dimp.dimp import DiMP
    from pytracking.utils import TrackerParams
    tvs, inds, flags = [], [], []
    for kw, scores, target_sz, sample_pos, sample_scales, pos in cases():
        trk = DiMP.__new__(DiMP)
        p = TrackerParams()
        for k, v in kw.items():
            setattr(p, k, v)
        p.target_neighborhood_scale = 2.2
        trk.params = p
        trk.output_window = None
        trk.kernel_size = torch.Tensor([4, 4])
        trk.img_support_sz = torch.Tensor([288, 288])
        trk.target_sz = target_sz
        trk.pos = pos
        tv, scale_ind, _, flag = trk.localize_target(scores.clone().unsqueeze(1), sample_pos, sample_scales)
        tvs.append(tv.numpy().astype(np.float32))
        inds.append(int(scale_ind))
        flags.append(FLAG[flag])
    out = os.path.join(GOLDEN, "localize_random.npz")
    np.savez_compressed(out, tv=np.stack(tvs), scale_ind=np.array(inds, dtype=np.int32), flag=np.array(flags, dtype=np.int32))
    print(out, np.bincount(flags))


if __name__ == "__main__":
    record()
