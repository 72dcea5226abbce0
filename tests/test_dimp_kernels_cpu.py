"""The two device kernels of the whole-frame DiMP call (csrc/dimp_tracker_kernels.cuh: the crop sampler of SURVEY 8 row f2 and the
localisation kernel of row f3) executed ON THE CPU: the same source file the CUDA build compiles, built as host code under
tests/cpu_emul/cuda_shim.h (tests/cpu_emul/dimp_emul.cpp; -ffp-contract=off so that the explicitly rounded operations stay single
operations).  These are the CPU-tier counterparts of the `-m gpu` tests in tests/test_tracker_gpu.py:
  * sample_patch_kernel against torch's CPU bilinear resampling of the reference's `sample_patch` -- bit-exact, nine geometries
    (decimation factors 1-4, crops hanging over every border, 4K frames, the windowed first-frame crop);
  * localize_kernel against the decisions recorded from the UNMODIFIED reference tracker (320 frames of two trajectories, every flag)
    and against the reference's own `localize_target` / `localize_advanced` on random score maps with ties.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    out = os.path.join(str(tmp_path_factory.mktemp("dimp_emul")), "libdimp_emul.so")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-pthread", "-shared", "-fPIC", "-ffp-contract=off", "-fno-gnu-unique", "-Wno-unknown-pragmas",
                    os.path.join(ROOT, "tests", "cpu_emul", "dimp_emul.cpp"), "-o", out], check=True, capture_output=True)
    return C.CDLL(out)


def _params(**kw):
    from tracker_cases import DIMP50
    from pytracking_b200.tracker import make_params
    return make_params(**dict(DIMP50, **kw))


def test_sample_patch_kernel_source_bit_exact_vs_torch_cpu(emul):
    from oracle import preprocessing_ref as R
    from pytracking_b200.tracker import HostLogic
    rng = np.random.RandomState(0)
    cases = [(480, 640, [300, 200, 80, 60], 2), (480, 640, [2, 3, 90, 70], None), (480, 640, [600, 440, 80, 60], None),
             (720, 1280, [500, 300, 400, 300], None), (1080, 1920, [1500, 900, 410, 170], 2), (240, 320, [150, 100, 9, 9], None),
             (480, 640, [100, 100, 3, 2], None), (2160, 3840, [1000, 1000, 1500, 900], None), (300, 300, [100, 100, 57.6, 57.6], None)]
    for (H, W, bb, ef) in cases:
        img = np.ascontiguousarray(rng.randint(0, 256, (H, W, 3)).astype(np.uint8))
        hl = HostLogic(_params(augmentation_expansion_factor=ef))
        g_init, _ = hl.init_state(H, W, bb)
        st = hl.state()
        im = R.numpy_to_torch(img)
        sz = torch.tensor([288.0, 288.0])
        for which in ("init", "frame"):
            if which == "init":
                g = g_init
                ref = R.sample_init_patch(im, torch.tensor([st[0], st[1]]).round(), torch.tensor(st[4]), sz, ef)
            else:
                g = hl.plan_crop()
                ref, coord = R.sample_patch(im, torch.tensor([st[0], st[1]]), torch.tensor(st[4]) * sz, sz)
                assert np.array_equal(np.array(g.coord, dtype=np.float32), coord.numpy().reshape(4))
            out = np.empty((3, 288, 288), np.float32)
            assert emul.dimp_emul_sample_patch(img.ctypes.data_as(C.c_void_p), H, W, C.byref(g), 288, 288, out.ctypes.data_as(C.c_void_p)) == 0
            diff = torch.from_numpy(out) != ref[0]
            assert not diff.any(), ((H, W, bb, which), int(diff.sum()), float((torch.from_numpy(out) - ref[0]).abs().max()), g.df, g.in_h)
        hl.close()


def _run_localize(emul, scores, params, neigh, pv):
    from pytracking_b200 import _lib
    s = np.ascontiguousarray(scores.numpy(), dtype=np.float32)
    n = np.ascontiguousarray(neigh, dtype=np.float32)
    p = np.ascontiguousarray(pv, dtype=np.float32)
    res = _lib.LocResult()
    assert emul.dimp_emul_localize(s.ctypes.data_as(C.c_void_p), s.shape[0], s.shape[1], s.shape[2], C.byref(params),
                                   n.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), C.byref(res)) == 0
    return res


def test_localize_kernel_source_matches_recorded_reference_trajectories(emul):
    from tracker_cases import OVERRIDES, _loc
    from pytracking_b200.tracker import HostLogic
    flags = set()
    for name in ("cfg2", "stress"):
        d = np.load(os.path.join(GOLDEN, "dimp_host_%s.npz" % name))
        params = _params(**OVERRIDES[name])
        hl = HostLogic(params)
        H, W = [int(v) for v in d["image_hw"]]
        hl.adopt(H, W, d["init_state"], d["init_sw"], d["init_counts"][0], d["init_counts"][1])
        for t in range(len(d["flag"])):
            g = hl.plan_crop()
            st = hl.state()
            neigh = [np.float32(np.float32(params.target_neighborhood_scale) * (st[2 + i] / np.float32(g.sample_scale))) * np.float32(18.0 / 288.0) for i in range(2)]
            pv = [(st[i] - np.float32(g.sample_pos[i])) / (np.float32(16.0) * np.float32(g.sample_scale)) for i in range(2)]
            out = _run_localize(emul, torch.from_numpy(d["scores"][t])[None], params, [neigh], [pv])
            assert out.flag == d["flag"][t], (name, t, out.flag, d["flag"][t])
            assert (out.r1, out.c1) == (int(d["m1"][t, 1]), int(d["m1"][t, 2])) and np.float32(out.score1) == np.float32(d["m1"][t, 0])
            if d["m2"][t, 1] >= 0:
                assert (out.r2, out.c2) == (int(d["m2"][t, 1]), int(d["m2"][t, 2])) and np.float32(out.score2) == np.float32(d["m2"][t, 0])
            assert out.use_second == d["use2"][t]
            flags.add(int(out.flag))
            hl.commit(g, _loc(d, t))
        hl.close()
    assert flags >= {1, 2, 3, 4}, flags                       # normal, hard negative, uncertain, not found all occur in the recordings


def test_localize_kernel_source_matches_reference_code_on_random_maps(emul):
    """Against the reference `DiMP.localize_target` on seeded random maps (recorded by oracle/gen_localize_golden.py)."""
    from oracle.gen_localize_golden import cases
    from pytracking_b200.tracker import FLAGS
    d = np.load(os.path.join(GOLDEN, "localize_random.npz"))
    img_support_sz, out_sz = torch.Tensor([288, 288]), torch.Tensor([18, 18])
    seen = set()
    for trial, (kw, scores, target_sz, sample_pos, sample_scales, pos) in enumerate(cases(200)):
        params = _params(**kw)
        S = scores.shape[0]
        neigh = [(2.2 * (target_sz / sample_scales[s]) * (out_sz / img_support_sz)).numpy() for s in range(S)]
        pv = [((pos - sample_pos[s]) / ((img_support_sz / out_sz) * sample_scales[s])).numpy() for s in range(S)]
        out = _run_localize(emul, scores, params, neigh, pv)
        assert out.flag == d["flag"][trial], (trial, FLAGS[out.flag], FLAGS[d["flag"][trial]])
        assert out.scale_ind == d["scale_ind"][trial]
        cell = (out.r2, out.c2) if out.use_second else (out.r1, out.c1)
        mine = (torch.Tensor(cell) - 9) * (img_support_sz / out_sz) * sample_scales[out.scale_ind]
        assert torch.equal(mine, torch.from_numpy(d["tv"][trial])), (trial, mine, d["tv"][trial])
        seen.add((FLAGS[out.flag], out.use_second))
    assert {("normal", 0), ("hard_negative", 0), ("hard_negative", 1), ("uncertain", 0), ("not_found", 0), (None, 0)} <= seen, seen
