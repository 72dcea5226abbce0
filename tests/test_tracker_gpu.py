"""-m gpu parity tests of the whole-frame path (SURVEY.md 8(f) rows f2, f3 and the drop-in boundary 8(b)):

  * the crop kernel against torch's own CPU bilinear resampling of the reference's `sample_patch` -- bit-exact;
  * the localisation kernel against what the UNMODIFIED reference `DiMP.localize_advanced` / `localize_target` returned on seeded
    random score maps that hit every branch (tests/golden/localize_random.npz), and against the recorded trajectories -- cells and
    flags identical;
  * the native tracker (`b200trk_dimp_track_host`: uint8 frame in, box out) against the recorded reference run and, in lock-step,
    against the reference tracker running above the engine -- `target_bbox` bit-identical, score maps <= 1e-4;
  * the UNMODIFIED reference DiMP tracker above the engine (`plugin.install()`) against the same tracker on stock PyTorch-CUDA
    (TF32 off) and stock PyTorch-CPU -- `target_bbox` bit-identical.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _ref():
    from baseline import ref_env
    if not ref_env.reference_available():
        pytest.skip("reference tree not staged (baseline/_ref)")
    from oracle import ref_shims
    ref_shims.install()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _params(**kw):
    from tracker_cases import DIMP50
    from pytracking_b200.tracker import make_params
    return make_params(**dict(DIMP50, **kw))


# ---------------------------------------------------------------------------------------------------------------------------
def test_sample_patch_kernel_bit_exact_vs_torch_cpu():
    from oracle import preprocessing_ref as R
    from pytracking_b200 import _lib
    from pytracking_b200.tracker import HostLogic
    L = _lib.lib()
    rng = np.random.RandomState(0)
    cases = [(480, 640, [300, 200, 80, 60], 2), (480, 640, [2, 3, 90, 70], None), (480, 640, [600, 440, 80, 60], None),
             (720, 1280, [500, 300, 400, 300], None), (1080, 1920, [1500, 900, 410, 170], 2), (240, 320, [150, 100, 9, 9], None),
             (480, 640, [100, 100, 3, 2], None), (2160, 3840, [1000, 1000, 1500, 900], None), (300, 300, [100, 100, 57.6, 57.6], None)]
    torch.set_num_threads(8)
    for (H, W, bb, ef) in cases:
        img = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
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
            out = torch.empty(3, 288, 288, device="cuda")
            _lib.check(L.b200trk_sample_patch(C.c_void_p(torch.from_numpy(img).cuda().data_ptr()), H, W, C.byref(g), 288, 288,
                                              C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "sample_patch")
            diff = (out.cpu() != ref[0])
            assert not diff.any(), ((H, W, bb, which), int(diff.sum()), float((out.cpu() - ref[0]).abs().max()), g.df, g.in_h)
        hl.close()


def _run_localize(scores, params, neigh, pv):
    from pytracking_b200 import _lib
    L = _lib.lib()
    s = scores.cuda().contiguous()
    res = torch.zeros(16, dtype=torch.int32, device="cuda")
    n = np.ascontiguousarray(neigh, dtype=np.float32)
    p = np.ascontiguousarray(pv, dtype=np.float32)
    _lib.check(L.b200trk_dimp_localize(C.c_void_p(s.data_ptr()), s.shape[0], s.shape[1], s.shape[2], C.byref(params),
                                       n.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), C.c_void_p(res.data_ptr()),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)), "dimp_localize")
    raw = res.cpu().numpy()
    out = _lib.LocResult.from_buffer_copy(raw.tobytes())
    return out


def test_localize_kernel_matches_recorded_reference_trajectories():
    from tracker_cases import OVERRIDES
    from pytracking_b200.tracker import HostLogic
    for name in ("cfg2", "stress"):
        d = np.load(os.path.join(GOLDEN, "dimp_host_%s.npz" % name))
        params = _params(**OVERRIDES[name])
        hl = HostLogic(params)
        H, W = [int(v) for v in d["image_hw"]]
        hl.adopt(H, W, d["init_state"], d["init_sw"], d["init_counts"][0], d["init_counts"][1])
        from tracker_cases import _loc
        for t in range(len(d["flag"])):
            g = hl.plan_crop()
            st = hl.state()
            neigh = [np.float32(np.float32(params.target_neighborhood_scale) * (st[2 + i] / np.float32(g.sample_scale))) * np.float32(18.0 / 288.0) for i in range(2)]
            pv = [(st[i] - np.float32(g.sample_pos[i])) / (np.float32(16.0) * np.float32(g.sample_scale)) for i in range(2)]
            out = _run_localize(torch.from_numpy(d["scores"][t])[None], params, [neigh], [pv])
            assert out.flag == d["flag"][t], (name, t, out.flag, d["flag"][t])
            assert (out.r1, out.c1) == (int(d["m1"][t, 1]), int(d["m1"][t, 2])) and np.float32(out.score1) == np.float32(d["m1"][t, 0])
            if d["m2"][t, 1] >= 0:
                assert (out.r2, out.c2) == (int(d["m2"][t, 1]), int(d["m2"][t, 2])) and np.float32(out.score2) == np.float32(d["m2"][t, 0])
            assert out.use_second == d["use2"][t]
            hl.commit(g, _loc(d, t))
        hl.close()


def test_localize_kernel_matches_reference_code_on_random_maps():
    """Against the reference `DiMP.localize_target` on seeded random maps (recorded by oracle/gen_localize_golden.py)."""
    from oracle.gen_localize_golden import cases
    from pytracking_b200.tracker import FLAGS
    d = np.load(os.path.join(GOLDEN, "localize_random.npz"))
    img_support_sz, out_sz = torch.Tensor([288, 288]), torch.Tensor([18, 18])
    seen = set()
    for trial, (kw, scores, target_sz, sample_pos, sample_scales, pos) in enumerate(cases(400)):
        params = _params(**kw)
        S = scores.shape[0]
        neigh = [(2.2 * (target_sz / sample_scales[s]) * (out_sz / img_support_sz)).numpy() for s in range(S)]
        pv = [((pos - sample_pos[s]) / ((img_support_sz / out_sz) * sample_scales[s])).numpy() for s in range(S)]
        out = _run_localize(scores, params, neigh, pv)
        assert out.flag == d["flag"][trial], (trial, FLAGS[out.flag], FLAGS[d["flag"][trial]])
        assert out.scale_ind == d["scale_ind"][trial]
        cell = (out.r2, out.c2) if out.use_second else (out.r1, out.c1)
        mine = (torch.Tensor(cell) - 9) * (img_support_sz / out_sz) * sample_scales[out.scale_ind]
        assert torch.equal(mine, torch.from_numpy(d["tv"][trial])), (trial, mine, d["tv"][trial])
        seen.add((FLAGS[out.flag], out.use_second))
    assert {("normal", 0), ("hard_negative", 0), ("hard_negative", 1), ("uncertain", 0), ("not_found", 0), (None, 0)} <= seen, seen


# ---------------------------------------------------------------------------------------------------------------------------
def test_native_tracker_reproduces_recorded_reference_run():
    """Native initialisation + 40 closed-loop frames from uint8 frames: boxes bit-identical to the reference tracker's (CPU,
    use_augmentation=False, filter_init_zero=True) and flags identical for as long as the trajectories coincide (at least 10 frames;
    they may part only at a near-tie of the recorded score map, see below), first-frame score map within 1e-4."""
    from tracker_cases import OVERRIDES
    from pytracking_b200 import synth
    from pytracking_b200.tracker import DiMPTracker, FLAGS
    d = np.load(os.path.join(GOLDEN, "dimp_host_noaug.npz"))
    sd = synth.make_dimp_state_dict("resnet50", seed=0, lut_seed=3)
    trk = DiMPTracker(sd, _params(**OVERRIDES["noaug"]))
    frames, bb = synth.make_sequence(2, num_frames=len(d["flag"]))
    trk.initialize(frames[0], {"init_bbox": bb})
    assert np.array_equal(trk.state(), d["init_state"])
    drift = []
    horizon = len(d["flag"])
    for t in range(len(d["flag"])):
        out = trk.track(frames[t + 1])
        s = trk.engine.scores[0].cpu().numpy()
        ref_s = d["scores"][t]
        if not np.array_equal(np.array(out["target_bbox"], dtype=np.float32), d["bbox"][t]):
            # A closed loop can only part ways at a discrete decision.  The closed-loop score drift against the recorded CPU run is
            # chaotic (the per-frame optimiser amplifies rounding differences: median 4e-3, max 4e-2 of the score range over these 40
            # frames even while every box is bit-identical, see the print below), so a frame whose two best cells are closer than
            # that drift can go either way: which one depends on the summation order of the split-K partial sums.  Accepted only if
            # the recorded run's own gap between the two cells is within twice the drift seen on the preceding frames, and not before
            # frame 10; the filter-synchronised lockstep tests below pin the later frames.
            mine, theirs = np.unravel_index(np.argmax(s), s.shape), np.unravel_index(np.argmax(ref_s), ref_s.shape)
            gap = abs(float(ref_s[mine]) - float(ref_s[theirs])) / float(np.abs(ref_s).max())
            recent = max(drift[-5:])
            print("native tracker leaves the recorded trajectory at frame %d: cells %s / %s, recorded score gap %.2e, recent drift %.2e" % (t, mine, theirs, gap, recent))
            assert gap <= 2 * recent, (t, out["target_bbox"], d["bbox"][t], mine, theirs, gap, recent)
            horizon = t
            break
        assert trk.info.flag == d["flag"][t], (t, FLAGS[trk.info.flag])
        drift.append(float(np.abs(s - ref_s).max() / np.abs(ref_s).max()))
    assert horizon >= 10, horizon
    # closed loop: the first frame sees the filter of the first-frame optimisation only; later frames accumulate the (chaotic)
    # amplification of rounding differences by the per-frame optimiser runs -- reported, and bounded loosely
    print("native tracker vs recorded CPU reference run: score-map rel. diff frame 1 %.2e, median %.2e, max %.2e" %
          (drift[0], float(np.median(drift)), max(drift)))
    assert drift[0] <= 1e-4, drift[0]
    trk.close()


def _lockstep(n_frames, seq, use_aug, overrides, sync_filter=False, use_iou_net=False):
    """Reference tracker above the engine and the native tracker (adopting the reference's initialisation) side by side.
    closed loop (sync_filter=False): boxes and flags must stay identical; the score maxima are reported (the 10-iteration-per-frame
    update of a random-init model amplifies last-bit differences, e.g. the summation order of the sample weights, frame after frame).
    sync_filter=True: the native filter is reset to the reference's before every frame -> per-frame scores and the filter after the
    frame's update are compared at the 1e-4 bar."""
    _ref()
    from baseline import ref_tracker
    from pytracking_b200 import plugin, synth
    from pytracking_b200.tracker import DiMPTracker, FLAGS, make_params
    frames, bb = synth.make_sequence(seq, num_frames=n_frames)
    plugin.install()
    drift, box_err, upd = [], [], []
    try:
        ref = ref_tracker.build_dimp("cuda", overrides=overrides, use_augmentation=use_aug, use_iou_net=use_iou_net)
        torch.manual_seed(0)
        ref.initialize(frames[0], {"init_bbox": list(bb)})
        nat = DiMPTracker(ref.params.net.net.state_dict(), make_params(ref.params))
        nat.torch_noise = True
        nat.adopt_reference(ref, frames[0].shape[:2])
        for t in range(1, n_frames + 1):
            if sync_filter:
                nat.engine.filter.copy_(ref.target_filter.reshape(nat.engine.filter.shape))
            rng = torch.get_rng_state()
            a = ref.track(frames[t], {})["target_bbox"]
            torch.set_rng_state(rng)                       # the native tracker draws the same proposal noise the reference just drew
            b = nat.track(frames[t])["target_bbox"]
            if use_iou_net:
                box_err.append(float(np.abs(np.array(a) - np.array(b)).max()))
                assert box_err[-1] < 1e-2, (t, a, b)
            else:
                assert a == b, (t, a, b)
            assert ref.debug_info["flag"] == FLAGS[nat.info.flag], (t, ref.debug_info["flag"], FLAGS[nat.info.flag])
            drift.append(abs(ref.debug_info["max_score"] - nat.info.max_score) / abs(ref.debug_info["max_score"]))
            if sync_filter:
                assert drift[-1] <= 1e-4, (t, drift[-1])
                f_ref = ref.target_filter.reshape(-1)
                f_nat = nat.engine.filter.reshape(-1)
                upd.append(float((f_ref - f_nat).abs().max() / f_ref.abs().max()))
                if upd[-1] > 1e-5:            # diagnostics of the rare large events
                    n_ = int(min(int(ref.num_stored_samples[0]), nat.params.sample_memory_size))
                    swd = float((ref.sample_weights[0][:n_] - nat.engine.sample_weights[:n_]).abs().max() / ref.sample_weights[0][:n_].abs().max())
                    memd = float((ref.training_samples[0][:n_] - nat.engine.memory[:n_]).abs().max())
                    boxd = float((ref.target_boxes[:n_] - nat.engine.boxes[:n_]).abs().max())
                    print("  frame %d: filter diff %.2e; flag %s; replace ref %s nat %d; iters nat %d; weights rel diff %.1e; memory abs diff %.1e; "
                          "boxes abs diff %.1e" % (t, upd[-1], ref.debug_info["flag"], ref.previous_replace_ind[0], nat.info.replace_ind,
                                                   nat.info.num_iter, swd, memd, boxd))
                # one optimiser call from identical filters, memories and boxes; the only input that can differ is the last bit of a
                # sample weight (torch sums them on the GPU, the tracker on the host) -- see test_sd_sensitivity_to_sample_weight_rounding below
                assert upd[-1] <= 2e-3, (t, upd[-1])
        nat.close()
    finally:
        plugin.uninstall()
    print("lockstep seq %d: %d frames, boxes %s; max-score drift first/median/last: %.2e / %.2e / %.2e%s" %
          (seq, n_frames, "within %.1e px" % max(box_err) if box_err else "bit-identical", drift[0], float(np.median(drift)), drift[-1],
           "; filter after one update: median %.2e, max %.2e" % (float(np.median(upd)), max(upd)) if upd else ""))


def test_sd_sensitivity_to_sample_weight_rounding():
    """Sensitivity of the BASELINE configs[1] update on a REAL tracker memory: the steepest-descent calls of a few consecutive frames
    run twice from the tracker's own state, the second time with the sample weights perturbed by 1e-6 relative (what the two
    implementations of `update_sample_weights` accumulate over ~100 frames).  Typically the filter moves by about as much -- the update
    is well conditioned -- but DiMP's loss is NOT smooth: the activation derivative contains sign(score) (LeakyReluParDeriv,
    ltr/models/layers/activation.py:40-44; optimizer.py:139-141), so a perturbation that flips the sign of one near-zero score changes
    a Gauss-Newton step discontinuously.  The filter-synchronised lock-step test shows exactly that pattern: median 2e-7 per update,
    sporadic 1e-4 .. 1.6e-3 (same memory, same boxes, weights 1e-6 apart), and BASELINE configs[1] applies such an update every frame."""
    from tracker_cases import OVERRIDES
    from pytracking_b200 import ops, synth
    from pytracking_b200.tracker import DiMPTracker
    sd = synth.make_dimp_state_dict("resnet50", seed=0, lut_seed=3)
    trk = DiMPTracker(sd, _params(**dict(OVERRIDES["cfg2"])))
    frames, bb = synth.make_sequence(0, num_frames=60)
    trk.initialize(frames[0], {"init_bbox": bb})
    for t in range(1, 61):
        trk.track(frames[t])
    torch.cuda.synchronize()
    e = trk.engine
    feat, boxes, sw, w0 = e.memory.contiguous().clone(), e.boxes.clone(), e.sample_weights.clone(), e.filter.clone()
    p = {k[len("classifier.filter_optimizer."):]: v for k, v in sd.items() if k.startswith("classifier.filter_optimizer.")}
    luts = [p[k].cuda() for k in ("label_map_predictor.weight", "target_mask_predictor.0.weight", "spatial_weight_predictor.weight")]
    # (a single-ulp change of one weight usually vanishes in the kernel's sqrt(sw): perturb every weight by a few ulps instead)
    eps = 1e-6
    sw2 = sw * (1 + eps * (2 * torch.rand(sw.shape, generator=torch.Generator().manual_seed(0)).to(sw.device) - 1))
    res = {}
    for calls in (1, 5, 20):
        out = []
        for weights in (sw, sw2):
            w = w0.clone()
            for _ in range(calls):
                w, _, _ = ops.dimp_sd_gn(w, feat, boxes, weights, *luts, 10, e.step_length, e.reg_weight)
            out.append(w)
        res[calls] = float((out[0] - out[1]).abs().max() / out[0].abs().max())
    print("sample weights of a real tracker memory perturbed by %.0e relative -> filter moved (relative) by %s after 1 / 5 / 20 update "
          "calls of 10 iterations (amplification x%s)" % (eps, ", ".join("%.2e" % res[c] for c in (1, 5, 20)),
                                                          ", x".join("%.0f" % (res[c] / eps) for c in (1, 5, 20))))
    a = ops.dimp_sd_gn(w0, feat, boxes, sw, *luts, 10, e.step_length, e.reg_weight)[0]
    assert torch.equal(a, ops.dimp_sd_gn(w0, feat, boxes, sw, *luts, 10, e.step_length, e.reg_weight)[0])      # the kernel itself is deterministic
    trk.close()


def test_native_tracker_lockstep_with_reference_above_engine_cfg2():
    # closed loop at 10 iterations per frame: kept inside the horizon over which the reference agrees with itself across its own
    # backends (test_reference_dimp_above_engine_boxes_cfg2: 27 frames)
    _lockstep(20, 0, True, {})


def test_native_tracker_lockstep_filter_synchronised():
    _lockstep(120, 1, True, {}, sync_filter=True)


def test_native_tracker_lockstep_default_dimp50_schedule():
    # the stock parameter file's schedule (train_skipping 20, 2 iterations, hard negatives 1) with the not-found test disabled
    _lockstep(200, 3, True, dict(train_skipping=20, net_opt_update_iter=2))


def test_native_tracker_lockstep_with_iounet():
    # default dimp50 incl. IoUNet refinement (9 random proposals, 5 ascent steps, top-3 mean): boxes are floating-point outputs here
    _lockstep(40, 4, True, dict(train_skipping=20, net_opt_update_iter=2), use_iou_net=True)


# ---------------------------------------------------------------------------------------------------------------------------
def _run_ref(kind, frames, bb, n, **kw):
    from baseline import ref_tracker
    from pytracking_b200 import plugin
    if kind == "engine":
        plugin.install()
        plugin.stats.clear()
    try:
        trk = ref_tracker.build_dimp("cpu" if kind == "cpu" else "cuda", **kw)
        scores = []
        orig = trk.classify_target
        trk.classify_target = lambda x: (scores.append(orig(x)) or scores[-1])
        r = ref_tracker.run_sequence(trk, frames[:n + 1], bb)
        r["scores"] = [s.detach().float().cpu().numpy() for s in scores]
        r["stats"] = dict(plugin.stats)
        return r
    finally:
        if kind == "engine":
            plugin.uninstall()


def _first_diff(a, b):
    n = min(len(a), len(b))
    same = np.all(a[:n] == b[:n], axis=1)
    return n if same.all() else int(np.argmin(same))


SEAMS_DIMP = ("extract_backbone", "extract_classification_feat", "apply_filter", "DiMPSteepestDescentGN.forward", "max2d")


def test_reference_dimp_above_engine_boxes_bit_identical_stock_schedule():
    """The UNMODIFIED reference DiMP with the stock parameter file's update schedule (train_skipping 20, 2 iterations; default
    augmentation without the device-RNG dropout entry; zero filter initialiser because a stock checkout has no working PrRoIPool) on
    stock PyTorch-CUDA (TF32 off), on stock PyTorch-CPU and above the engine: 200 frames, `target_bbox` lists bit-identical."""
    _ref()
    from pytracking_b200 import synth
    torch.set_num_threads(16)
    n = 200
    frames, bb = synth.make_sequence(0, num_frames=n)
    kw = dict(overrides=dict(filter_init_zero=True, train_skipping=20, net_opt_update_iter=2), dropout=False)
    eng = _run_ref("engine", frames, bb, n, **kw)
    cuda = _run_ref("cuda", frames, bb, n, **kw)
    cpu = _run_ref("cpu", frames, bb, n, **kw)
    for seam in SEAMS_DIMP:
        assert eng["stats"].get(seam, 0) > 0, (seam, eng["stats"])
    assert np.array_equal(eng["target_bbox"], cuda["target_bbox"]), _first_diff(eng["target_bbox"], cuda["target_bbox"])
    assert np.array_equal(eng["target_bbox"], cpu["target_bbox"]), _first_diff(eng["target_bbox"], cpu["target_bbox"])
    # score maps before the first online update (frames 1..19 use the filter of the first-frame optimisation)
    for t in range(19):
        ref = cpu["scores"][t]
        assert np.abs(eng["scores"][t] - ref).max() <= 1e-4 * np.abs(ref).max() + 2e-6, (t, float(np.abs(eng["scores"][t] - ref).max() / np.abs(ref).max()))


def test_reference_dimp_above_engine_boxes_cfg2():
    """BASELINE configs[1] (10 steepest-descent iterations every frame) on a random-init network is a chaotic iteration: the stock
    reference itself, run on its two own backends (PyTorch-CPU, PyTorch-CUDA with TF32 off), produces score maps that differ by tens
    of percent after a few frames and boxes that part ways after a few dozen.  The engine is held to the reference's own consistency:
    wherever the two stock backends agree on the box, the engine's box is bit-identical to it."""
    _ref()
    from pytracking_b200 import synth
    torch.set_num_threads(16)
    n = 120
    frames, bb = synth.make_sequence(0, num_frames=n)
    kw = dict(overrides=dict(filter_init_zero=True), dropout=False)
    eng = _run_ref("engine", frames, bb, n, **kw)
    cuda = _run_ref("cuda", frames, bb, n, **kw)
    cpu = _run_ref("cpu", frames, bb, n, **kw)
    stock_agree = _first_diff(cpu["target_bbox"], cuda["target_bbox"])
    e_cpu, e_cuda = _first_diff(eng["target_bbox"], cpu["target_bbox"]), _first_diff(eng["target_bbox"], cuda["target_bbox"])
    print("cfg2: stock CPU vs stock CUDA agree for %d frames; engine vs CPU %d, engine vs CUDA %d (of %d)" % (stock_agree, e_cpu, e_cuda, n))
    assert stock_agree >= 10
    assert min(e_cpu, e_cuda) >= stock_agree, (stock_agree, e_cpu, e_cuda)
    assert max(e_cpu, e_cuda) >= min(n, stock_agree + 1) or stock_agree == n       # beyond that it follows one of the two
    ref = cpu["scores"][0]
    assert np.abs(eng["scores"][0] - ref).max() <= 1e-4 * np.abs(ref).max() + 2e-6


def test_reference_dimp_with_iounet_above_engine():
    """Default dimp50 (use_iou_net=True): the IoUNet refinement differentiates through the library's PrRoIPool
    (`_prroi_pooling` seam).  Stock PyTorch-CUDA cannot run this (the reference's native module does not build on current torch),
    so the comparison is against the CPU run with the oracle's PrRoIPool; boxes are floating-point outputs here (mean of refined
    proposals): compared to 1e-3 px while the runs coincide."""
    _ref()
    from pytracking_b200 import synth
    torch.set_num_threads(16)
    n = 12
    frames, bb = synth.make_sequence(0, num_frames=n)
    eng = _run_ref("engine", frames, bb, n, use_iou_net=True, dropout=False)
    cpu = _run_ref("cpu", frames, bb, n, use_iou_net=True, dropout=False)
    for seam in ("prroi_pooling_forward", "predict_iou", "get_iou_feat"):
        assert eng["stats"].get(seam, 0) > 0, (seam, eng["stats"])
    d = np.abs(eng["target_bbox"] - cpu["target_bbox"]).max(axis=1)
    print("IoUNet boxes, engine vs CPU reference, max abs diff per frame [px]:", np.round(d, 5).tolist())
    assert d.max() < 1e-2, d
    # (later score maps are not comparable: a 1e-5 px difference in the refined size can change the integer crop size by one pixel)
    ref = cpu["scores"][0]
    assert np.abs(eng["scores"][0] - ref).max() <= 1e-4 * np.abs(ref).max() + 2e-6
