#!/usr/bin/env python
"""bench.py -- DiMP-50 tracked frames/sec on the synthetic sequence (BASELINE.json configs[1]: 288x288 search crops, 10 SD iters/frame).

One "step" = one tracked frame, uint8 camera frame in -> bounding box out, of the steady-state tracker (50-sample memory full):
crop sampling -> ResNet-50 backbone to layer3 -> clf head -> apply_filter -> localisation -> state update -> memory insert ->
10 steepest-descent iterations over the 50 samples.  Both arms run the SAME tracker configuration (`CONFIG`), the same frames, the
same pre-roll (PREROLL untimed frames after initialisation so that the memory is full), W warm-up frames, then K timed frames.

  --impl b200 (default)
      value : frames/s of `b200trk_dimp_track_device` -- the uint8 frames already resident in HBM (device-timed with CUDA events,
              max over ranks); L2 is flushed before the timed region and every step reads a frame nobody touched before.
      e2e   : frames/s of `DiMPTracker.track(frame)` -- the public call: pinned HOST uint8 frame in, box out; the H2D copy of the
              frame and the D2H of the localisation result are inside the timed region (wall clock around the loop, max over ranks).
      roofline[]         : per-kernel CUDA-event timings inside this run (steepest-descent optimiser, backbone+head, apply_filter).
      cpu_baseline       : the unmodified reference tracker (baseline/_ref) on rank 0's host cores, bounded sample.
      torch_cuda_baseline: the unmodified reference tracker on stock PyTorch-CUDA (cuDNN, TF32 off) on the same GPU -- what a
                           pytracking user runs today -- and the same reference tracker above the engine (`plugin.install()`).
  --impl reference
      The UNMODIFIED reference `DiMP` tracker (baseline/_ref, staged from /root/reference by baseline/stage_reference.py), stock
      PyTorch CPU path, timed as the reference times itself (time.time() around `tracker.track`,
      pytracking/evaluation/tracker.py:226-233).  One reference process per rank, host threads split evenly between the ranks,
      whole-job value = world * K / max-over-ranks time (gloo gather).

Multi-GPU: one process per GPU, sequence q = rank (weak scaling), no collective in the frame loop; at the end ONE NCCL all_gather of the
per-sequence boxes / times (pytracking_b200/shard.py) from which the aggregate FPS and mean IoU against the synthetic ground truth
are computed (pytracking/analysis/extract_results.py:29-39).
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CROP, MEMORY, SD_ITERS, PREROLL = 288, 50, 10, 56
# pytracking/parameter/dimp/dimp50.py + the BASELINE configs[1] overrides of SURVEY.md 8(d); identical in both arms
TRACKER_PARAMS = dict(image_sample_size=CROP, search_area_scale=5, sample_memory_size=MEMORY, learning_rate=0.01,
                      init_samples_minimum_weight=0.25, train_skipping=1, update_classifier=True, net_opt_iter=10,
                      net_opt_update_iter=SD_ITERS, net_opt_hn_iter=1, advanced_localization=True, target_not_found_threshold=-1e9,
                      distractor_threshold=0.8, hard_negative_threshold=0.5, target_neighborhood_scale=2.2, dispalcement_scale=0.8,
                      hard_negative_learning_rate=0.02, augmentation_expansion_factor=2, use_iou_net=False)
REF_OVERRIDES = dict(target_not_found_threshold=-1e9, train_skipping=1, net_opt_update_iter=SD_ITERS, filter_init_zero=True)
METRIC = "DiMP-50 tracked frames/sec (uint8 frame -> box; 288x288 search crops, 10 SD iters/frame over a 50-sample memory)"
CONFIG = {"workload": "DiMP-50 single-GPU, synthetic 288x288 crops, 10 SD iters/frame (BASELINE configs[1]); synthetic 480x640 uint8 "
                      "sequence of SURVEY.md 8(d), one independent sequence per GPU / rank",
          "tracker": "pytracking/parameter/dimp/dimp50.py + target_not_found_threshold=-1e9, train_skipping=1, net_opt_update_iter=10, "
                     "use_iou_net=False, use_augmentation=False, filter_init_zero=True",
          "backbone": "resnet50->layer3", "memory": MEMORY, "sd_iters": SD_ITERS, "use_iou_net": False, "preroll_frames": PREROLL,
          "network": "random init (seed 0), identical state_dict in both arms",
          "l2": "L2 flushed (256 MB write) before the timed region; every step reads a frame not touched before; network weights and "
                "the sample memory are the tracker's steady-state working set"}


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures of the same kernels at the same
# sizes (profiles/r02x_ncu_summary_all_kernels.txt, profiles/r02x_ncu_summary_conv_tc.txt; tools/ncu_round.sh) -- not measured in this run
NCU_TRAFFIC = {"sd_tc": 36251000 + 394000, "conv_chain": 149774000, "apply_filter": 726000}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", type=int, default=0)
    ap.add_argument("--no-baselines", action="store_true", help="skip cpu_baseline / torch_cuda_baseline (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each leg returned as DIR/<name>.npy (dimp50 --impl b200 only): "
                         "target_bbox, scores and filter of the device-resident leg, e2e_target_bbox of the host-buffer leg")
    ap.add_argument("--config", default="dimp50", choices=["dimp50", "prdimp50", "atom", "tomp101", "eco", "dimp_simple"],
                    help="dimp50 = BASELINE configs[1] (the metric of record, native whole-frame tracker); the others time the UNMODIFIED "
                         "reference tracker of BASELINE configs[2] / [0] / [3] above the engine (plugin.install()) against the same tracker "
                         "on stock PyTorch-CUDA and PyTorch-CPU; eco / dimp_simple: the same for the reference ECO and SuperDiMPSimple trackers "
                         "(not BASELINE configurations; their optimiser seams were bound last)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)),
                "bf16_tflops_burst": d.get("bf16_tflops", 1590.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_burst": 1590.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
                for n, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_cores():
    """Cores this process may really use: scheduler affinity, capped by the cgroup CPU quota if there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def make_frames(rank, count):
    from pytracking_b200 import synth
    frames, bb = synth.make_sequence(rank, num_frames=count)
    return frames, bb, synth.sequence_ground_truth(rank, count)


# ------------------------------------------------------------------------------------------------------------
# reference tracker (unmodified, baseline/_ref): shared by --impl reference, cpu_baseline and torch_cuda_baseline
# ------------------------------------------------------------------------------------------------------------
def reference_available():
    from baseline import ref_env
    return ref_env.reference_available()


def run_reference_tracker(device, frames, bb, warmup, steps, threads=None, above_engine=False):
    """init + PREROLL + warmup untimed frames, then `steps` frames timed with the reference's own clock. -> (seconds, boxes)"""
    from baseline import ref_env, ref_tracker
    ref_env.install()
    if threads:
        torch.set_num_threads(threads)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    if above_engine:
        from pytracking_b200 import plugin
        plugin.install()
    try:
        trk = ref_tracker.build_dimp(device, use_iou_net=False, overrides=REF_OVERRIDES, use_augmentation=False)
        sync = torch.cuda.synchronize if device != "cpu" else None
        r = ref_tracker.run_sequence(trk, frames[:1 + PREROLL + warmup + steps], bb, sync=sync)
    finally:
        if above_engine:
            from pytracking_b200 import plugin
            plugin.uninstall()
    t = r["time"][PREROLL + warmup:]
    return float(t.sum()), r["target_bbox"]


def cpu_port_sample(steps):
    """Fallback when the reference tree is not staged: the torch-CPU restatement (oracle/) of the same per-frame tensor path."""
    from oracle import dimp_oracle as O
    from pytracking_b200 import synth
    from pytracking_b200.frame_engine import SampleWeights
    sd = synth.make_dimp_state_dict("resnet50", seed=0, lut_seed=3)
    p = {k[len("classifier.filter_optimizer."):]: v for k, v in sd.items() if k.startswith("classifier.filter_optimizer.")}
    memory, boxes = synth.make_clf_features(11, MEMORY, 512, 18, 18), synth.make_boxes(12, MEMORY)
    sw = SampleWeights(MEMORY, 15)
    for _ in range(MEMORY - 15):
        sw.step()
    w = torch.zeros(1, 512, 4, 4)
    crops = synth.make_crop(13, 4, CROP)
    t0 = None
    for i in range(steps + 1):
        if i == 1:
            t0 = time.perf_counter()
        with torch.no_grad():
            bf = O.resnet_forward(sd, O.preprocess_image(crops[i % 4:i % 4 + 1]), "resnet50", output_layers=("layer3",))
            clf = O.clf_head_dimp50(sd, bf["layer3"])
            O.max2d(O.apply_filter_conv(clf, w)[:, 0])
            memory[sw.step()] = clf[0]
            w = O.dimp_sd_gn_conv(w, memory, boxes, torch.from_numpy(sw.w), p, SD_ITERS)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    K, W = args.steps, args.warmup
    cores = host_cores()
    threads = max(1, cores // world)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group(backend="gloo")
    frames, bb, gt = make_frames(rank, PREROLL + W + K)
    if reference_available():
        secs, boxes = run_reference_tracker("cpu", frames, bb, W, K, threads=threads)
        kind = "reference"
        sample = ("%d frames of the unmodified reference DiMP tracker (baseline/_ref, stock PyTorch CPU path, fp32) after init + %d "
                  "pre-roll + %d warm-up frames; time.time() around tracker.track" % (K, PREROLL, W))
    else:
        torch.set_num_threads(threads)
        secs = cpu_port_sample(K)
        kind = "port"
        sample = "%d frames of the torch-CPU restatement (oracle/) -- baseline/_ref is not staged on this machine" % K
    t = torch.tensor([secs], dtype=torch.float64)
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        torch.distributed.all_gather(allt, t)
        t = torch.stack(allt).max(dim=0).values
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    secs = float(t[0])
    v = world * K / secs
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": secs / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": threads * world, "kind": kind, "sample": sample,
                         "processes": world, "threads_per_process": threads},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------------------
# b200 arm
# ------------------------------------------------------------------------------------------------------------
def event_time_us(fn, reps, stream_sync=True):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev])) * 1e3


def run_b200(args, rank, world, local_rank):
    from pytracking_b200 import _lib, shard, synth
    from pytracking_b200.tracker import DiMPTracker, make_params
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    K, W = args.steps, args.warmup
    n_frames = PREROLL + 2 * (W + K)
    frames, bb, gt = make_frames(rank, n_frames)
    H, Wd = frames[0].shape[:2]
    sd = synth.make_dimp_state_dict("resnet50", seed=0, lut_seed=3)
    trk = DiMPTracker(sd, make_params(**TRACKER_PARAMS), arch="resnet50", precision=args.precision, device=dev)
    pinned = torch.empty(n_frames + 1, H, Wd, 3, dtype=torch.uint8).pin_memory()
    for i, f in enumerate(frames):
        pinned[i] = torch.from_numpy(f)
    barrier = (lambda: torch.distributed.barrier()) if world > 1 else (lambda: None)
    boxes = []

    # ---- setup (untimed): initialise on frame 0, pre-roll until the 50-sample memory is full ----
    trk.initialize(pinned[0], {"init_bbox": bb})
    f = 1
    for _ in range(PREROLL):
        boxes.append(trk.track(pinned[f])["target_bbox"]); f += 1
    assert trk.info.n_stored == MEMORY, trk.info.n_stored

    # ---- device-resident leg (value) ----
    dev_frames = pinned[f:f + W + K].to(dev)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    for i in range(W):
        trk.track_device(dev_frames[i]); boxes.append(list(trk.info.bbox))
    torch.cuda.synchronize(); barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.3)
    launches0 = _lib.lib().b200trk_launch_count()
    flush.fill_(1.0)                                                    # L2 flush: 256 MB written right before the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gc.collect(); gc.disable()                                          # no collector pauses inside the timed regions (re-enabled below)
    torch.cuda.synchronize(); barrier()
    e0.record()
    for i in range(K):
        trk.track_device(dev_frames[W + i]); boxes.append(list(trk.info.bbox))
    e1.record()
    torch.cuda.synchronize(); barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = _lib.lib().b200trk_launch_count() - launches0
    # what the last timed track_device returned, read back after the timed region
    outputs = {"target_bbox": np.array(trk.info.bbox, dtype=np.float64), "scores": trk.engine.scores.float().cpu().numpy(),
               "filter": trk.engine.filter.float().cpu().numpy()}
    f += W + K
    del dev_frames

    # ---- host-buffer leg (e2e): the public call, pinned uint8 frame in, box out ----
    per_frame = []
    for i in range(W):
        boxes.append(trk.track(pinned[f])["target_bbox"]); f += 1
    flush.fill_(2.0)
    torch.cuda.synchronize(); barrier()
    t0 = time.perf_counter()
    for i in range(K):
        ts = time.perf_counter()
        boxes.append(trk.track(pinned[f])["target_bbox"]); f += 1
        per_frame.append(time.perf_counter() - ts)
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - t0) * 1e3
    gc.enable()
    outputs["e2e_target_bbox"] = np.array(boxes[-1], dtype=np.float64)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    barrier()
    clocks = sampler.finish() if sampler else None

    # ---- per-kernel timings for the roofline entries (CUDA events on the launching stream, same process, same state) ----
    eng = trk.engine
    sw_host = np.full(MEMORY, 1.0 / MEMORY, dtype=np.float32)
    eng.sample_weights.copy_(torch.from_numpy(sw_host).to(dev))
    box_host = np.array([120, 120, 50, 50], dtype=np.float32)
    sd_us = event_time_us(lambda: eng.update(0, 7, box_host, sw_host, MEMORY, SD_ITERS), 20)
    sd_tc = int(_lib.lib().b200trk_sd_last_kernel())
    crop_dev = synth.make_crop(5, 1, CROP).to(dev)
    net_us = event_time_us(lambda: eng.backbone.forward(crop_dev, want=("classification",)), 20)
    import ctypes as C
    L = _lib.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def apply_only():
        _lib.check(L.b200trk_apply_filter(C.c_void_p(eng.clf.data_ptr()), C.c_void_p(eng.filter.data_ptr()), C.c_void_p(eng.scores.data_ptr()),
                                          1, 512, 18, 18, 4, None, None, st), "apply_filter")
    af_us = event_time_us(apply_only, 50)

    # ---- gather: max over ranks + the final result gather (boxes, per-frame times) ----
    t = torch.tensor([dev_ms, host_ms, sd_us, net_us, af_us], device=dev, dtype=torch.float64)
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        torch.distributed.all_gather(allt, t)
        t = torch.stack(allt).max(dim=0).values
    dev_ms, host_ms, sd_us, net_us, af_us = [float(x) for x in t.cpu()]
    bx = torch.tensor(np.array(boxes, dtype=np.float32))
    times = torch.zeros(bx.shape[0]); times[-K:] = torch.tensor(per_frame)
    merged = shard.gather_results({rank: (bx, times)}, world, n_frames, device=dev if world > 1 else None)
    if rank != 0:
        return
    ious = []
    for q, (b, _) in merged.items():
        g = torch.tensor(synth.sequence_ground_truth(q, n_frames)[1:1 + b.shape[0]], dtype=torch.float32)
        ious.append(float(shard.iou_overlap(b, g).mean()))
    peaks = load_peaks()
    # SURVEY.md 8(d): SD-GN algorithmic bytes per iteration = 3*n*663552 + 8*n*1444 + 3*32768 B (n = 50)
    sd_bytes = SD_ITERS * (3 * MEMORY * 663552 + 8 * MEMORY * 1444 + 3 * 32768)
    sd_once = MEMORY * 663552 + SD_ITERS * (8 * MEMORY * 1444 + 3 * 32768)      # the fused lower bound: sample memory read once per call
    net_flops = float(eng.backbone.flops)
    af_bytes = 4 * (512 * 18 * 18 + 512 * 16 + 19 * 19)
    roof = [
        {"kernel": ("sd_tc_kernel<18,0>" if sd_tc else "sd_kernel<18,4,0>") + " (DiMP steepest descent, n=50, 10 it, one launch)",
         "bound": "hbm", "achieved": sd_bytes / (sd_us * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
         "frac": sd_bytes / (sd_us * 1e-6) / 1e9 / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC["sd_tc"] if sd_tc else None, "us_per_launch": sd_us,
         "us_per_sd_iteration": sd_us / SD_ITERS, "algorithmic_bytes": sd_bytes,
         "fused_lower_bound": {"bytes": sd_once, "us_at_peak": sd_once / (peaks["hbm_gbs"] * 1e3), "frac": sd_once / (peaks["hbm_gbs"] * 1e3) / sd_us}},
        {"kernel": "conv_tc_kernel chain (ResNet-50 -> layer3 + clf head, batch 1, 3xTF32 on tcgen05; whole forward)", "bound": "tensor",
         "achieved": net_flops / (net_us * 1e-6) / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
         "frac": net_flops / (net_us * 1e-6) / 1e12 / peaks["bf16_tflops"], "traffic": NCU_TRAFFIC["conv_chain"], "us_per_launch": net_us,
         "algorithmic_flops": net_flops, "mma_issue_flops": 3 * net_flops},
        {"kernel": "apply_filter_kernel<18,16> (classify, 1 sample)", "bound": "hbm", "achieved": af_bytes / (af_us * 1e-6) / 1e9,
         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": af_bytes / (af_us * 1e-6) / 1e9 / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC["apply_filter"],
         "us_per_launch": af_us, "algorithmic_bytes": af_bytes},
    ]
    out = {
        "metric": METRIC, "value": world * K / (dev_ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (3xTF32 error-compensated tcgen05 convolutions and optimiser sweeps; fp32 CUDA-core correlation)" if args.precision == 0 else "f32",
        "data": "synthetic", "config": CONFIG,
        "e2e": {"value": world * K / (host_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": H * Wd * 3 + 16 + MEMORY * 4,
                "d2h_bytes_per_step": 64, "api": "pytracking_b200.tracker.DiMPTracker.track(uint8 frame) -> {'target_bbox'}",
                "ms_per_frame_median": float(np.median(per_frame) * 1e3)},
        "gpu_launches": int(launches),
        "roofline": roof[0], "rooflines": roof, "peak_source": peaks["source"],
        "traffic_source": "ncu --set full captures committed under profiles/r02x_ncu_summary_*.txt (same kernels, same sizes, separate run)",
        "tracking": {"mean_iou_vs_synthetic_ground_truth": float(np.mean(ious)), "sequences": len(ious), "frames_per_sequence": len(boxes),
                     "gather": "one all_gather of [frames,6] per sequence at the end (pytracking_b200/shard.py)"},
        "clocks": clocks,
    }
    if not args.no_baselines and world == 1:            # the CPU / stock-CUDA baselines are N = 1 lines
        out["rooflines"] = roof + eco_rows(peaks)
        out.update(baselines(frames, bb, W))
    print(json.dumps(out))


def eco_rows(peaks):
    """SURVEY 8 row f4 (ECO's Fourier-domain optimisers), N = 1 / rank 0 only, AFTER the timed regions: tools/eco_bench.py in a subprocess
    (its own CUDA context, bounded by a timeout), CUDA-event medians at ECO's default block sizes.  `achieved` counts the sample memory
    once per call (the kernels keep the slabs resident in shared memory); `reference_sweep_bytes` is what the reference's mtimes pairs read."""
    import subprocess
    import tempfile
    name = "eco_cg_kernel / eco_joint_kernel (ECO FilterOptim.run / first-frame GaussNewtonCG.run, SURVEY 8 f4)"
    try:
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "eco_bench.json")
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "eco_bench.py"), "--json", path], capture_output=True, text=True,
                               timeout=240, cwd=ROOT)
            if r.returncode != 0 or not os.path.exists(path):
                return [{"kernel": name, "unavailable": ("rc=%d " % r.returncode) + r.stderr.strip()[-300:]}]
            data = json.load(open(path))
    except Exception as e:      # noqa: BLE001 -- a timing row must never take the bench line down
        return [{"kernel": name, "unavailable": repr(e)[:300]}]
    return eco_rows_from(data, peaks)


def eco_rows_from(data, peaks):
    rows = []
    for k, v in data.items():
        if k.startswith("joint "):
            rows.append({"kernel": "eco_joint_kernel (ECO first frame, GaussNewtonCG 10 x 10 on FactorizedConvProblem; %s)" % k[6:], "bound": "hbm",
                         "achieved": v["sample_bytes"] / (v["us_median"] * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": v["sample_bytes"] / (v["us_median"] * 1e-6) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                         "us_per_launch": v["us_median"], "algorithmic_bytes": v["sample_bytes"],
                         "note": "100 CG iterations with 4 grid barriers each: barrier / latency bound, the HBM figure is nominal"})
        elif k.startswith("scores "):
            rows.append({"kernel": "eco_preprocess_kernel x 2 + eco_apply_filter_kernel x 2 + eco_sample_fs_kernel + max2d_kernel (ECO.preprocess_sample / apply_filter / localize_target scores; %s)" % k[7:],
                         "bound": "hbm", "achieved": v["bytes"] / (v["us_median"] * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": v["bytes"] / (v["us_median"] * 1e-6) / 1e9 / peaks["hbm_gbs"], "traffic": None, "us_per_launch": v["us_median"],
                         "algorithmic_bytes": v["bytes"], "note": "six launches of a few microseconds each: launch / latency bound"})
        else:
            rows.append({"kernel": "eco_cg_kernel (ECO FilterOptim.run, 5 CG iterations; %s)" % k, "bound": "hbm", "achieved": v["GBps_vs_one_read"],
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": v["GBps_vs_one_read"] / peaks["hbm_gbs"], "traffic": None,
                         "us_per_launch": v["us_median"], "algorithmic_bytes": v["sample_memory_bytes"],
                         "reference_sweep_bytes": v["reference_sweep_bytes"], "achieved_vs_reference_sweeps": v["GBps_vs_reference_sweeps"]})
    return rows


def baselines(frames, bb, W):
    """Rank 0 only, after the timed regions: the unmodified reference on the host cores (bounded sample) and on PyTorch-CUDA."""
    res = {}
    cores = host_cores()
    if not reference_available():
        torch.set_num_threads(min(cores, 16))
        secs = cpu_port_sample(3)
        res["cpu_baseline"] = {"value": 3 / secs, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": "3 frames of the torch-CPU restatement (oracle/): baseline/_ref is not staged here"}
        return res
    n_cpu = 8
    secs, _ = run_reference_tracker("cpu", frames, bb, 1, n_cpu, threads=cores)
    res["cpu_baseline"] = {"value": n_cpu / secs, "unit": "frames/s", "cores": cores, "kind": "reference",
                           "sample": "%d frames of the unmodified reference DiMP tracker (baseline/_ref, stock PyTorch CPU path) after init + "
                                     "%d pre-roll + 1 warm-up frames; time.time() around tracker.track" % (n_cpu, PREROLL)}
    try:
        n_gpu = 60
        secs, b_cuda = run_reference_tracker("cuda", frames, bb, W, n_gpu)
        secs_e, b_eng = run_reference_tracker("cuda", frames, bb, W, n_gpu, above_engine=True)
        res["torch_cuda_baseline"] = {
            "value": n_gpu / secs, "unit": "frames/s", "kind": "unmodified reference tracker on stock PyTorch-CUDA (cuDNN / cuBLAS, TF32 "
            "off), same GPU, same frames; time.time() + cuda.synchronize() around tracker.track", "frames": n_gpu,
            "reference_above_engine": {"value": n_gpu / secs_e, "unit": "frames/s", "kind": "the same unmodified reference tracker with "
                                       "pytracking_b200.plugin.install() (every tensor seam served by libb200trk.so)",
                                       "boxes_identical_to_stock_cuda_frames": int(np.argmin(np.all(b_cuda == b_eng, axis=1))) if not np.array_equal(b_cuda, b_eng) else int(len(b_cuda)),
                                       "frames_compared": int(len(b_cuda)),
                                       "note": "10 iterations/frame on a random-init net is chaotic: the stock reference's own CPU and CUDA "
                                               "backends part ways after ~27 frames (tests/test_tracker_gpu.py)"}}
    except Exception as e:                                                         # the product numbers above must survive a baseline failure
        res["torch_cuda_baseline"] = {"error": repr(e)[:300]}
    return res


# ------------------------------------------------------------------------------------------------------------
# the other BASELINE configurations: frame-level lines through the unmodified reference trackers above the engine
# ------------------------------------------------------------------------------------------------------------
OTHER = {
    "prdimp50": ("PrDiMP-50 tracked frames/sec (352x352 crops, 22x22 features, 10 SD-Newton iters/frame over a 50-sample memory)",
                 "BASELINE configs[2]: parameter/dimp/prdimp50.py + target_not_found_threshold=-1e9, train_skipping=1, net_opt_update_iter=10, "
                 "use_iou_net=False, no dropout augmentation", 56),
    "atom": ("ATOM ResNet-18 tracked frames/sec (5 scales, Fourier score interpolation, 5 CG iters/frame over the 250-sample memory)",
             "BASELINE configs[0]: parameter/atom/multiscale_no_iounet.py + train_skipping=1, target_not_found_threshold=-1e9", 10),
    "tomp101": ("ToMP-101 tracked frames/sec (ResNet-101, 6+6 layer transformer model predictor over 972 tokens x 2)",
                "BASELINE configs[3]: parameter/tomp/tomp101.py + target_not_found_threshold=-1e9", 5),
    # not BASELINE configurations (SURVEY 8 f4 and its "also"): the trackers whose optimiser seams round 2 added last
    "eco": ("ECO tracked frames/sec (ResNet18m1 vggconv1 + layer3 features, 5 scales, Fourier-domain CG every frame over the 200-sample memory)",
            "parameter/eco/default.py + train_skipping=1 (5 CG iterations every frame), random-init resnet18_vggmconv1", 10),
    "dimp_simple": ("SuperDiMPSimple tracked frames/sec (352x352 crops, GNSteepestDescent over LinearFilterHinge, 2 iterations/frame)",
                    "parameter/dimp_simple/super_dimp_simple.py + target_not_found_threshold=-1e9, train_skipping=1, use_iou_net=False", 10),
}


def build_other(config, device):
    from baseline import ref_env, ref_tracker
    ref_env.install()
    if config == "prdimp50":
        return ref_tracker.build_prdimp(device, use_iou_net=False, dropout=False)
    if config == "atom":
        return ref_tracker.build_atom(device)
    if config == "eco":
        return ref_tracker.build_eco(device, overrides=dict(train_skipping=1))
    if config == "dimp_simple":
        return ref_tracker.build_dimp_simple(device, overrides=dict(train_skipping=1, use_iou_net=False))
    return ref_tracker.build_tomp(device)


def time_other(config, device, frames, bb, preroll, warmup, steps, above_engine=False, threads=None):
    from baseline import ref_env, ref_tracker
    ref_env.install()
    if threads:
        torch.set_num_threads(threads)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    stats = {}
    if above_engine:
        from pytracking_b200 import plugin
        plugin.install()
        plugin.stats.clear()
    try:
        trk = build_other(config, device)
        r = ref_tracker.run_sequence(trk, frames[:1 + preroll + warmup + steps], bb, sync=torch.cuda.synchronize if device != "cpu" else None)
        if above_engine:
            stats = dict(plugin.stats)
    finally:
        if above_engine:
            plugin.uninstall()
    return float(r["time"][preroll + warmup:].sum()), r["target_bbox"], stats


def run_other(args, rank, world, local_rank):
    metric, tracker_desc, preroll = OTHER[args.config]
    K, W = args.steps, args.warmup
    frames, bb, _ = make_frames(rank, preroll + W + K)
    cfg = {"workload": tracker_desc, "preroll_frames": preroll, "network": "random init (seeded), identical in every arm",
           "api": "unmodified reference tracker object: tracker.track(uint8 frame) -> {'target_bbox'}"}
    if args.impl == "reference":
        if rank != 0:
            return
        cores = host_cores()
        secs, _, _ = time_other(args.config, "cpu", frames, bb, preroll, W, K, threads=cores)
        v = K / secs
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
                          "ms_per_step": secs / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": cfg, "gpu_launches": 0,
                          "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference", "sample": "%d frames" % K},
                          "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    from pytracking_b200 import _lib
    torch.cuda.set_device(local_rank)
    l0 = _lib.lib().b200trk_launch_count()
    secs_e, b_eng, stats = time_other(args.config, "cuda", frames, bb, preroll, W, K, above_engine=True)
    launches = _lib.lib().b200trk_launch_count() - l0
    secs_c, b_cuda, _ = time_other(args.config, "cuda", frames, bb, preroll, W, K)
    n = min(len(b_eng), len(b_cuda))
    same = np.all(b_eng[:n] == b_cuda[:n], axis=1)
    out = {"metric": metric, "value": K / secs_e, "unit": "frames/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": secs_e / K * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
           "e2e": {"value": K / secs_e, "unit": "frames/s", "h2d_bytes_per_step": int(frames[0].nbytes), "d2h_bytes_per_step": 64,
                   "note": "the reference tracker's own host code (crop sampling, localisation) is inside the timed region"},
           "gpu_launches": int(launches), "seams_served": stats,
           "torch_cuda_baseline": {"value": K / secs_c, "unit": "frames/s", "kind": "the same unmodified reference tracker on stock PyTorch-CUDA (TF32 off)"},
           "speedup_vs_torch_cuda": secs_c / secs_e,
           "boxes_identical_to_stock_cuda_frames": int(n if same.all() else np.argmin(same)), "frames_compared": int(n),
           "max_box_abs_diff_first_10_frames_px": float(np.abs(b_eng[:10] - b_cuda[:10]).max())}
    from pytracking_b200 import plugin as _pl
    if _pl.seam_seconds:
        out["seam_seconds_per_frame"] = {k: v / (preroll + W + K) for k, v in _pl.seam_seconds.items()}
    if not args.no_baselines:
        cores = host_cores()
        k_cpu = min(K, 6)
        secs, _, _ = time_other(args.config, "cpu", frames, bb, preroll, 1, k_cpu, threads=cores)
        out["cpu_baseline"] = {"value": k_cpu / secs, "unit": "frames/s", "cores": cores, "kind": "reference",
                               "sample": "%d frames of the unmodified reference tracker on PyTorch-CPU after %d pre-roll frames" % (k_cpu, preroll)}
    print(json.dumps(out))


def main():
    args = parse()
    if args.dump_outputs and (args.config != "dimp50" or args.impl != "b200"):
        sys.exit("--dump-outputs: only the dimp50 workload of --impl b200 has outputs to write")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config != "dimp50":
        if rank == 0:
            run_other(args, rank, world, local_rank)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    run_b200(args, rank, world, local_rank)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
