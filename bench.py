#!/usr/bin/env python
"""Headline benchmark: detector FPS @1280x720 rpn300 (ResNet-101-FPN Faster-RCNN, batch 8 per GPU).

  python bench.py --gpus N --steps K --warmup W                (N>1: launched under torchrun, one rank/GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W   (the reference arm: CPU oracle port)
  python bench.py ... --dump-outputs DIR                           (also writes the last timed step's outputs to DIR)

A step = one pass of the hot path over one batch of synthetic frames.  `value` is whole-job FPS with
frames resident in HBM; `e2e` is the same through the host-buffer C-ABI call (pinned H2D of the frames
and D2H of boxes/probs/labels/box features inside the timed region).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # a benchmark run leaves the source tree as it found it (no __pycache__)

METRIC = "detector FPS @1280x720 rpn300 (ResNet-101-FPN Faster-RCNN)"
H, W, BATCH = 720, 1280, 8
CONV_GFLOP_PER_FRAME = 490.4      # SURVEY.md section 8: conv stack 245.2 GMAC
FC_GFLOP_PER_FRAME = 8.4


def workload_config(n_gpus, precision="split", input_dtype="float32"):
    """The workload both arms (--impl b200 / --impl reference) run; identical keys and values in both lines.  `precision`
    and `input_dtype` name the arithmetic of the GPU arm's operands at the boundary; the reference arm computes the same
    graph in float32 on the host (its own line says so under "arith")."""
    return {"workload": "ResNet-101-FPN Faster-RCNN rpn300 1280x720 batch=8 per GPU, detection only "
                        "(BASELINE configs[1], batch graph Mask_RCNN_FPN_multi); one stream per GPU, no data-path collective",
            "frame": [H, W, 3], "batch_per_gpu": BATCH, "global_batch": BATCH * n_gpus, "num_class": 15,
            "rpn_topk": 300, "precision": precision, "input_dtype": input_dtype,
            "weights": "seeded synthetic (synth.py, seed 1234)",
            "l2": "inputs rotate over distinct batches larger than the 126 MB L2 (4 x 88 MB float32 / 8 x 22 MB uint8) "
                  "and the per-step activation footprint (> 2 GB) exceeds L2",
            "parallelism": "replicas x%d" % n_gpus}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (B200_PROFILING.md): NVML every 10 ms
    (nvidia-smi every 200 ms as a fallback when the NVML binding is unavailable)."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.sm = []
        self.sm_max = None
        self.reason_bits = 0
        self.stop = threading.Event()
        self.how = "nvml"

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        # LOCAL_RANK indexes the visible devices; map through CUDA_VISIBLE_DEVICES when it is a plain index list
        idx = self.index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        if vis and all(v.strip().isdigit() for v in vis.split(",")):
            idx = int(vis.split(",")[self.index])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        while not self.stop.is_set():
            self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
            try:
                self.reason_bits |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                self.reason_bits |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            self.stop.wait(0.01)

    def _run_smi(self):
        self.how = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        bits = [0x8, 0x40, 0x20, 0x4]
        while not self.stop.is_set():
            r = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
            parts = [p.strip() for p in r.stdout.strip().split(",")]
            if len(parts) >= 6:
                self.sm.append(float(parts[0]))
                self.sm_max = float(parts[1])
                for b, v in zip(bits, parts[2:6]):
                    if v.lower().startswith("active"):
                        self.reason_bits |= b
            self.stop.wait(0.2)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            try:
                self._run_smi()
            except Exception:
                pass

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unsampled"], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.sm_max,
                "reasons": [n for b, n in self.REASONS.items() if self.reason_bits & b],
                "samples": len(sm), "source": self.how}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def ncu_traffic(precision):
    """dram__bytes_read.sum + dram__bytes_write.sum per conv_tc_kernel launch (average over the launches of one
    pass) from the committed ncu capture of the same workload, or None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "r2_conv_tc_dram_%s_b8.json" % precision)     # this round's capture first
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r1_conv_tc_dram_%s_b8.json" % precision)
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    return {"bytes_per_launch_avg": d["dram_bytes_total"] / d["launches"], "launches": d["launches"],
            "source": "profiles/" + os.path.basename(p)}


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the whole machine and oversubscribes a quota-limited container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def cpu_oracle_fps(n_frames, threads):
    """Times the CPU oracle (the port of the reference's TF graph) on `n_frames` 720x1280 frames."""
    import torch
    torch.set_num_threads(threads)
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from oracle import frcnn      # cpu_baseline / reference arm: the one place bench.py executes oracle/
    cfg = make_config()
    Wt = synth_weights(cfg, 1234)
    # the batch graph (Mask_RCNN_FPN_multi semantics, the workload both arms name), one frame per call
    frcnn.forward_multi(cfg, Wt, [synth_frame(H, W, 99).astype(np.float32)])           # warm-up
    t0 = time.perf_counter()
    for i in range(n_frames):
        frcnn.forward_multi(cfg, Wt, [synth_frame(H, W, i).astype(np.float32)])
    dt = time.perf_counter() - t0
    return n_frames / dt, dt


def stream_record(cfg, device, precision, n_frames=48, opt_in=False):
    """BASELINE configs[0] / [3] shape of work: ONE video stream, batch 1, the per-frame loop of
    obj_detect_tracking.py:597-696 -- Session.run (upload of the float32 frame, pass, download of boxes / probs / labels /
    box features) -> create_obj_infos -> pre-tracker NMS -> Tracker.predict / update with the GPU appearance metric.
    Every class is tracked (up to 100 objects per frame: the stress case).  Returns ms per stage and FPS per stream.
    opt_in=True: the two boundary extensions of INTEGRATION.md 2d / 2e -- the frame crosses PCIe as uint8 (what the decoder
    produces; the reference casts to float32 on the host first) and `fpn_box_feat` comes back mean-pooled over the 7x7 grid
    ([R,256], feat_mode 1: the mean create_obj_infos would take on the host)."""
    from object_detection_tracking_b200.backend import Session, get_model
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from object_detection_tracking_b200.tracking import (GpuNearestNeighborDistanceMetric, Tracker, create_obj_infos,
                                                         non_max_suppression)
    model = get_model(cfg, gpuid=device, precision=precision, input_dtype="uint8" if opt_in else "float32",
                      feat_mode=1 if opt_in else 0)
    model.set_weights(synth_weights(cfg, 1234))
    sess = Session()
    id2class = {i: "class%d" % i for i in range(1, cfg.num_class)}
    tracked = list(id2class.values())
    tracker = Tracker(GpuNearestNeighborDistanceMetric("cosine", 0.5, 5, device=device, precision=precision),
                      max_iou_distance=0.5, max_age=60, n_init=1, device=device, precision=precision)
    # a video: the same scene drifting by a few pixels per frame (np.roll of a synthetic frame)
    base = synth_frame(H, W, seed=321, n_rects=12).astype(np.uint8 if opt_in else np.float32)
    frames = [np.ascontiguousarray(np.roll(base, (2 * f, 3 * f), axis=(0, 1))) for f in range(8)]
    t_det = t_glue = t_assoc = 0.0
    n_obj = 0
    kept = []                     # the tracker inputs of the timed frames (for the reference-loop leg of cpu_baseline)
    fetches = [model.final_boxes, model.final_labels, model.final_probs, model.fpn_box_feat]
    for f in range(n_frames + 4):
        a = time.perf_counter()
        boxes, labels, probs, feats = sess.run(fetches, feed_dict=model.get_feed_dict_forward(frames[f % 8]))
        b = time.perf_counter()
        dets = create_obj_infos(f, boxes, probs, labels, feats, id2class, tracked, 0.0, 0, 1.0)
        if dets:
            keep = non_max_suppression(np.array([d.tlwh for d in dets]), 0.85, np.array([d.confidence for d in dets]))
            dets = [dets[i] for i in keep]
        c = time.perf_counter()
        tracker.predict()
        tracker.update(dets)
        live = [t for t in tracker.tracks if t.is_confirmed() and t.time_since_update <= 1]
        d = time.perf_counter()
        if f >= 4:                    # first frames: graph capture, workspace growth
            t_det += b - a; t_glue += c - b; t_assoc += d - c; n_obj += len(dets)
        kept.append([(x.tlwh.copy(), x.confidence, x.feature.copy()) for x in dets])
    tracker.close()
    total = t_det + t_glue + t_assoc
    return {"what": "one stream, batch 1: Session.run -> create_obj_infos -> NMS -> Tracker.predict/update (GPU cosine metric)"
                    + ("; uint8 frame in, pooled [R,256] features out" if opt_in else "; float32 frame in, [R,256,7,7] features out (reference semantics)"),
            "frames": n_frames, "objects_per_frame": n_obj / n_frames, "detect_ms": t_det / n_frames * 1e3,
            "glue_ms": t_glue / n_frames * 1e3, "associate_ms": t_assoc / n_frames * 1e3,
            "fps_per_stream": n_frames / total, "live_tracks_last_frame": len(live),
            "timing": "host clock around synchronous calls (each call ends with a device sync)", "_dets": kept}


def dump_outputs(det, out_dir):
    """Writes the results the last timed pass left in the context -- what detect_device hands a caller that passes output
    buffers -- as out_dir/<name>.npy: boxes [B,R,4], probs [B,R] and the box features [B*R,256,7,7] in float32, labels
    [B,R] and valid [B] (detections per frame) as float64.  The frames and weights are seeded, so two builds run with the
    same arguments can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    shapes = det.alloc_outputs(feat_mode=0)
    for name, stage in (("boxes", "final_boxes"), ("probs", "final_probs"), ("labels", "final_labels"),
                        ("valid", "final_count"), ("feat", "fpn_box_feat")):
        a = det.get_stage(stage).reshape(shapes[name].shape)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def reference_assoc_ms(dets_per_frame):
    """The reference's own association loop (deep_sort/tracker.py:57-138 restated in oracle/deepsort.py, numpy metric) on the
    detections the stream record fed to the native tracker: ms per frame on the host (part of cpu_baseline)."""
    from oracle import deepsort, nn_matching
    trk = deepsort.Tracker(nn_matching.NearestNeighborDistanceMetric("cosine", 0.5, 5))
    t0 = time.perf_counter()
    for dets in dets_per_frame:
        trk.predict()
        trk.update([deepsort.Detection(t, c, f) for t, c, f in dets])
    return (time.perf_counter() - t0) / max(1, len(dets_per_frame)) * 1e3


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = min(usable_cores(), 32)   # the conv stack stops scaling (and oversubscribes) beyond ~32 threads
    frames_per_step = 1
    import torch
    torch.set_num_threads(threads)
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from oracle import frcnn
    cfg = make_config()
    Wt = synth_weights(cfg, 1234)
    frames = [synth_frame(H, W, i).astype(np.float32) for i in range(4)]
    for i in range(args.warmup):
        frcnn.forward_multi(cfg, Wt, [frames[i % 4]])        # the batch graph's semantics, one frame per step
    t0 = time.perf_counter()
    for i in range(args.steps):
        frcnn.forward_multi(cfg, Wt, [frames[i % 4]])
    dt = time.perf_counter() - t0
    fps = args.steps * frames_per_step / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, args.precision, args.input_dtype),
            "arith": "float32 on the host CPU (PyTorch port of the reference TF graph), 1 frame per step",
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": "%d steps x 1 frame 720x1280 through the CPU oracle (PyTorch fp32 port of "
                                       "the reference TF graph; TensorFlow is not installable here)" % args.steps},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="split", choices=["split", "fp16"])
    ap.add_argument("--input-dtype", default="float32", choices=["float32", "uint8"],
                    help="frame dtype at the boundary: float32 = the reference placeholder (models.py:283), uint8 = decoder output")
    ap.add_argument("--cpu-frames", type=int, default=5, help="frames in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-json", default="", help="write the per-layer roofline table here")
    ap.add_argument("--single-semantics", action="store_true", help="batch of 8 through the single-image graph semantics")
    ap.add_argument("--sustained-seconds", type=float, default=5.0, help="length of the sustained replay record (0 = skip)")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-1 detect+track stream record")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0; about 40 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.engine import Detector
    from object_detection_tracking_b200.synth import synth_frame, synth_weights

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = make_config()
    # configs[1] is the reference's batch graph (Mask_RCNN_FPN_multi: combined NMS, zero-padded level merge, models.py:2058-2409)
    det = Detector(cfg, BATCH, H, W, device=local_rank, input_dtype=args.input_dtype, precision=args.precision,
                   use_cuda_graph=True, multi_semantics=not args.single_semantics)
    det.load_weights(synth_weights(cfg, 1234))
    # 4 distinct batches of synthetic frames (seeded per rank), resident on device and in pinned host memory
    np_dt = np.float32 if args.input_dtype == "float32" else np.uint8
    nb = 4 if args.input_dtype == "float32" else 8            # rotating input set larger than the 126 MB L2
    host = [torch.from_numpy(np.stack([synth_frame(H, W, seed=1000 * rank + 8 * j + i) for i in range(BATCH)])
                             .astype(np_dt)).pin_memory() for j in range(nb)]
    dev = [h.cuda(local_rank) for h in host]
    outs = det.alloc_outputs(feat_mode=0, pinned=True)

    # ---------------- device-resident throughput ----------------
    for i in range(args.warmup):
        det.detect_device(dev[i % nb], None, sync=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ev0 = torch.cuda.Event(enable_timing=True)   # recorded on torch's stream; the pass runs on the ctx stream and
    t0 = time.perf_counter()                     # is fenced by sync=True below, so wall-clock + device sync is exact
    for i in range(args.steps):
        det.detect_device(dev[i % nb], None, sync=(i == args.steps - 1))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    barrier()
    sampler.stop.set()
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(det, args.dump_outputs)     # before the records below run the context again
    # ---------------- sustained: the same graph replayed for >= 5 s (what the board settles at under its power cap) ----------------
    sustained = None
    if args.sustained_seconds > 0:
        s2 = ClockSampler(local_rank)
        s2.start()
        barrier()
        n_s, t_s = 0, time.perf_counter()
        while True:
            for _ in range(16):
                det.detect_device(dev[n_s % nb], None, sync=False)
                n_s += 1
            det.detect_device(dev[n_s % nb], None, sync=True)
            n_s += 1
            if time.perf_counter() - t_s >= args.sustained_seconds:
                break
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t_s
        s2.stop.set()
        s2.join(timeout=2)
        sustained = {"seconds": dt_s, "steps": n_s, "clocks": s2.summary(), "dt": dt_s}
    # device-side time of one steady-state pass from CUDA events on the launching (context) stream
    det.run_phases(255)
    phase_ms = det.phase_times()

    # ---------------- end to end through the host-buffer C-ABI calls ----------------
    # (a) one synchronous b2_detect_host per step (what Session.run does): upload, pass, download back to back
    for i in range(2):
        det.detect_host(host[i % nb], outs)
    barrier()
    t1 = time.perf_counter()
    for i in range(args.steps):
        det.detect_host(host[i % nb], outs)
    torch.cuda.synchronize()
    dt_sync = time.perf_counter() - t1
    barrier()
    # (b) the streaming pair b2_submit_host / b2_wait with two slots (queue-fed drivers): every step still uploads its
    # frames from pinned host memory and downloads all outputs inside the timed region; the upload of step i+1 overlaps
    # the pass of step i
    outs2 = [outs, det.alloc_outputs(feat_mode=0, pinned=True)]
    det.submit_host(host[0], outs2[0], 0)
    det.wait(0)
    barrier()
    t1 = time.perf_counter()
    det.submit_host(host[0], outs2[0], 0)
    for i in range(1, args.steps):
        det.submit_host(host[i % nb], outs2[i & 1], i & 1)
        det.wait((i - 1) & 1)
    det.wait((args.steps - 1) & 1)
    torch.cuda.synchronize()
    dt_e2e = time.perf_counter() - t1
    barrier()

    from object_detection_tracking_b200 import replicas
    dt, dt_e2e, dt_sync = replicas.max_over_ranks([dt, dt_e2e, dt_sync], device="cuda")     # slowest rank bounds the job
    if sustained is not None:
        (dts,) = replicas.max_over_ranks([sustained["dt"] / sustained["steps"]], device="cuda")
        sustained = {"value": replicas.aggregate_fps(BATCH, dts, world), "unit": "frames/s", "seconds": sustained["seconds"],
                     "steps_rank0": sustained["steps"], "ms_per_step": dts * 1e3, "clocks": sustained["clocks"]}
    stream = stream_opt = None
    if not args.no_stream and rank == 0:
        stream = stream_record(cfg, local_rank, args.precision)
        stream_opt = stream_record(cfg, local_rank, args.precision, opt_in=True)
        stream_opt.pop("_dets", None)
    value = replicas.aggregate_fps(args.steps * BATCH, dt, world)
    e2e_value = replicas.aggregate_fps(args.steps * BATCH, dt_e2e, world)
    h2d = host[0].numel() * host[0].element_size()
    d2h = sum(v.numel() * v.element_size() for v in outs.values())

    if rank == 0:
        # ---------------- roofline of the dominant kernel (tcgen05 conv), live CUDA-event timing ----------------
        prof = det.profile_steps(reps=3)
        conv = [p for p in prof if p["kind"] == 0]
        conv_ms = sum(p["ms"] for p in conv)
        conv_flops = sum(p["flops"] for p in conv)
        total_ms = sum(p["ms"] for p in prof)
        peaks, peak_src = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        achieved_tf = conv_flops / (conv_ms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 implicit GEMM, %d launches/step)" % len(conv),
                    "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                    "peak_source": peak_src + ", fp16/bf16 dense sustained",
                    "algorithmic_gflop_per_launch_avg": conv_flops / len(conv) / 1e9,
                    "avg_launch_ms": conv_ms / len(conv), "share_of_step": conv_ms / total_ms,
                    "mma_flop_multiplier": 3 if args.precision == "split" else 1,
                    "tensor_pipe_work_frac": achieved_tf * (3 if args.precision == "split" else 1) / peak_tf,
                    "traffic": ncu_traffic(args.precision),
                    # the timed pass forks the backbone / FPN / RPN-head phases over two streams (half-batch launches
                    # that overlap each other's tails); avg_launch_ms above is the serial full-batch launch
                    "conv_tflops_over_whole_step": conv_flops / (dt / args.steps) / 1e12}
        if args.profile_json:
            with open(args.profile_json, "w") as f:
                json.dump({"precision": args.precision, "batch": BATCH, "steps": prof}, f, indent=1)
        cpu = None
        if not args.no_cpu_baseline:
            threads = min(usable_cores(), 32)
            fps, secs = cpu_oracle_fps(args.cpu_frames, threads)
            cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                   "sample": "%d frames 720x1280 (batch 1) through the CPU oracle in %.1f s" % (args.cpu_frames, secs)}
            if stream is not None:
                cpu["associate_ms_per_frame_reference_loop"] = reference_assoc_ms(stream["_dets"])
        if stream is not None:
            stream.pop("_dets", None)
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "f16x2-split (fp32-equivalent products, fp32 accumulate)" if args.precision == "split"
                else "f16 (fp32 accumulate)",
                "data": "synthetic", "config": workload_config(world, args.precision, args.input_dtype),
                "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": dt_e2e / args.steps * 1e3,
                        "api": "b2_submit_host/b2_wait (2 slots, pinned %s frames in, all outputs out, every step)" % args.input_dtype,
                        "sync_call_value": replicas.aggregate_fps(args.steps * BATCH, dt_sync, world)},
                "gpu_launches": det.kernel_launches() * args.steps,
                "clocks": sampler.summary(), "roofline": roofline, "cpu_baseline": cpu,
                "phase_ms": phase_ms, "sustained": sustained, "stream_c1": stream, "stream_c1_uint8_pooled": stream_opt}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()              # rank 0 is the only one with the stream / cpu_baseline legs: the others wait for it
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
