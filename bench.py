#!/usr/bin/env python
"""Benchmark of the FastMOT per-frame hot path on B200 (BASELINE.json metric: frames/sec/stream @1080p, 200 tracks).

    python bench.py --gpus N --steps K --warmup W [--config 3] [--repeats R] [--dump-outputs DIR]   # our arm
    python bench.py --impl reference --steps K --warmup W [--config 3]         # reference CPU arm (host cores)

A "step" is one `MOT.step(frame)` on the next 1920x1080 frame of a deterministic synthetic stream.  `--config`
selects the BASELINE.json configuration (default 3 = configs[2], the one the metric is quoted on):
    1  configs[0]: 64 tracks, Kalman warp/predict/update + cost matrix + Hungarian only (KLT bypassed, no nets)
    2  configs[1]: YOLOv4-tiny 416 + OSNet x0.25, detector every frame, 50 tracks
    3  configs[2]: YOLOv4-csp 640 letterbox + OSNet x1.0, KLT on, detector every 5th frame, 200 tracks
    4  configs[3]: 70 overlapping objects, YOLOv4-p5 (896 as in the reference; --p5-input 1280), full association
Weights are synthetic (no trained weights offline), so the detector's OUTPUT rows are replaced by the scripted
ground-truth boxes AFTER the whole detector pipeline (letterbox, conv stack, decode, DIoU-NMS) has run at full cost --
random weights cannot detect, and the tracker must see the tracks.  Everything else is real data flow: ReID crops come
from the frame, OSNet embeddings feed the association kernels.

Timing: W warm-up steps (at least two detector periods after init; the conv engines are additionally replayed 3 times
at build), then R windows of exactly K steps (R = 1 by default, so K steps are timed), each bracketed by barrier +
synchronize, CUDA events on the launching stream, max over ranks; the line reports the MEDIAN window (`repeats` holds
min / max).
`value`  : frames already resident in HBM (all distinct; their total size is in `config.l2`) when the timed region
           starts.
`e2e`    : the same steps through the public API with frames in pinned HOST memory (6.2 MB H2D inside every step,
           track ids / boxes read back every step; bytes counted from the arrays actually copied).
`roofline_stages`: a third pass with per-stage CUDA events (fastmot_b200/stagetime.py) -> ms per call, algorithmic
           bytes / flops (SURVEY.md 8d figures), fraction of the measured peak or "latency" for the serial stages.

--dump-outputs DIR writes what the caller holds after the last timed step of the `value` pass (rank 0's stream): the
visible tracks' ids, boxes, labels, Kalman mean / covariance and running-mean ReID embedding, one DIR/<name>.npy each.
The stream, the scripted detections and the synthetic weights are seeded, so two builds run with the same arguments
can be compared array by array.
"""
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

METRIC = "frames/sec/stream @1080p, 200 tracks"

CONFIGS = {
    1: dict(workload="configs[0]: 64 tracks / 64 detections, Kalman warp+predict+update, cost matrix, Hungarian only "
                     "(KLT bypassed with the scripted boxes, no nets), update every step",
            kind="assoc", n=64, skip=1),
    2: dict(workload="configs[1]: single 1080p stream per GPU, YOLOv4-tiny 416 + OSNet x0.25, KLT on, detector every "
                     "frame, 50 tracks",
            kind="mot", yolo="YOLOv4Tiny", reid="OSNet025", n=50, skip=1),
    3: dict(workload="configs[2]: single 1080p stream per GPU, YOLOv4-csp 640 letterbox + OSNet x1.0, KLT on, "
                     "detector every 5th frame, 200 tracks",
            kind="mot", yolo="YOLOv4CSP", reid="OSNet10", n=200, skip=5),
    4: dict(workload="configs[3]: 70 overlapping objects (MOT17-03-like density), YOLOv4-p5 letterbox, DIoU-NMS, full "
                     "association, detector every 5th frame",
            kind="mot", yolo="YOLOv4P5", reid="OSNet10", n=70, skip=5, overlap=True, synth_head_gain=0.015),
}


def _cfg(c, args):
    from types import SimpleNamespace as NS
    from fastmot_b200.config import default_tracker_cfg
    yolo = c["yolo"]
    if yolo == "YOLOv4P5" and args.p5_input == 1280:
        yolo = "YOLOv4P5_1280"
    return dict(detector_type='YOLO', detector_frame_skip=c["skip"], class_ids=(0,),
                yolo_detector_cfg=NS(model=yolo, conf_thresh=0.25, nms_thresh=0.5, max_area=800000,
                                     min_aspect_ratio=1.2),
                feature_extractor_cfgs=(NS(model=c["reid"], batch_size=16),),
                tracker_cfg=NS(**default_tracker_cfg()))


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def track_outputs(tracks, feat_dim):
    """What a caller of MOT.step / MultiTracker reads from the visible tracks, as float32 / float64 arrays."""
    tracks = list(tracks)
    n = len(tracks)
    states = [t.state for t in tracks]
    feats = [t.avg_feat() for t in tracks]
    return {
        "track_ids": np.array([t.trk_id for t in tracks], np.float64),
        "track_tlbr": np.array([t.tlbr for t in tracks], np.float64).reshape(n, 4),
        "track_label": np.array([t.label for t in tracks], np.float64),
        "track_mean": np.array([m for m, _ in states], np.float64).reshape(n, 8),
        "track_cov": np.array([c for _, c in states], np.float64).reshape(n, 8, 8),
        "track_feature": np.array([np.zeros(feat_dim, np.float32) if f is None else f for f in feats],
                                  np.float32).reshape(n, feat_dim),
    }


def dump_outputs(arrays, out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_scene(c, seed):
    from fastmot_b200.synth import SyntheticScene
    # objects bounce inside their grid cell (+-16 px): the stream holds its tracks for any number of steps
    return SyntheticScene(c["n"], seed=seed, label=0, dropout_frames=(), bounce_radius=16,
                          overlap=bool(c.get("overlap")))


def det_override(scene, upto=0):
    """frame id -> scripted detections.  The rows for frames [0, upto) are generated up front: producing the synthetic
    ground truth is the harness' job, not part of the measured step."""
    from fastmot_b200.detector import DET_DTYPE
    cache = {}

    def make(t):
        tl, lb, cf, _ = scene.detections(t)
        d = np.zeros(len(tl), DET_DTYPE)
        d['tlbr'], d['label'], d['conf'] = tl, lb, cf
        return d.view(np.recarray)

    for t in range(upto):
        cache[t] = make(t)

    def f(t):
        d = cache.get(t)
        return make(t) if d is None else d.copy()
    return f


def reduce_max_ms(ms, world, device):
    """Timing of a multi-rank run = max over ranks (one all_reduce on the given device; NCCL on GPUs, gloo in the
    CPU test)."""
    if world <= 1:
        return float(ms)
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(ms)], device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def pin_rank_to_numa(local):
    """One process per GPU: keep the launching thread on the cores of the GPU's NUMA node (the tracker is
    launch-bound; cross-socket launches showed up as scaling jitter)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:00.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = []
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids)
        return node
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------------------
STAGE_MODEL = {
    # stage: (bound, algorithmic bytes per call as f(cfg) or None, note)     -- SURVEY.md 8(d)
    "preproc": ("hbm", lambda c, m: 1920 * 1080 * 3 + 3 * m["in_h"] * m["in_w"] * 2, "frame read + network input write"),
    "decode+nms": ("latency", lambda c, m: m["cand"] * 12 + m["cand"] * 28, "K0 candidates, mask K^2/8"),
    "crops": ("hbm", lambda c, m: c["n"] * (18e3 + 3 * 256 * 128 * 2), "crop reads + fp16 crops"),
    "klt-image": ("hbm", lambda c, m: 6.22e6 + 2.07e6 + 0.52e6 + 2 * 2 * 0.69e6 + 2.76e6, "gray, 0.5x, 0.1x, pyramid, derivs"),
    "keypoints": ("latency", lambda c, m: 1.2e6, "ROI corner detection + FAST on 192x108"),
    "lk": ("latency", lambda c, m: 30e6, "L2-resident pyramid traffic, ~13k points x 6 levels"),
    "ransac": ("latency", lambda c, m: 16.0 * 13000, "P x 16 B"),
    "kalman": ("latency", lambda c, m: c["n"] * 1208.0, "T x (2 x 576 + 32 + 72) B"),
    "cost": ("latency", lambda c, m: 2 * c["n"] * 2048.0 + c["n"] * c["n"] * 8.0, "(T + D) x 2 KB + T x D x 8 B"),
    "lsa": ("latency", lambda c, m: c["n"] * c["n"] * 8.0, "T x D x 8 B"),
    "cost+lsa": ("latency", lambda c, m: 2 * c["n"] * 2048.0 + c["n"] * c["n"] * 16.0, "fused cascade"),
    "feature-update": ("latency", lambda c, m: c["n"] * 512 * 4 * 3.0, "running mean of embeddings"),
}


def stage_rooflines(stage_ms, conv, c, meta, peaks, steps):
    bw, tf = peaks.get("hbm_gbs"), peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    out = []
    for name in ("yolo", "osnet"):
        calls = conv.get(name + "_calls", 0)
        if not calls:
            continue
        ms = conv[name + "_ms"] / calls
        fl, by = conv[name + "_flops"] / calls, conv[name + "_bytes"] / calls
        ent = {"stage": name, "ms_per_call": round(ms, 4), "calls": calls,
               "ms_per_step": round(conv[name + "_ms"] / steps, 4), "flops": fl, "bytes": by,
               "tflops": round(fl / ms / 1e9, 2), "gbs": round(by / ms / 1e6, 1),
               "frac_tensor": round(fl / ms / 1e9 / tf, 4) if tf else None,
               "frac_hbm": round(by / ms / 1e6 / bw, 4) if bw else None,
               "bound": "tensor" if name == "yolo" else "hbm"}
        ent["frac"] = ent["frac_tensor"] if ent["bound"] == "tensor" else ent["frac_hbm"]
        out.append(ent)
    for name, (tot, calls) in sorted(stage_ms.items()):
        bound, fbytes, note = STAGE_MODEL.get(name, ("latency", None, ""))
        ms = tot / max(calls, 1)
        by = float(fbytes(c, meta)) if fbytes else None
        ent = {"stage": name, "ms_per_call": round(ms, 4), "calls": calls, "ms_per_step": round(tot / steps, 4),
               "bytes": by, "bound": bound, "note": note}
        if by and ms > 0:
            ent["gbs"] = round(by / ms / 1e6, 2)
            ent["frac_hbm"] = round(by / ms / 1e6 / bw, 5) if bw else None
        ent["frac"] = ent.get("frac_hbm") if bound == "hbm" else "latency"
        out.append(ent)
    return out


# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    numa = pin_rank_to_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from fastmot_b200 import _lib, stagetime
    from fastmot_b200 import engine as eng_mod
    _lib.require_device()
    c = CONFIGS[args.config]
    # the first detector periods after init are transient (the association update at frame `skip` is the first one and
    # the tracks have no history yet): the warm-up always covers two periods, so the timed window is steady state
    K, W, R = args.steps, max(args.warmup, 2 * c["skip"]), args.repeats
    sampler = ClockSampler(local)
    sampler.start()          # nvidia-smi needs ~1 s to start and slows launches meanwhile: start before the model build
    dev = torch.device("cuda", local)
    scene = make_scene(c, rank)
    total = W + R * K
    frames = [scene.frame(t) for t in range(total)] if c["kind"] == "mot" else [None] * total

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if c["kind"] == "mot":
        from fastmot_b200 import MOT
        # Synthetic (random) weights fire on noise.  In the deep models the head logits of real frames have a far
        # larger variance than the calibration input gave them, so nearly half of the anchors would pass conf_thresh;
        # `synth_head_gain` scales the synthetic head weights so that the candidate count stays in the range the
        # workload describes (K ~ 10 x D .. a few thousand; chosen with the CPU oracle, which reproduces the GPU's
        # count) and inside the detector's key capacity.  The gain and the count are reported in `config`.
        g0 = float(c.get("synth_head_gain", 1.0))
        for gain in [g0] + [g for g in (0.25, 0.06, 0.015, 0.004) if g < g0]:
            os.environ["FM_SYNTH_HEAD_GAIN"] = str(gain)
            mot = MOT(scene.size, detections_override=det_override(scene, total), **_cfg(c, args))
            try:
                mot.reset(1 / 30.)
                mot.step(frames[0])
            except RuntimeError as e:
                if "key_cap" not in str(e):
                    raise
                continue
            if mot.detector.last_num_candidates <= mot.detector.key_cap // 2:
                break
        else:
            raise RuntimeError("no synthetic head gain keeps the candidate count inside key_cap")
        mot.extractors[0]._engine(c["n"])      # build + warm the ReID engine outside the timed region
        for e in [mot.detector.backend] + list(mot.extractors[0]._engines.values()):
            e.warm(3)

        def reset():
            mot.reset(1 / 30.)

        def step(f):
            mot.step(f)
            return sum(1 for _ in mot.visible_tracks())

        def visible():
            return mot.visible_tracks()
        tracker = mot.tracker
    else:
        from fastmot_b200 import MultiTracker
        from fastmot_b200.config import default_tracker_cfg
        dets = det_override(scene, total)
        trk = MultiTracker(scene.size, 'cosine', **{k: v for k, v in default_tracker_cfg().items() if k != 'flow_cfg'})
        state = {"t": 0}

        def reset():
            trk.reset(1 / 30.)
            state["t"] = 0

        def step(_):
            t = state["t"]
            d = dets(t)
            if t == 0:
                trk.init(None, d)
            else:
                ids = scene.detections(t)[3]
                klt = {tid: tr.tlbr for tid, tr in trk.tracks.items()}      # KLT bypass: previous boxes as flow result
                trk.inject_flow(klt, np.eye(3), {tid: 1.0 for tid in klt})
                trk.compute_flow(None)
                trk.apply_kalman()
                trk.update(t, d, scene.embeddings(ids, t))
            state["t"] = t + 1
            return sum(1 for v in trk.tracks.values() if v.confirmed and v.active)

        def visible():
            return (v for v in trk.tracks.values() if v.confirmed and v.active)
        tracker = trk

    def readback_bytes():
        return sum(t.tlbr.nbytes + 8 for t in visible())

    prof = eng_mod.enable_profiling()

    def run_pass(inputs, prefetch=False):
        """W warm-up steps, then R windows of K steps.  Returns per-window ms (max over ranks), per-step ms of the last
        window, visible tracks.  prefetch: MOT.prefetch(next frame) before every step (read-ahead upload stream)."""
        reset()
        pre = (lambda f: mot.prefetch(f)) if (prefetch and c["kind"] == "mot") else None
        for i, f in enumerate(inputs[:W]):
            if pre is not None:          # the first timed frame arrives prefetched, like every later one
                pre(inputs[i + 1])
            step(f)
        win_ms, step_ms, n_vis = [], [], 0
        for r in range(R):
            chunk = inputs[W + r * K: W + (r + 1) * K]
            barrier()
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
            evs[0].record()
            for i, f in enumerate(chunk):
                if pre is not None and W + r * K + i + 1 < len(inputs):
                    pre(inputs[W + r * K + i + 1])
                n_vis = step(f)
                evs[i + 1].record()
            barrier()
            win_ms.append(reduce_max_ms(evs[0].elapsed_time(evs[-1]), world, dev))
            step_ms = [(W + r * K + i, evs[i].elapsed_time(evs[i + 1])) for i in range(K)]
        return win_ms, step_ms, n_vis

    # ---- pass 1: frames resident in HBM ----
    dev_frames = [torch.as_tensor(f).to(dev) if f is not None else None for f in frames]
    prof.reset()
    sampler.rows.clear()
    launches0 = _lib.launch_count()
    win_dev, step_dev, n_vis = run_pass(dev_frames)
    launches = (_lib.launch_count() - launches0)
    conv = prof.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(track_outputs(visible(), tracker.pool.feat_dim), args.dump_outputs)
    # ---- pass 2: end to end from pinned host memory through the public API ----
    if c["kind"] == "mot":
        host_frames = [torch.as_tensor(f).pin_memory().numpy() for f in frames]
        h2d = int(frames[0].nbytes)
    else:
        host_frames, h2d = frames, int(scene.detections(0)[0].nbytes + 64 * 512 * 4)
    win_e2e, _, _ = run_pass(host_frames, prefetch=not args.no_prefetch)
    clocks = sampler.stop()          # over both timed passes: one window of K steps can be shorter than a sample
    d2h = int(readback_bytes())
    # ---- pass 3: per-stage CUDA events (not part of the timed numbers above) ----
    prof.reset()
    stagetime.enable()
    reset()
    for f in dev_frames[:W + K]:
        step(f)
    stage_ms = stagetime.collect()
    stagetime.disable()
    conv_stage = prof.summary()

    if rank == 0:
        peaks, peak_src = _peaks()
        med = float(np.median(win_dev))
        med_e2e = float(np.median(win_e2e))
        fps = world * K / (med / 1e3)
        fps_e2e = world * K / (med_e2e / 1e3)
        skip = c["skip"]
        det_steps = [ms for t, ms in step_dev if t % skip == 0]
        trk_steps = [ms for t, ms in step_dev if t % skip != 0]
        steps_per_launchcount = (W + R * K)
        meta = {"in_h": 0, "in_w": 0, "cand": 0}
        out = {
            "metric": METRIC, "value": round(fps, 2), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(med / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 conv (fp32 accumulate in TMEM; depthwise 3x3 taps in fp16), u8/fixed-point KLT, "
                     "fp64 Kalman/assignment",
            "data": f"synthetic 1920x1080 stream, {c['n']} moving textured objects, synthetic (seeded, BN-calibrated) "
                    "weights",
            "config": {"workload": c["workload"], "config_id": args.config, "streams": world,
                       "value_is": "aggregate over all streams (one stream per GPU); per-stream = value / n_gpus",
                       "parallelism": f"{world} independent streams, one per GPU, no collective",
                       "l2": (f"{W + R * K} distinct frames, 6.2 MB each: {(W + R * K) * 6.22:.0f} MB in total "
                              "(B200 L2: 126 MB)") if c["kind"] == "mot" else "no frames",
                       "detections": "scripted ground-truth boxes replace the detector output rows after the full "
                                     "detector pipeline ran (random weights cannot detect)",
                       "visible_tracks_last_step": int(n_vis), "conv_path": conv.get("conv_path"),
                       "synthetic_head_gain": (float(os.environ["FM_SYNTH_HEAD_GAIN"])
                                               if "FM_SYNTH_HEAD_GAIN" in os.environ else None),
                       "numa_node": numa},
            "repeats": {"windows": R, "ms_per_step_min": round(min(win_dev) / K, 4),
                        "ms_per_step_max": round(max(win_dev) / K, 4),
                        "ms_per_step_all": [round(w / K, 4) for w in win_dev]},
            "e2e": {"value": round(fps_e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                    "upload": "MOT.prefetch(next frame) before every step: the 6.2 MB copy of frame t+1 runs on an "
                              "upload stream under step t (inside the timed region)" if not args.no_prefetch
                              else "synchronous upload at the start of every step",
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(med_e2e / K, 4),
                    "ms_per_step_min": round(min(win_e2e) / K, 4), "ms_per_step_max": round(max(win_e2e) / K, 4)},
            "gpu_launches": int(round(launches * K / steps_per_launchcount)),
            "gpu_launches_note": "kernels per K-step window (counted over warm-up + all windows, scaled)",
            "clocks": clocks,
            "tracker_only": {"frames_per_s": round(1e3 / float(np.median(trk_steps)), 1) if trk_steps else None,
                             "ms_per_frame": round(float(np.median(trk_steps)), 4) if trk_steps else None,
                             "what": "median step without a detector pass (KLT + Kalman; the part the reference runs "
                                     "on its CPU every frame)"},
            "detector_frame_ms": round(float(np.median(det_steps)), 4) if det_steps else None,
        }
        if c["kind"] == "mot":
            eng = list(mot.extractors[0]._engines.values())[0]
            ih, iw = mot.detector.backend.inp.shape[:2]
            meta = {"in_h": int(ih), "in_w": int(iw), "cand": int(getattr(mot.detector, "last_num_candidates", 0))}
            out["config"]["detector_candidates_last_frame"] = meta["cand"]
            os_calls = max(conv.get("osnet_calls", 0), 1)
            os_ms = conv.get("osnet_ms", 0.0) / os_calls
            os_bytes = conv.get("osnet_bytes", 0.0) / os_calls
            os_gbs = os_bytes / os_ms / 1e6 if os_ms > 0 else 0.0
            traffic = None
            tp = os.path.join(ROOT, "profiles", "r02_osnet_traffic.json")
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get("osnet_forward_dram_bytes")
            peak_bw = peaks.get("hbm_gbs")
            peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
            os_fl = conv.get("osnet_flops", 0.0) / os_calls
            out["roofline"] = {
                "bound": "hbm", "achieved": round(os_gbs, 1), "peak": peak_bw, "unit": "GB/s",
                "frac": round(os_gbs / peak_bw, 4) if peak_bw else None, "traffic": traffic,
                "kernel": f"OSNet stack on {c['n']} crops: fused OSBlock kernels (osb_streams + osb_merge), stem, "
                          "transitions; algorithmic bytes = every fused kernel's input + output moved once",
                "peak_source": peak_src, "bytes_per_launch": os_bytes, "ms_per_launch": round(os_ms, 4),
                "tensor_view": {"tflops": round(os_fl / os_ms / 1e9, 2) if os_ms > 0 else None, "peak": peak_tf,
                                "frac": round(os_fl / os_ms / 1e9 / peak_tf, 4) if os_ms > 0 and peak_tf else None},
                "kernels_per_forward": int(eng.kernels_per_replay())}
            yl_calls = max(conv.get("yolo_calls", 0), 1)
            yl_ms = conv.get("yolo_ms", 0.0) / yl_calls
            yl_fl = conv.get("yolo_flops", 0.0) / yl_calls
            out["roofline_tensor"] = {
                "bound": "tensor", "achieved": round(yl_fl / yl_ms / 1e9, 2) if yl_ms > 0 else None, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": round(yl_fl / yl_ms / 1e9 / peak_tf, 4) if yl_ms > 0 and peak_tf else None,
                "kernel": "detector conv stack (implicit-GEMM tcgen05), batch 1", "ms_per_launch": round(yl_ms, 4),
                "yolo_tflops": round(yl_fl / yl_ms / 1e9, 2) if yl_ms > 0 else None}
        out["roofline_stages"] = stage_rooflines(stage_ms, conv_stage, c, meta, _peaks()[0], W + K)
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(args.config, args.cpu_steps, 1, args, with_nets=False)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
def cpu_baseline(config, steps, warmup, args, with_nets=True):
    """The reference's CPU path restated in oracle/ (kind "port": the reference is Python + TensorRT and cannot be
    installed here; its tracker path is pinned bit-identical to it), timed on the host cores: KLT via OpenCV, numpy
    Kalman / SciPy-equivalent assignment, cv2 crops, Numba-equivalent NMS.  `value` is the frame rate of THAT path with
    scripted detections and embeddings; the conv stacks never ran on the reference's CPU (TensorRT), so their fp32
    PyTorch-CPU time is reported separately and labelled."""
    import torch
    import cv2
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    cv2.setNumThreads(ncpu)
    from oracle.pipeline import OraclePipeline
    c = CONFIGS[config]
    scene = make_scene(c, 0)
    frames = [scene.frame(t) if c["kind"] == "mot" else None for t in range(warmup + steps + 1)]
    d0 = det_override(scene)

    def ov(t):
        d = d0(t)
        return d.tlbr, d.label, d.conf
    kw = dict(frame_skip=c["skip"], detections_override=ov)
    if c["kind"] == "mot":
        yolo = c["yolo"] + ("_1280" if c["yolo"] == "YOLOv4P5" and args.p5_input == 1280 else "")
        kw.update(yolo=yolo, reid=c["reid"])
    pipe = OraclePipeline(scene.size, run_nets=False, embeddings_override=lambda t, ids: scene.embeddings(ids, t),
                          scene_ids=lambda t: scene.detections(t)[3], klt=c["kind"] == "mot", **kw)
    for f in frames[:warmup + 1]:          # frame 0 (init) + warm-up
        pipe.step(f)
    pipe.stage_s.clear()
    t0 = time.perf_counter()
    for f in frames[warmup + 1:]:
        pipe.step(f)
    dt = time.perf_counter() - t0
    n = steps
    out = {"value": round(n / dt, 4), "unit": "frames/s", "cores": ncpu, "kind": "port",
           "threads": {"torch": torch.get_num_threads(), "opencv": cv2.getNumThreads()},
           "sample": f"{n} steps after {warmup} warm-up steps of the same stream: tracker path on the CPU (letterbox "
                     "resize, NMS filter, ReID crops, KLT via OpenCV, Kalman, cost matrices, assignment) with scripted "
                     "detections and embeddings; conv stacks excluded (the reference runs them in TensorRT)",
           "stages_s": {k: round(v, 4) for k, v in pipe.stage_s.items()}}
    if with_nets and c["kind"] == "mot":
        t0 = time.perf_counter()
        nets_s = pipe.time_nets(frames[0], scene.detections(0)[0])
        out["conv_stacks_fp32_torch_cpu"] = {"not_the_reference": True, "seconds_per_detector_frame": nets_s,
                                            "measured_s": round(time.perf_counter() - t0, 2)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    steps, warmup = args.steps, args.warmup
    cap = 60 if c["kind"] == "mot" else 400       # bounded sample: each CPU step costs 30-300 ms
    capped = steps > cap
    steps = min(steps, cap)
    cb = cpu_baseline(args.config, steps, min(warmup, 5), args, with_nets=not args.no_nets)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": steps, "warmup": min(warmup, 5),
           "ms_per_step": round(1e3 / cb["value"], 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8/fixed-point KLT (OpenCV), fp64 Kalman/assignment", "data": "synthetic",
           "config": {"workload": c["workload"], "config_id": args.config,
                      "arm": "reference CPU path (oracle port, pinned bit-identical to the reference's tracker) on the "
                             "host cores; ONE stream on rank 0 regardless of --gpus",
                      "requested_steps": args.steps, "requested_warmup": args.warmup,
                      "steps_capped": capped, "sample": cb["sample"]},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=1, help="timed windows of --steps steps each")
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--p5-input", type=int, default=896, choices=[896, 1280])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-nets", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the visible tracks after the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
