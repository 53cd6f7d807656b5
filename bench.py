#!/usr/bin/env python
"""bench.py — post-backbone detection images/s @1024^2 on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--check] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[1], SURVEY.md §8d cfg 2): Mask R-CNN COCO-shape inference heads, 1024x1024,
261,888 anchors, 6000 pre-NMS -> 1000 proposals, ROIAlign 7x7 and 14x14 over P2-P5 (D=256), 81 classes, batch 2 per
GPU (weak scaling: every rank owns its own 2 images; N>1 adds one all-gather of the detections).

One step = Proposals -> { DetectionLayer (synthetic head outputs) || PyramidROIAlign 7x7 (1000 ROIs/img) }
           -> PyramidROIAlign 14x14 (1000 ROIs/img)   [+ all_gather(detections) on the DetectionLayer branch when N>1]
           (DetectionLayer and the 7x7 ROIAlign both depend on the proposals only and run on two streams; the step ends
           when both branches and the 14x14 launch are done; the ROI processing order is computed once per step and
           shared by the two pooling calls).
Consecutive steps work on different images and share nothing: --lanes L (default 4) keeps L steps in flight (step i on
lane i % L: own streams, input set and outputs), so the latency-bound proposal front of one step runs underneath the
HBM-bound ROIAlign launches of the others. All K steps run between the two timing events.

Reported on ONE JSON line (rank 0):
  value        images/s with the inputs resident in HBM, CUDA events around exactly K steps, max over ranks
  e2e          the same step with every input copied from pinned HOST buffers inside the timed region (H2D into the
               buffers the layer classes read) and the detections read back (D2H) every step; next to it the bare
               concurrent-H2D ceiling of the same buffers on the same ranks
  roofline     the dominant kernel (the 14x14 ROIAlign launch, crop_rows_kernel): algorithmic bytes / CUDA-event
               duration, against MEASURED_PEAKS.json. Measured in a second timed pass of the same step with the steps
               issued one at a time (with_steps_in_flight = the same events inside the headline region, where the launch
               shares HBM and SMs with other steps); traffic = ncu DRAM bytes of the same build (profiles/ncu_traffic.json)
  cpu_baseline the CPU oracle (C restatement of the reference's algorithm, OpenMP) on the same workload, all host
               threads and one thread
  scaling_b64  BASELINE.json configs[4]: the same heads at GLOBAL batch 64 sharded 64/N images per GPU (strong scaling),
               every N, device-timed, max over ranks
  extra        (N=1) configs[2] training chain, configs[3] Faster R-CNN heads, the 100k-box NMS stress case - each with
               the CPU oracle timed beside it - the step time without CUDA graphs and with one step at a time
`--impl reference` times the CPU restatement alone on the same global batch (the reference itself is TF-1.x graph code;
TensorFlow is not installable in this image, see DESIGN.md) and prints the same line with "impl": "reference".
`--check` compares the gathered detections of every shard (headline and batch-64 runs) with the CPU oracle.
`--dump-outputs DIR` (rank 0) writes what the last timed step returned to its caller as float32 .npy files: detections
[B,100,6], proposals [B,1000,4] and pooled_7x7_sample / pooled_14x14_sample, the same DUMP_ROIS rows (a seeded choice)
of the two [1,B*1000,P,P,256] pooled tensors. With N > 1 the detections are the gathered batch of all ranks, while the
proposals and pooled samples are rank 0's own images. The inputs are seeded, so two builds run with the same arguments
can be compared file by file.
The bench writes nothing into the source tree (no bytecode either), so it also runs from a read-only checkout.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree for the project modules imported below

IMAGE = 1024
B_PER_GPU = 2
GLOBAL_B64 = int(os.environ.get("OD_BENCH_GLOBAL_B", "64"))   # BASELINE configs[4]: 64 (the override is a developer aid: the 8-images-per-GPU shape of N=8 on one GPU)
N_ROIS = 1000
N_CLASSES = 81
DEPTH = 256
DUMP_ROIS = 128                          # --dump-outputs: pooled ROIs kept of B*N_ROIS (32 MB for 7x7 + 14x14)
WINDOW_PX = [131, 0, 893, 1024]          # test_detection.ipynb window
WORKLOAD = ("maskrcnn-coco-heads-1024: 261888 anchors, 6000->1000 proposals, ROIAlign 7x7+14x14 over P2-P5 (D=256), "
            "81 classes, batch 2 per GPU")
METRIC = "post-backbone detection images/s @1024^2"


def shared_config(world: int) -> dict:
    """The `config` object both arms print (identical keys and values for the same N)."""
    return {"workload": WORKLOAD, "images_per_gpu": B_PER_GPU, "images_per_step": world * B_PER_GPU, "image": IMAGE,
            "anchors": 261888, "pre_nms": 6000, "post_nms": N_ROIS, "classes": N_CLASSES, "pool": "7x7+14x14", "depth": DEPTH}


# ----------------------------------------------------------------------------- synthetic inputs (SURVEY §8d cfg 2)
def synth_rpn_head(seed: int, B: int, A: int):
    """RPN outputs + head outputs of B images (host, numpy): fg prob ~ Beta(0.5, 4), deltas ~ N(0,1); head probs =
    softmax of N(0,3) logits with 20 % of the rows boosted on a random foreground class."""
    rs = np.random.RandomState(seed)
    f32 = np.float32
    fg = rs.beta(0.5, 4, size=(B, A)).astype(f32)
    probs = np.stack([f32(1) - fg, fg], axis=2).astype(f32)                      # [B,A,2] (bg,fg)
    bbox = rs.standard_normal(size=(B, A, 4)).astype(f32)                        # [B,A,4]
    logits = (rs.standard_normal(size=(B, N_ROIS, N_CLASSES)) * 3).astype(np.float64)
    rows = rs.random_sample((B, N_ROIS)) < 0.2
    cls = rs.randint(1, N_CLASSES, size=(B, N_ROIS))
    bi, ni = np.nonzero(rows)
    logits[bi, ni, cls[bi, ni]] += 12
    e = np.exp(logits - logits.max(-1, keepdims=True))
    hprobs = (e / e.sum(-1, keepdims=True)).astype(f32)                          # [B,N,C]
    hbbox = rs.standard_normal(size=(B, N_ROIS, N_CLASSES, 4)).astype(f32)       # [B,N,C,4]
    return dict(probs=probs, bbox=bbox, hprobs=hprobs, hbbox=hbbox)


def synth_inputs(seed: int, B: int, A: int):
    d = synth_rpn_head(seed, B, A)
    rs = np.random.RandomState(seed + 7919)
    d["fmaps"] = [rs.random_sample((B, s, s, DEPTH)).astype(np.float32) for s in (256, 128, 64, 32)]
    return d


def rois_log_uniform(seed: int, B: int, N: int, image=IMAGE, lo=16, hi=512):
    """Stand-alone ROIAlign recipe: sqrt(area) log-uniform [16,512] px, aspect log-uniform [0.5,2], centre uniform."""
    rs = np.random.RandomState(seed)
    s = np.exp(rs.uniform(np.log(lo), np.log(hi), size=(B, N)))
    r = np.exp(rs.uniform(np.log(0.5), np.log(2.0), size=(B, N)))
    h, w = s / np.sqrt(r), s * np.sqrt(r)
    cy, cx = rs.uniform(0, image, size=(B, N)), rs.uniform(0, image, size=(B, N))
    boxes = np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], axis=2)
    return (np.clip(boxes, 0, image - 1) / (image - 1)).astype(np.float32)


def roialign_algorithmic_bytes(rois: np.ndarray, levels: np.ndarray, P: int, D: int, sizes=(256, 128, 64, 32),
                               min_level=2) -> dict:
    """Algorithmic HBM bytes of one PyramidROIAlign launch (SURVEY §8d): the compulsory output N*P*P*D*4 plus
    U*D*4, U = number of DISTINCT feature-map pixels touched by any valid bilinear tap of any ROI of the same image
    (crop_and_resize grid: in = y1*(H-1) + i*(y2-y1)*(H-1)/(P-1), fp32; taps floor/ceil; out-of-range rows/cols
    read nothing). The smallest defensible figure, so it cannot flatter the kernel."""
    f32 = np.float32
    B, N = rois.shape[:2]
    out_bytes = B * N * P * P * D * 4
    U = 0
    for b in range(B):
        for li, S in enumerate(sizes):
            sel = levels[b] == (min_level + li)
            if not sel.any():
                continue
            r = rois[b][sel].astype(f32)
            Hm1 = f32(S - 1)
            grid = np.arange(P, dtype=f32)[None, :]
            taps = []
            for lo, hi in ((r[:, 0:1], r[:, 2:3]), (r[:, 1:2], r[:, 3:4])):
                if P > 1:
                    step = (hi - lo) * Hm1 / f32(P - 1)
                    pos = lo * Hm1 + grid * step
                else:
                    pos = (f32(0.5) * (lo + hi) * Hm1) + grid * f32(0)
                ok = (pos >= 0) & (pos <= Hm1)
                fl = np.where(ok, np.floor(pos), S).astype(np.int64)      # S = dummy slot for "no tap"
                ce = np.where(ok, np.ceil(pos), S).astype(np.int64)
                taps.append(np.concatenate([fl, ce], axis=1))            # [n,2P]
            mask = np.zeros((S + 1, S + 1), dtype=bool)
            mask[taps[0][:, :, None], taps[1][:, None, :]] = True
            U += int(mask[:S, :S].sum())
    return dict(out_bytes=out_bytes, unique_in_bytes=U * D * 4, total=out_bytes + U * D * 4)


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        for fields in (self.FIELDS, self.FIELDS.replace("clocks_event_reasons", "clocks_throttle_reasons")):
            try:
                self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={fields}",
                                              "--format=csv,noheader,nounits", "-lms", "20"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except OSError:
                self.proc = None
                return
            time.sleep(0.25)
            if self.proc.poll() is None:
                threading.Thread(target=self._pump, daemon=True).start()
                return
        self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], [], set(), []
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.lines]
        for l in rows:
            c = [x.strip() for x in l.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); smax.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_ncu_traffic(lib_hash: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of the 14x14 ROIAlign launch from the committed `ncu --set full`
    capture (profiles/ncu_traffic.json, written by tools/gpu/ncu_traffic.sh) - only if that capture was taken with the
    very library this run loads (same source hash); otherwise null."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        rec = json.load(open(path))
    except Exception:
        return None, "no ncu capture recorded"
    if rec.get("source_hash") != lib_hash:
        return None, f"recorded capture is of another build ({str(rec.get('source_hash'))[:12]})"
    return rec.get("roialign_p14_pipeline_bytes"), f"ncu --set full, {rec.get('capture')}"


# ----------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def omp_set_threads(n: int):
    try:    # libgomp may already be initialised with torchrun's OMP_NUM_THREADS=1
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(n))
    except OSError:
        pass


def cpu_step(oracle, conf, inp, anchors, win_norm):
    """The bench step on the CPU oracle: Proposals -> ROIAlign 7x7 -> DetectionLayer -> ROIAlign 14x14."""
    p = oracle.proposal_forward(inp["probs"], inp["bbox"], anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD)
    oracle.pyramid_roi_align(inp["fmaps"], p, IMAGE, IMAGE, 7, 7)
    det = oracle.detection_forward(p, inp["hprobs"], inp["hbbox"], win_norm, conf.BBOX_STD_DEV,
                                   conf.DETECTION_MIN_THRESHOLD, conf.DETECTION_NMS_THRESHOLD,
                                   conf.DETECTION_POST_NMS_INSTANCES)
    oracle.pyramid_roi_align(inp["fmaps"], p, IMAGE, IMAGE, 14, 14)
    return det


def cpu_detections(oracle, conf, inp, anchors, win_norm):
    """Proposals -> DetectionLayer only (what --check compares; no pyramid needed)."""
    p = oracle.proposal_forward(inp["probs"], inp["bbox"], anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD)
    return oracle.detection_forward(p, inp["hprobs"], inp["hbbox"], win_norm, conf.BBOX_STD_DEV,
                                    conf.DETECTION_MIN_THRESHOLD, conf.DETECTION_NMS_THRESHOLD,
                                    conf.DETECTION_POST_NMS_INSTANCES)


def cpu_setup(B, seed=1000, with_fmaps=True):
    import oracle
    from objectdetection_b200.config import config
    oracle.build()
    oracle.lib()
    omp_set_threads(cpu_threads())
    conf = config()
    shapes = oracle.get_resnet_stage_shapes(conf.RESNET_STRIDES, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    inp = synth_inputs(seed, B, anchors.shape[1]) if with_fmaps else synth_rpn_head(seed, B, anchors.shape[1])
    win = oracle.norm_boxes(np.array([WINDOW_PX] * B), (IMAGE, IMAGE))
    return oracle, conf, inp, anchors, win


def timed_reps(fn, budget_s, min_reps=2, max_reps=2000):
    fn()      # warm-up (page in, OpenMP pool)
    reps, t0 = 0, time.perf_counter()
    while reps < max_reps and (time.perf_counter() - t0 < budget_s or reps < min_reps):
        fn()
        reps += 1
    return reps, time.perf_counter() - t0


def run_cpu_baseline(budget_s=10.0):
    """The oracle port on the same workload (batch 2 per step): all host threads for ~budget_s, then one thread."""
    os.environ.setdefault("OMP_NUM_THREADS", str(cpu_threads()))
    oracle, conf, inp, anchors, win = cpu_setup(B_PER_GPU)
    reps, dt = timed_reps(lambda: cpu_step(oracle, conf, inp, anchors, win), budget_s)
    omp_set_threads(1)
    reps1, dt1 = timed_reps(lambda: cpu_step(oracle, conf, inp, anchors, win), 4.0, min_reps=2)
    omp_set_threads(cpu_threads())
    return {"value": reps * B_PER_GPU / dt, "unit": "images/s", "cores": cpu_threads(), "kind": "port",
            "sample": f"{reps} steps x {B_PER_GPU} images of the bench workload in {dt:.1f} s "
                      f"(oracle/odhead_oracle.c, OpenMP over rows/ROIs)",
            "value_1thread": reps1 * B_PER_GPU / dt1,
            "sample_1thread": f"{reps1} steps x {B_PER_GPU} images in {dt1:.1f} s, omp_set_num_threads(1)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(int(args.gpus), 1)
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host thread it can get
    os.environ["OMP_NUM_THREADS"] = str(cpu_threads())
    B = world * B_PER_GPU                          # the same global batch per step as the GPU arm at this N
    oracle, conf, inp, anchors, win = cpu_setup(B)
    t = time.perf_counter()
    cpu_step(oracle, conf, inp, anchors, win)
    first = time.perf_counter() - t
    # bounded sample: the whole --steps K --warmup W run must stay within a few minutes; a step that is too slow is cut
    # to a sub-batch of the same workload (throughput in images/s is what is reported either way)
    note = ""
    while first * (args.steps + args.warmup) > 170.0 and B > 1:
        B = max(B // 2, 1)
        first /= 2
        note = f" (step bounded to {B} of the {world * B_PER_GPU} images to fit the time budget)"
    if B != world * B_PER_GPU:
        inp = {k: ([f[:B] for f in v] if isinstance(v, list) else v[:B]) for k, v in inp.items()}
        anchors, win = anchors[:B], win[:B]
    for _ in range(max(args.warmup - 1, 0)):
        cpu_step(oracle, conf, inp, anchors, win)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(oracle, conf, inp, anchors, win)
    dt = time.perf_counter() - t0
    v = args.steps * B / dt
    cores = cpu_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(world),
        "device": "host CPU", "images_timed_per_step": B,
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps x {B} images{note}; CPU restatement of the reference's TF graph "
                                   f"(oracle/odhead_oracle.c, OpenMP, {cores} threads); TensorFlow itself is not "
                                   f"installable in this image"},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def pin_rank_to_gpu_cpus(local: int) -> dict:
    """CPU affinity of this rank = the CPUs NVML reports as local to its GPU (NUMA placement of the pinned staging
    buffers follows by first touch). Returns what was done, for the JSON line."""
    info = {"affinity": "unchanged"}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"affinity": f"{len(allowed)} CPUs local to GPU {local} ({allowed[0]}-{allowed[-1]})"}
        try:
            info["numa_node"] = pynvml.nvmlDeviceGetNumaNodeId(h)
        except Exception:
            pass
    except Exception as e:       # affinity is an optimisation, never a requirement
        info = {"affinity": f"unchanged ({type(e).__name__})"}
    return info


def run_ours(args):
    import torch
    import torch.distributed as dist

    from objectdetection_b200 import DetectionLayer, Proposals, _lib, utils
    from objectdetection_b200.config import config
    from objectdetection_b200.distributed import gather_detections
    from objectdetection_b200.maskrcnn import pyramid_roi_align, roi_processing_order

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (objectdetection_b200 has no CPU path; use --impl reference)")
    placement = pin_rank_to_gpu_cpus(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    conf = config()
    B = B_PER_GPU
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = utils.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE, device=dev)
    A = anchors.shape[1]
    window = np.array([WINDOW_PX] * B, np.int32)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs: NSETS rotating sets, each in pinned host memory and resident in HBM
    NSETS = max(2, min(int(args.lanes), 8))
    host_sets, dev_sets = [], []
    for s in range(NSETS):
        raw = synth_inputs(1000 + 17 * rank + s, B, A)
        h = {k: ([torch.from_numpy(f).pin_memory() for f in v] if isinstance(v, list) else torch.from_numpy(v).pin_memory())
             for k, v in raw.items()}
        d = {k: ([f.to(dev) for f in v] if isinstance(v, list) else v.to(dev)) for k, v in h.items()}
        host_sets.append(h)
        dev_sets.append(d)
    h2d_bytes = sum(t.numel() * 4 for k, v in host_sets[0].items() for t in (v if isinstance(v, list) else [v]))
    # one set of outputs per input set: with two lanes, two consecutive steps are in flight at the same time
    pooled7s = [torch.empty((1, B * N_ROIS, 7, 7, DEPTH), dtype=torch.float32, device=dev) for _ in range(NSETS)]
    pooled14s = [torch.empty((1, B * N_ROIS, 14, 14, DEPTH), dtype=torch.float32, device=dev) for _ in range(NSETS)]
    pooled7, pooled14 = pooled7s[0], pooled14s[0]
    roi_ev = []

    def propose(inp):
        return Proposals(conf, B, inp["probs"], inp["bbox"], anchors).get_proposals()

    # The 7x7 and the 14x14 pooling of a step walk the same proposals: their processing order (level by level, top to
    # bottom) is computed once per step - in front of the 7x7 launch - and handed to both calls (--no-shared-order: every
    # call runs its own pre-pass, as it does for any caller that passes no order).
    roi_orders = [None] * NSETS

    def roi7(inp, proposals, s_=0):
        if not args.no_shared_order:
            roi_orders[s_] = roi_processing_order(proposals, conf.IMAGE_SHAPE)
        pyramid_roi_align(inp["fmaps"], proposals, conf.IMAGE_SHAPE, [7, 7], out=pooled7s[s_], order=roi_orders[s_])

    def detect(inp, proposals):
        return DetectionLayer(conf, conf.IMAGE_SHAPE, B, window, proposals, inp["hprobs"], inp["hbbox"]).get_detections()

    # The layer classes are called unchanged inside torch.cuda.graph: per resident input set, graph A = Proposals,
    # graph B = DetectionLayer, graph C = ROIAlign 7x7. B (a chain of small latency-bound kernels on a few SMs) and C
    # (HBM-bound, all SMs) only depend on the proposals: B replays on a second, high-priority stream next to C. The
    # 14x14 ROIAlign launch - the roofline kernel - stays an eager call after C so that CUDA events bracket it inside the
    # timed region; the step joins both streams at its end.
    # LANES: consecutive steps work on different images and do not depend on each other. With two lanes, step i runs on
    # lane i % 2 (own streams, own input set, own outputs), so that the latency-bound proposal front of step i+1 (top-k,
    # NMS mask + scan: ~70 us on a few SMs) runs while the HBM-bound ROIAlign launches of step i stream. Every kernel of
    # every step still runs inside the timed region; ms_per_step is the total divided by the number of steps.
    LANES = max(1, min(args.lanes, NSETS))
    graphs_a, graphs_b, graphs_c = [None] * NSETS, [None] * NSETS, [None] * NSETS
    static_prop, static_det = [None] * NSETS, [None] * NSETS
    graph_launches = [0] * NSETS      # kernels captured per step (od_launch_count delta during the captures)
    main_stream = torch.cuda.current_stream()
    lane_main = [main_stream] + [torch.cuda.Stream() for _ in range(LANES - 1)]
    lane_det = [torch.cuda.Stream(priority=-1) for _ in range(LANES)]   # high priority: small CTAs slip in between ROIAlign CTAs
    lane_cap = [torch.cuda.Stream() for _ in range(LANES)]              # capture streams (their workspaces belong to the graphs)
    lane_roi7 = [torch.cuda.Stream() for _ in range(LANES)]             # --roi-concurrent: the 7x7 launch next to the 14x14 one
    ev_roi7 = [torch.cuda.Event() for _ in range(NSETS)]
    det_stream = lane_det[0]
    # N > 1: every all_gather of every lane goes through ONE stream, in step order - collectives of one NCCL communicator
    # must be enqueued in the same order on all ranks and must not run concurrently with each other
    gather_stream = torch.cuda.Stream(priority=-1) if world > 1 else None
    ev_prop = [torch.cuda.Event() for _ in range(NSETS)]
    ev_det = [torch.cuda.Event() for _ in range(NSETS)]
    ev_det_local = [torch.cuda.Event() for _ in range(NSETS)]

    def lane_of(s_):
        return s_ % LANES

    def capture_graphs():
        for s_ in range(NSETS):                      # eager runs on the capture streams: workspaces + constant caches exist
            l_ = lane_of(s_)
            for cap_stream in (lane_cap[l_], lane_det[l_]):
                cap_stream.wait_stream(main_stream)
                with torch.cuda.stream(cap_stream):
                    p_ = propose(dev_sets[s_])
                    roi7(dev_sets[s_], p_, s_)
                    detect(dev_sets[s_], p_)
                main_stream.wait_stream(cap_stream)
        torch.cuda.synchronize()
        for s_ in range(NSETS):
            l_ = lane_of(s_)
            n0 = L.od_launch_count()
            ga, gb, gc = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(ga, stream=lane_cap[l_]):
                static_prop[s_] = propose(dev_sets[s_])
            with torch.cuda.graph(gb, stream=lane_det[l_]):
                static_det[s_] = detect(dev_sets[s_], static_prop[s_])
            with torch.cuda.graph(gc, stream=lane_cap[l_]):
                roi7(dev_sets[s_], static_prop[s_], s_)
            graph_launches[s_] = L.od_launch_count() - n0
            graphs_a[s_], graphs_b[s_], graphs_c[s_] = ga, gb, gc

    def step(s_, time_roi=False, use_graphs=True):
        inp = dev_sets[s_]
        lm, ld = lane_main[lane_of(s_)], lane_det[lane_of(s_)]
        with torch.cuda.stream(lm):
            if use_graphs and graphs_a[s_] is not None:
                graphs_a[s_].replay()
                proposals = static_prop[s_]
                ev_prop[s_].record(lm)
                with torch.cuda.stream(ld):
                    ld.wait_event(ev_prop[s_])
                    if world > 1:      # the previous gather of this set has read static_det before it is overwritten
                        ld.wait_event(ev_det[s_])
                    graphs_b[s_].replay()
                    det = static_det[s_]
                    if world > 1:      # the path's only collective, hidden under the ROIAlign launches
                        ev_det_local[s_].record(ld)
                    else:
                        ev_det[s_].record(ld)
                if world > 1:
                    with torch.cuda.stream(gather_stream):
                        gather_stream.wait_event(ev_det_local[s_])
                        det = gather_detections(det, batch=world * B)
                        ev_det[s_].record(gather_stream)
                if args.roi_concurrent:      # both ROIAlign launches walk the same ROIs in the same order: share L2 lines
                    lr = lane_roi7[lane_of(s_)]
                    with torch.cuda.stream(lr):
                        lr.wait_event(ev_prop[s_])
                        graphs_c[s_].replay()
                        ev_roi7[s_].record(lr)
                else:
                    graphs_c[s_].replay()
            else:
                proposals = propose(inp)
                roi7(inp, proposals, s_)
                det = detect(inp, proposals)
                if world > 1:
                    ev_det_local[s_].record(lm)
                    det.record_stream(gather_stream)          # read there after this stream may have moved on
                    with torch.cuda.stream(gather_stream):
                        gather_stream.wait_event(ev_det_local[s_])
                        det = gather_detections(det, batch=world * B)
                        ev_det[s_].record(gather_stream)
            if time_roi:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(lm)
            pyramid_roi_align(inp["fmaps"], proposals, conf.IMAGE_SHAPE, [14, 14], out=pooled14s[s_], order=roi_orders[s_])
            if time_roi:
                e1.record(lm)
                roi_ev.append((e0, e1))
            # join: the lane's step ends when both branches are done. With N > 1 the lane waits for its OWN detections
            # only; the all_gather trails on the gather stream (the ranks then synchronise through a queue of collectives,
            # not once per step) and the timed region ends after the last one (join_lanes).
            if world > 1:
                lm.wait_event(ev_det_local[s_])
            elif use_graphs and graphs_a[s_] is not None:
                lm.wait_event(ev_det[s_])
            if use_graphs and graphs_a[s_] is not None and args.roi_concurrent:
                lm.wait_event(ev_roi7[s_])
        return det, proposals

    def fork_lanes():      # the lanes start after everything already queued on the main stream
        for l_ in range(1, LANES):
            lane_main[l_].wait_stream(main_stream)

    def join_lanes():      # ... and the main stream continues when every lane (and every all_gather) is done
        for l_ in range(1, LANES):
            main_stream.wait_stream(lane_main[l_])
        if gather_stream is not None:
            main_stream.wait_stream(gather_stream)

    if not args.no_graph:
        capture_graphs()
    # every lane's graphs replay at least twice before the timed region (first replays upload the graph)
    n_warm = max(args.warmup, 3, 2 * NSETS)
    for i in range(n_warm):
        step(i % NSETS)
    torch.cuda.synchronize()

    if args.kernel_times:
        kernel_times(torch, step, NSETS)

    # ---- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    # starting the clock sampler kept the host (and so the GPU) idle for 0.25 s: bring the device back to its loaded
    # state before the first timed kernel (untimed, like the warm-up steps above; a 20-step region is only ~3 ms long)
    for i in range(n_warm):
        step(i % NSETS)
    torch.cuda.synchronize()
    if world > 1:      # the host barrier releases the ranks ~0.1 ms apart; one tiny all_reduce in front of the first event
        align = torch.zeros(1, device=dev)      # lines the timed regions up on the device clock (it is not timed itself)
        dist.all_reduce(align)
    launches0 = L.od_launch_count()
    wall0 = time.time()
    ev0.record()
    fork_lanes()
    for i in range(args.steps):
        det, proposals = step(i % NSETS, time_roi=True)
    join_lanes()
    ev1.record()
    torch.cuda.synchronize(); barrier()
    wall1 = time.time()
    # read before the passes below reuse the output buffers of the input sets
    dump = None
    if args.dump_outputs and rank == 0:
        last = (args.steps - 1) % NSETS
        dump = last_step_outputs(torch, det, proposals, pooled7s[last], pooled14s[last])
    launches = L.od_launch_count() - launches0     # eager launches ...
    launches += sum(graph_launches[i % NSETS] for i in range(args.steps)) if graphs_a[0] is not None else 0   # + replayed ones
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)
    roi14_ms_lanes = float(np.mean([a.elapsed_time(b) for a, b in roi_ev]))

    # ---- one step at a time (lane i+1 waits for lane i): the step's latency, and the 14x14 ROIAlign launch timed with
    # nothing of another step running next to it - this is the duration the kernel's roofline is computed from
    roi14_ms, serial_ms = roi14_ms_lanes, ms_per_step
    if LANES > 1:
        del roi_ev[:]
        n_s = max(5, min(args.steps, 200))
        sa_, sb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        sa_.record()
        for i in range(n_s):
            fork_lanes()
            step(i % NSETS, time_roi=True)
            join_lanes()
        sb_.record()
        torch.cuda.synchronize(); barrier()
        serial_ms = max_over_ranks(sa_.elapsed_time(sb_) / n_s)
        roi14_ms = float(np.mean([a.elapsed_time(b) for a, b in roi_ev]))

    # ---- the same step launched eagerly (no CUDA graph), for the record
    eager_ms = None
    if graphs_a[0] is not None:
        for i in range(3):
            step(i % NSETS, use_graphs=False)
        n_e = max(5, min(args.steps, 50))
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ea.record()
        fork_lanes()
        for i in range(n_e):
            step(i % NSETS, use_graphs=False)
        join_lanes()
        eb.record()
        torch.cuda.synchronize()
        eager_ms = max_over_ranks(ea.elapsed_time(eb) / n_e)

    # ---- --check: the gathered detections of every shard against the CPU oracle (same seeds regenerate the inputs)
    check = None
    if args.check:
        det_all, _ = step(0)
        torch.cuda.synchronize()
        det_all = det_all.cpu().numpy()
        if rank == 0:
            import oracle
            ok, worst = True, 0
            for r in range(world):
                raw = synth_rpn_head(1000 + 17 * r + 0, B, A)
                o_, conf_, _, anc_, win_ = cpu_setup(B, with_fmaps=False)
                want = cpu_detections(o_, conf_, raw, anc_, win_)
                got = det_all[r * B:(r + 1) * B]
                same = np.array_equal(got.view(np.uint32), want.view(np.uint32))
                ok &= same
                worst = max(worst, int((got.view(np.uint32) != want.view(np.uint32)).sum()))
            check = {"headline_detections_bit_exact_vs_oracle": bool(ok), "shards": world, "mismatching_words": worst}

    # ---- roofline of the dominant kernel (14x14 ROIAlign), bytes from the ROIs the step really used
    peak, peak_src = measured_peaks()
    roof_bytes = []
    for s in range(NSETS):
        _, props = step(s)
        torch.cuda.synchronize()
        _, lv = pyramid_roi_align(dev_sets[s]["fmaps"], props, conf.IMAGE_SHAPE, [14, 14], out=pooled14, return_levels=True)
        roof_bytes.append(roialign_algorithmic_bytes(props.cpu().numpy(), lv.cpu().numpy(), 14, DEPTH))
    alg = float(np.mean([r["total"] for r in roof_bytes]))
    achieved = alg / (roi14_ms * 1e-3) / 1e9
    lib_hash = L.od_source_hash().decode()
    traffic, traffic_src = recorded_ncu_traffic(lib_hash)
    roi_kernel = "crop_bins_kernel" if os.environ.get("OD_ROI_KERNEL") == "flat" else "crop_rows_kernel"
    roofline = {"bound": "hbm", "kernel": f"{roi_kernel} (PyramidROIAlign 14x14, 2x1000 ROIs)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                "ms_per_launch": roi14_ms,
                "measured": "CUDA events around the launch, in this run, steps issued one at a time" if LANES > 1 else
                            "CUDA events around the launch inside the timed region",
                "with_steps_in_flight": {"ms_per_launch": roi14_ms_lanes, "frac": alg / (roi14_ms_lanes * 1e-3) / 1e9 / peak,
                                             "note": "the same events inside the headline timed region; the launch shares "
                                                     "HBM and SMs with the other lane's kernels"} if LANES > 1 else None}

    # ---- timed region 2: end to end, inputs in pinned HOST memory. Every step copies all of its inputs H2D (into the
    # buffers the layer classes read), runs the step and reads the detections back D2H. The copy of step i+1 runs on
    # a second stream while step i computes (two input sets = double buffer); everything is inside the timed region.
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(NSETS)]      # H2D of set s finished
    consumed = [torch.cuda.Event() for _ in range(NSETS)]   # compute on set s finished (buffers may be overwritten)
    det_host = [torch.empty((B, conf.DETECTION_POST_NMS_INSTANCES, 6), dtype=torch.float32).pin_memory() for _ in range(NSETS)]

    def h2d(s_, wait=True):
        h, d_ = host_sets[s_], dev_sets[s_]
        with torch.cuda.stream(copy_stream):
            if wait:
                copy_stream.wait_event(consumed[s_])
            for k_, v in h.items():
                if isinstance(v, list):
                    for hv, dv in zip(v, d_[k_]):
                        dv.copy_(hv, non_blocking=True)
                else:
                    d_[k_].copy_(v, non_blocking=True)
            ready[s_].record(copy_stream)

    def e2e_loop(n):
        join_lanes()
        for s_ in range(NSETS):
            consumed[s_].record(main_stream)
        h2d(0)
        out = None
        for i in range(n):
            s_ = i % NSETS
            lm = lane_main[lane_of(s_)]
            if i + 1 < n:
                h2d((i + 1) % NSETS)                 # overlaps with this step's kernels
            lm.wait_event(ready[s_])
            d, _ = step(s_)
            if world > 1:
                lm.wait_event(ev_det[s_])            # the D2H below reads the gathered detections
            with torch.cuda.stream(lm):
                det_host[s_].copy_(d[rank * B:(rank + 1) * B], non_blocking=True)   # D2H of this rank's detections
                consumed[s_].record(lm)
            lm.synchronize()                         # the caller reads the result of every step
            out = det_host[s_]
        join_lanes()
        return out

    e2e_loop(3)
    e2e_steps = max(4, min(args.steps, 40))
    barrier(); torch.cuda.synchronize()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    out = e2e_loop(e2e_steps)
    ev3.record()
    torch.cuda.synchronize(); barrier()
    e2e_ms = max_over_ranks(ev2.elapsed_time(ev3))
    d2h_bytes = out.numel() * 4
    # the bare H2D ceiling: the same pinned buffers copied by all ranks at the same time, nothing else running
    for s_ in range(NSETS):
        h2d(s_, wait=False)
    torch.cuda.synchronize(); barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_c = 6
    c0.record(copy_stream)
    for i in range(n_c):
        h2d(i % NSETS, wait=False)
    c1.record(copy_stream)
    torch.cuda.synchronize(); barrier()
    ceil_ms = max_over_ranks(c0.elapsed_time(c1)) / n_c
    ceiling_gbs = world * h2d_bytes / ceil_ms / 1e6               # aggregate over the ranks
    e2e_val = world * B * e2e_steps / (e2e_ms * 1e-3)
    e2e = {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
           "h2d_ceiling_gbs": ceiling_gbs, "h2d_ceiling_ms_per_step": ceil_ms,
           "frac_of_ceiling": ceil_ms / (e2e_ms / e2e_steps), "placement": placement,
           "note": "H2D of step i+1 overlaps the kernels of step i (2 streams); bound by the host->device copies: "
                   "h2d_ceiling_* is the same pinned buffers copied by all ranks concurrently with nothing else running"}

    # ---- BASELINE configs[4]: global batch 64 sharded 64/N per GPU (strong scaling), every N
    scaling_b64 = None
    if not args.no_extras and GLOBAL_B64 % world == 0:
        scaling_b64 = run_b64(torch, dist, world, rank, dev, conf, args, barrier, max_over_ranks)

    # ---- stand-alone ROIAlign on the SURVEY §8d ROI recipe (seed 1234), L2 flushed between launches
    standalone = {}
    if rank == 0:
        standalone = run_standalone_roialign(torch, dev, conf, dev_sets, pooled7, pooled14, det, peak, serial_ms,
                                             roofline["ms_per_launch"], world, B, NSETS)

    extra = None
    cpu_baseline = None
    if rank == 0 and world == 1:
        if not args.no_extras:
            extra = run_extras(torch, dev, conf, with_cpu=not args.no_cpu_baseline)
        if not args.no_cpu_baseline:
            cpu_baseline = run_cpu_baseline()
    if extra is None:
        extra = {}
    extra["eager_ms_per_step"] = eager_ms
    extra["ms_per_step_one_at_a_time"] = serial_ms

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(world),
            "launch": "eager, one stream" if args.no_graph else
                      "CUDA graph A (Proposals), then graph B (DetectionLayer, 2nd stream) || graph C (ROIAlign 7x7), "
                      "then eager ROIAlign 14x14" + (f"; {LANES} steps in flight (step i on lane i % {LANES}: own streams, "
                      "inputs and outputs), every kernel of every step inside the timed region" if LANES > 1 else ""),
            "lanes": LANES,
            "l2": f"{NSETS} rotating input sets; each step reads 2x89 MB of pyramid and writes 0.5 GB of pooled ROIs "
                  f"(> 126 MB L2)",
            "collective": "all_gather(detections) per step" if world > 1 else "none",
            "parallelism": f"image-sharded x{world}",
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "clocks": clocks, "scaling_b64": scaling_b64, "roialign_standalone": standalone, "extra": extra,
            "check": check, "lib_source_hash": lib_hash,
            "detections_per_image": float((det[:, :, 4] > 0).sum().item()) / det.shape[0],
        }
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def last_step_outputs(torch, det, proposals, pooled7, pooled14) -> dict:
    """Host copies of what one step hands its caller (--dump-outputs). The pooled tensors (0.5 GB at 14x14) are cut to
    DUMP_ROIS rows drawn with a fixed seed, the same rows at both pool sizes."""
    rows = np.sort(np.random.RandomState(0).choice(pooled7.shape[1], DUMP_ROIS, replace=False))
    rows = torch.from_numpy(rows).to(pooled7.device)
    return {"detections": det.cpu().numpy(), "proposals": proposals.cpu().numpy(),
            "pooled_7x7_sample": pooled7[0].index_select(0, rows).cpu().numpy(),
            "pooled_14x14_sample": pooled14[0].index_select(0, rows).cpu().numpy()}


def kernel_times(torch, step, NSETS):
    """developer aid (not a bench number): per-kernel device times of a few live steps via CUPTI, to stderr"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(4):
            step(i % NSETS)
        torch.cuda.synchronize()
    agg = {}
    evs = [ev for ev in prof.events() if ev.device_type is not None and "cuda" in str(ev.device_type).lower()]
    for ev in evs:
        a = agg.setdefault(ev.name[:70], [0, 0.0])
        a[0] += 1
        a[1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    tot = sum(v[1] for v in agg.values()) / 4
    for name, (cnt, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print(f"{us / 4:9.1f} us/step  x{cnt / 4:4.1f}  {name}", file=sys.stderr)
    print(f"{tot:9.1f} us/step  total kernel time", file=sys.stderr)
    seq = sorted(evs, key=lambda ev: ev.time_range.start)
    per_step = len(seq) // 4
    print("  -- launch order, last profiled step (start offset us, duration us) --", file=sys.stderr)
    t0 = seq[-per_step].time_range.start
    for ev in seq[-per_step:]:
        dur = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        print(f"  +{ev.time_range.start - t0:8.1f}  {dur:7.1f}  {ev.name[:60]}", file=sys.stderr)


def event_time(torch, fn, iters=10, warm=2):
    """median CUDA-event time of fn() in ms (eager calls on the current stream)"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def run_b64(torch, dist, world, rank, dev, conf, args, barrier, max_over_ranks):
    """BASELINE configs[4] / SURVEY §8e: the 1024^2 heads at GLOBAL batch 64, B_local = 64 / N images per GPU. The RPN and
    head outputs come from the same host recipe as the headline (seeded per image block, so --check can regenerate them);
    the 5.7 GB/64 images of feature pyramid are drawn on the device. One step = the headline step over B_local images,
    eager launches (at 8+ images per launch nothing is launch-bound)."""
    from objectdetection_b200 import DetectionLayer, Proposals, utils
    from objectdetection_b200.distributed import gather_detections, shard_range
    from objectdetection_b200.maskrcnn import pyramid_roi_align, roi_processing_order
    lo, hi = shard_range(GLOBAL_B64, rank, world)
    Bl = hi - lo
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = utils.gen_anchors(conf.IMAGE_SHAPE, Bl, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE, device=dev)
    A = anchors.shape[1]
    blocks = [synth_rpn_head(5000 + img // 2, 2, A) for img in range(lo, hi, 2)]       # 2 images per seed
    inp = {k: torch.from_numpy(np.concatenate([b[k] for b in blocks], 0)[:Bl]).to(dev) for k in blocks[0]}
    g = torch.Generator(device=dev)
    g.manual_seed(640 + rank)
    fmaps = [torch.rand((Bl, s, s, DEPTH), device=dev, generator=g) for s in (256, 128, 64, 32)]
    window = np.array([WINDOW_PX] * Bl, np.int32)
    p7 = torch.empty((1, Bl * N_ROIS, 7, 7, DEPTH), dtype=torch.float32, device=dev)
    p14 = torch.empty((1, Bl * N_ROIS, 14, 14, DEPTH), dtype=torch.float32, device=dev)

    # The local batch is cut into `chunks` groups of images, one stream each: every layer of the path is per image, so
    # the latency-bound proposal front / DetectionLayer of one group runs next to the HBM-bound ROIAlign launches of
    # another (the same overlap as the headline's lanes, inside one step).
    chunks = max(1, min(int(args.lanes), Bl // 2 if Bl >= 2 else 1))
    spans = [shard_range(Bl, c, chunks) for c in range(chunks)]
    cur = torch.cuda.current_stream()
    streams = [cur] + [torch.cuda.Stream() for _ in range(chunks - 1)]
    part = []
    for (c0, c1) in spans:
        n = c1 - c0
        part.append(dict(n=n, anchors=anchors[c0:c1], window=window[c0:c1],
                         inp={k: v[c0:c1] for k, v in inp.items()}, fmaps=[f[c0:c1] for f in fmaps],
                         p7=p7[0, c0 * N_ROIS:c1 * N_ROIS], p14=p14[0, c0 * N_ROIS:c1 * N_ROIS]))
    det_all_buf = torch.empty((Bl, conf.DETECTION_POST_NMS_INSTANCES, 6), dtype=torch.float32, device=dev)

    def chunk_step(q, c0, c1):
        props = Proposals(conf, q["n"], q["inp"]["probs"], q["inp"]["bbox"], q["anchors"]).get_proposals()
        order = None if args.no_shared_order else roi_processing_order(props, conf.IMAGE_SHAPE)
        pyramid_roi_align(q["fmaps"], props, conf.IMAGE_SHAPE, [7, 7], out=q["p7"], order=order)
        det = DetectionLayer(conf, conf.IMAGE_SHAPE, q["n"], q["window"], props, q["inp"]["hprobs"], q["inp"]["hbbox"]).get_detections()
        pyramid_roi_align(q["fmaps"], props, conf.IMAGE_SHAPE, [14, 14], out=q["p14"], order=order)
        det_all_buf[c0:c1].copy_(det)

    graphs = [None] * chunks

    def step64():
        for st_ in streams[1:]:
            st_.wait_stream(cur)
        for c, (q, (c0, c1), st_) in enumerate(zip(part, spans, streams)):
            with torch.cuda.stream(st_):
                if graphs[c] is not None:
                    graphs[c].replay()
                else:
                    chunk_step(q, c0, c1)
        for st_ in streams[1:]:
            cur.wait_stream(st_)
        return gather_detections(det_all_buf, batch=GLOBAL_B64) if world > 1 else det_all_buf

    # one eager pass per stream (workspaces, constant caches), then every group's chain becomes one CUDA graph: at 8-16
    # images per GPU the ~25 launches of a group are launch-bound when issued one by one from Python
    step64()
    torch.cuda.synchronize()
    if not args.no_graph:
        cap = [torch.cuda.Stream() for _ in range(chunks)]
        for c, (q, (c0, c1)) in enumerate(zip(part, spans)):
            cap[c].wait_stream(cur)
            with torch.cuda.stream(cap[c]):
                chunk_step(q, c0, c1)            # eager on the capture stream: its workspaces exist before the capture
            torch.cuda.synchronize()
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_, stream=cap[c]):
                chunk_step(q, c0, c1)
            graphs[c] = g_
        torch.cuda.synchronize()

    for _ in range(3):
        det = step64()
    steps = max(3, min(args.steps, 10))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        det = step64()
    b.record()
    torch.cuda.synchronize(); barrier()
    ms = max_over_ranks(a.elapsed_time(b)) / steps
    res = {"global_batch": GLOBAL_B64, "images_per_gpu": Bl, "scaling": "strong", "steps": steps, "warmup": 3,
           "ms_per_step": ms, "value": GLOBAL_B64 / (ms * 1e-3), "unit": "images/s",
           "launch": (f"{chunks} groups of images, one CUDA graph each, on {chunks} streams" if graphs[0] is not None else
                      f"eager, {chunks} groups of images on {chunks} streams"), "collective": "all_gather(detections) per step" if world > 1 else "none"}
    if args.check:
        det_all = det.cpu().numpy()
        if rank == 0:
            o_, conf_, _, anc_, win_ = cpu_setup(2, with_fmaps=False)
            bad = 0
            for img in range(0, GLOBAL_B64, 2):
                want = cpu_detections(o_, conf_, synth_rpn_head(5000 + img // 2, 2, A), anc_, win_)
                bad += int((det_all[img:img + 2].view(np.uint32) != want.view(np.uint32)).sum())
            res["detections_bit_exact_vs_oracle"] = bad == 0
            res["mismatching_words"] = bad
    del fmaps, p7, p14, inp
    torch.cuda.empty_cache()
    return res


def run_standalone_roialign(torch, dev, conf, dev_sets, pooled7, pooled14, det, peak, ms_per_step, roi14_ms, world, B, NSETS):
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    standalone = {}
    rois_np = rois_log_uniform(1234, B, N_ROIS)
    rois = torch.from_numpy(rois_np).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def timed(fmaps_of, rois_, P, outbuf):
        ts = []
        for it in range(12):
            flush.fill_(float(it))
            flush.sum()      # read pass: leaves CLEAN lines in L2 (no write-back charged to the launch)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            pyramid_roi_align(fmaps_of(it), rois_, conf.IMAGE_SHAPE, [P, P], out=outbuf)
            b.record()
            torch.cuda.synchronize()
            if it >= 2:
                ts.append(a.elapsed_time(b))
        return float(np.mean(ts))

    for P, outbuf in ((7, pooled7), (14, pooled14)):
        _, lv = pyramid_roi_align(dev_sets[0]["fmaps"], rois, conf.IMAGE_SHAPE, [P, P], out=outbuf, return_levels=True)
        ab = roialign_algorithmic_bytes(rois_np, lv.cpu().numpy(), P, DEPTH)
        ms = timed(lambda it: dev_sets[it % NSETS]["fmaps"], rois, P, outbuf)
        standalone[f"p{P}"] = {"ms": ms, "algorithmic_bytes": ab["total"], "GBps": ab["total"] / ms / 1e6,
                               "frac": ab["total"] / ms / 1e6 / peak, "images_per_s": B / (ms * 1e-3)}
    # SURVEY §8d also asks for matterport's mask-branch shape: 14x14 pooled over the <= 100 detections of an image
    # instead of all 1000 ROIs (reported next to the headline, which keeps the BASELINE-config 1000-ROI variant)
    det_rois = det[:B, :, :4].contiguous()
    out_det = torch.empty((1, B * det_rois.shape[1], 14, 14, DEPTH), dtype=torch.float32, device=dev)
    ms_det = timed(lambda it: dev_sets[it % NSETS]["fmaps"], det_rois, 14, out_det)
    step_det = ms_per_step - roi14_ms + ms_det
    standalone["p14_on_detections"] = {"ms": ms_det, "rois_per_image": int(det_rois.shape[1]),
                                       "step_ms_with_it": step_det, "images_per_s_with_it": world * B / (step_det * 1e-3)}
    return standalone


def run_extras(torch, dev, conf, with_cpu=True):
    """BASELINE configs[2], [3] and the 100k-box stress case of [4] through the layer classes (eager calls, CUDA events,
    median of 10), each with the CPU oracle timed beside it on a bounded sample (rank 0, N=1 only)."""
    import oracle
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _synth
    from objectdetection_b200 import BuildDetectionTargets, Proposals, fasterrcnn, utils
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    from objectdetection_b200.proposals import non_max_suppression
    cu = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    rs = np.random.RandomState(77)
    extra = {}
    omp_set_threads(cpu_threads())
    cores = cpu_threads()

    # ---- configs[2]: training chain, batch 8: Proposals(training: 6000 -> 2000) -> DetectionTargetLayer (100 GT, 200 ROIs,
    # 33 % positive) -> PyramidROIAlign 7x7 on the sampled ROIs (training.py:168-192)
    B, G = 8, 100
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = utils.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE, device=dev)
    A = anchors.shape[1]
    probs, bbox = _synth.rpn_outputs(rs, B, A)
    p_d, b_d = cu(probs), cu(bbox)
    props0 = Proposals(conf, B, p_d, b_d, anchors, training=True).get_proposals()
    props_np = props0.cpu().numpy()
    gt = np.zeros((B, G, 4), np.float32)
    gcls = np.zeros((B, G), np.int32)
    for b in range(B):
        nv = int(rs.randint(1, G + 1))
        src = rs.choice(1500, nv, replace=False)
        gt[b, :nv] = props_np[b, src] + rs.normal(0, 0.01, size=(nv, 4)).astype(np.float32)
        gcls[b, :nv] = rs.randint(1, 81, nv)
    pp = np.stack([rs.permutation(2000) for _ in range(B)]).astype(np.int32)
    pn = np.stack([rs.permutation(2000) for _ in range(B)]).astype(np.int32)
    g_d, c_d, pp_d, pn_d = cu(gt), cu(gcls), cu(pp), cu(pn)
    g8 = torch.Generator(device=dev)
    g8.manual_seed(3)
    fm8 = [torch.rand((B, s, s, DEPTH), device=dev, generator=g8) for s in (256, 128, 64, 32)]
    pooled = torch.empty((1, B * 200, 7, 7, DEPTH), dtype=torch.float32, device=dev)

    def chain():
        pr = Proposals(conf, B, p_d, b_d, anchors, training=True).get_proposals()
        t = BuildDetectionTargets(conf, pr, c_d, g_d, perm_pos=pp_d, perm_neg=pn_d)
        rois = t.get_target_rois()[0]
        pyramid_roi_align(fm8, rois, conf.IMAGE_SHAPE, [7, 7], out=pooled)
    ms_chain = event_time(torch, chain)
    ms_tgt = event_time(torch, lambda: BuildDetectionTargets(conf, props0, c_d, g_d, perm_pos=pp_d, perm_neg=pn_d))
    cfg3 = {"what": "Proposals(training, 6000->2000) -> DetectionTargetLayer (100 GT, 200 ROIs) -> ROIAlign 7x7 on the "
                    "sampled ROIs, batch 8", "ms_per_step": ms_chain, "images_per_s": B / (ms_chain * 1e-3),
            "detection_target_layer_ms": ms_tgt}
    if with_cpu:
        anc_np = anchors.cpu().numpy()
        fm_np = [f[:2].cpu().numpy() for f in fm8]

        def cpu_chain(nimg=2):
            pr = oracle.proposal_forward(probs[:nimg], bbox[:nimg], anc_np[:nimg], conf.RPN_BBOX_STDDEV,
                                         conf.PRE_NMS_ROIS_COUNT, conf.POST_NMS_ROIS_TRAINING, conf.RPN_NMS_THRESHOLD)
            rois = np.stack([oracle.detection_targets(pr[b], gcls[b], gt[b], pp[b], pn[b], conf.MRCNN_TRAIN_ROIS_PER_IMAGE,
                                                      conf.BBOX_STD_DEV)[0] for b in range(nimg)])
            oracle.pyramid_roi_align(fm_np, rois, IMAGE, IMAGE, 7, 7)
        reps, dt = timed_reps(cpu_chain, 3.0)
        cfg3["cpu_baseline"] = {"value": reps * 2 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                                "sample": f"{reps} x 2 images of the same chain in {dt:.1f} s"}
    extra["cfg3_training_chain_b8"] = cfg3
    del fm8, pooled

    # ---- configs[3]: Faster R-CNN single-level heads, 600x1000, 21,546 anchors, 12000 -> 2000, thr 0.7; roi_pool 7x7 D=512
    h, w, na = 38, 63, 9
    fp = rs.random_sample((1, h, w, 2 * na)).astype(np.float32)
    fb = rs.normal(0, 0.5, size=(1, h, w, 4 * na)).astype(np.float32)
    fp_d, fb_d = cu(fp), cu(fb)
    fmap = torch.rand((1, h, w, 512), device=dev)

    def frcnn():
        P = fasterrcnn.Proposals('train', fp_d, fb_d, image_shape=(600, 1000, 3), nms_threshold=0.7)
        fasterrcnn.roi_pool(fmap, P.proposals_padded, (600, 1000, 3))
    ms_fr = event_time(torch, frcnn)
    cfg4 = {"what": "FasterRCNN Proposals 600x1000 (21546 anchors, 12000->2000, thr 0.7) -> roi_pool 7x7 over the 2000 "
                    "padded rows (D=512), 1 image", "ms_per_step": ms_fr, "images_per_s": 1 / (ms_fr * 1e-3)}
    if with_cpu:
        fmap_np = fmap.cpu().numpy()

        def cpu_fr():
            pr = oracle.frcnn_proposals(fp, fb, 600, 1000, 12000, 2000, 0.7)
            oracle.roi_pool(fmap_np, pr, 600.0, 1000.0)
        try:
            reps, dt = timed_reps(cpu_fr, 3.0)
            cfg4["cpu_baseline"] = {"value": reps / dt, "unit": "images/s", "cores": cores, "kind": "port",
                                    "sample": f"{reps} images in {dt:.1f} s"}
        except Exception as e:      # the extras never take the bench line down
            cfg4["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    extra["cfg4_faster_rcnn"] = cfg4

    # ---- configs[4] stress: NMS over 100,000 boxes of one image (thr 0.5, max_out 100,000; replicas only, does not shard)
    n = 100000
    s = np.exp(rs.uniform(np.log(8), np.log(256), n))
    cy, cx = rs.uniform(0, 4096, n), rs.uniform(0, 4096, n)
    bx = (np.stack([cy - s / 2, cx - s / 2, cy + s / 2, cx + s / 2], 1) / 4096).astype(np.float32)
    sc = rs.random_sample(n).astype(np.float32)
    bx_d, sc_d = cu(bx)[None], cu(sc)[None]
    ms_nms = event_time(torch, lambda: non_max_suppression(bx_d, sc_d, n, 0.5), iters=5, warm=1)
    stress = {"what": "tf.image.non_max_suppression over 100,000 boxes, thr 0.5, max_out 100,000", "ms": ms_nms,
              "boxes_per_s": n / (ms_nms * 1e-3)}
    if with_cpu:
        m = 20000
        t0 = time.perf_counter()
        keep = oracle.nms(bx[:m], sc[:m], m, 0.5)
        dt = time.perf_counter() - t0
        stress["cpu_baseline"] = {"value": m / dt, "unit": "boxes/s", "cores": 1, "kind": "port",
                                  "sample": f"the first {m} of the boxes in {dt:.2f} s ({keep.shape[0]} kept); greedy NMS "
                                            f"is O(n * kept), so the full 100k case is ~25x slower per box"}
    extra["nms_stress_100k"] = stress
    return extra


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip scaling_b64 and the configs[2]/[3]/stress extras")
    ap.add_argument("--check", action="store_true", help="compare every shard's detections with the CPU oracle")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly (no CUDA graph)")
    ap.add_argument("--no-shared-order", action="store_true", help="every ROIAlign call computes its own ROI processing order")
    ap.add_argument("--roi-concurrent", action="store_true", help="experiment: 7x7 ROIAlign on its own stream next to the 14x14 launch")
    ap.add_argument("--lanes", type=int, default=4, help="steps in flight (1: strictly one step after the other)")
    ap.add_argument("--kernel-times", action="store_true", help="print per-kernel device times (CUPTI) to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
