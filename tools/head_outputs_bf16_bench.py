"""Times the layers that read network-head outputs, with bfloat16 inputs read as they are against today's route for bf16
inputs (``t.float()`` of every head output, then the fp32 call), at BASELINE config 2 (B = 2, 1024x1024, 261,888
anchors, N = 1000 ROIs, C = 81). One GPU, one process:

    python tools/head_outputs_bf16_bench.py [--reps 100] [--warmup 10]

Three comparisons:
  * Proposals.run_levels (6000 -> 1000, fused anchors): bf16 logits and deltas; the upcast route; fp32 inputs holding
    the same (bf16-representable) values, so that all three rank the same scores and run the same top-k and NMS;
  * DetectionLayer: fp32 probabilities with bf16 mrcnn_bbox; the upcast route;
  * Loss.rpn_losses and Loss.mrcnn_losses (B = 2, R = 200 training ROIs) with bf16 predictions; the upcast route.

Each timing is a pair of CUDA events around the whole call, conversions included. The routes of a comparison alternate
within every repetition, after a warm-up of each. The card name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _time(routes, reps, warmup):
    import torch
    for _ in range(warmup):
        for fn in routes.values():
            fn()
    torch.cuda.synchronize()
    times = {r: [] for r in routes}
    for _ in range(reps):
        for r, fn in routes.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            times[r].append(a.elapsed_time(b))
    return {r: {"ms_median": float(np.median(t)), "ms_min": float(np.min(t)), "ms_max": float(np.max(t))}
            for r, t in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps must be at least 50")
    import torch
    import bench
    from objectdetection_b200 import DetectionLayer, Proposals, utils
    from objectdetection_b200.config import config as Conf
    from objectdetection_b200.loss_optimize import Loss
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip() or "nvidia-smi unavailable"
    f32, bf16 = torch.float32, torch.bfloat16
    conf = Conf()
    B, N, C, R = 2, 1000, 81, 200
    rs = np.random.RandomState(1234)

    def t(a, dt=f32):
        return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(dev).to(dt)

    # Proposals on the per-level RPN head outputs
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                             conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    na = len(conf.RPN_ANCHOR_RATIOS)
    lg16 = [t(rs.normal(0, 2, (B, int(h), int(w), 2 * na)), bf16) for h, w in shapes]
    bb16 = [t(rs.normal(0, 1, (B, int(h), int(w), 4 * na)), bf16) for h, w in shapes]
    lg32, bb32 = [x.float() for x in lg16], [x.float() for x in bb16]
    A = sum(x.shape[1] * x.shape[2] * na for x in lg32)
    P = Proposals(conf, B, anchor_spec=spec)
    res = {"proposals": _time({
        "bf16": lambda: P.run_levels(lg16, bb16),
        "bf16 upcast": lambda: P.run_levels([x.float() for x in lg16], [x.float() for x in bb16]),
        "f32": lambda: P.run_levels(lg32, bb32)}, args.reps, args.warmup)}

    # DetectionLayer: fp32 softmax probabilities (autocast's softmax), bf16 box head
    props = t(bench.rois_log_uniform(1234, B, N))
    e = np.exp(rs.normal(0, 3, (B, N, C)))
    probs32, bbox16 = t(e / e.sum(-1, keepdims=True)), t(rs.normal(0, 1, (B, N, C, 4)), bf16)
    win = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], "int32")
    res["detection"] = _time({
        "f32 probs + bf16 boxes": lambda: DetectionLayer(conf, [1024, 1024, 3], B, win, props, probs32, bbox16),
        "bf16 boxes upcast": lambda: DetectionLayer(conf, [1024, 1024, 3], B, win, props, probs32, bbox16.float())},
        args.reps, args.warmup)

    # head losses
    tc = torch.from_numpy(rs.choice([-1, 0, 1], size=(B, A), p=[.3, .69, .01]).astype(np.int32)).to(dev)
    tb = t(rs.normal(0, 1, (B, conf.RPN_TRAIN_ANCHORS_PER_IMAGE, 4)))
    rl16, rp16 = t(rs.normal(0, 2, (B, A, 2)), bf16), t(rs.normal(0, 1, (B, A, 4)), bf16)
    ids = torch.from_numpy(np.where(rs.random_sample((B, R)) < 0.33, rs.randint(1, C, (B, R)), 0).astype(np.int32)).to(dev)
    ml16, mp16 = t(rs.normal(0, 2, (B, R, C)), bf16), t(rs.random_sample((B, R, C, 4)), bf16)
    act, mt = t(np.ones((B, C))), t(rs.random_sample((B, R, 4)))
    res["losses"] = _time({
        "bf16": lambda: (Loss.rpn_losses(tc, rl16, tb, rp16), Loss.mrcnn_losses(ids, ml16, act, mt, mp16)),
        "bf16 upcast": lambda: (Loss.rpn_losses(tc, rl16.float(), tb, rp16.float()),
                                Loss.mrcnn_losses(ids, ml16.float(), act, mt, mp16.float()))}, args.reps, args.warmup)

    print(f"card: {card}")
    print(f"BASELINE config 2: B = {B}, A = {A}, N = {N}, C = {C}; losses R = {R}; "
          f"{args.reps} alternating repetitions after {args.warmup} warm-up rounds; CUDA events around each whole call")
    print(f"{'layer':11s} {'route':24s} {'ms median':>9s} {'ms min':>8s} {'ms max':>8s}")
    for layer, routes in res.items():
        for r, v in routes.items():
            print(f"{layer:11s} {r:24s} {v['ms_median']:9.4f} {v['ms_min']:8.4f} {v['ms_max']:8.4f}")
    print(json.dumps({"card": card, "reps": args.reps, "results": res}))


if __name__ == "__main__":
    main()
