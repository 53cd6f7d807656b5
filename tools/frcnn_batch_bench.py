#!/usr/bin/env python
"""Times the Faster R-CNN proposal layer on a batch of B images in one call against B single-image calls on the same
inputs (developer aid; run on a GPU: python tools/frcnn_batch_bench.py [--repeats 2] [--iters 20]).

Workload: 600x1000 images (38x63 feature map, 21,546 anchors), fp32 RPN outputs drawn like bench.py's cfg4, in 'train'
(12000 -> 2000, thr 0.7) and 'test' (6000 -> 300, thr 0.7) mode, each call followed by roi_pool 7x7 on a [B,38,63,512]
map over the proposals get_proposals() returns. A call is what a user runs: fasterrcnn.Proposals (which ends in one
host read of the row count) and then roi_pool. Times are CUDA-event medians over --iters runs after a warm-up, with the
batched call and the B single calls alternating. Every batched result is checked against the single calls' rows.
Prints one JSON line per (repeat, mode, B) and a markdown table; the device name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from objectdetection_b200 import fasterrcnn  # noqa: E402

IMAGE = (600, 1000, 3)
H, W, NA, D = 38, 63, 9, 512
MODES = {"train": 2000, "test": 300}


def device_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        smi = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        smi = f"nvidia-smi unavailable: {e}"
    return {"device": name, "nvidia_smi": smi}


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,2,4,8,16,32")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is nothing to time without one")
    batches = [int(b) for b in args.batches.split(",")]
    info = device_info()
    print(json.dumps(info), flush=True)
    rs = np.random.RandomState(4)
    Bmax = max(batches)
    probs = torch.from_numpy(rs.random_sample((Bmax, H, W, 2 * NA)).astype(np.float32)).cuda()
    bbox = torch.from_numpy(rs.normal(0, 0.5, size=(Bmax, H, W, 4 * NA)).astype(np.float32)).cuda()
    fmap = torch.rand((Bmax, H, W, D), device="cuda")
    rows = []
    for rep in range(args.repeats):
        for mode in MODES:
            for B in batches:
                p, b, fm = probs[:B], bbox[:B], fmap[:B]

                def batched():
                    P = fasterrcnn.Proposals(mode, p, b, image_shape=IMAGE, nms_threshold=0.7)
                    return P, fasterrcnn.roi_pool(fm, P.get_proposals(), IMAGE)

                def single():
                    out = []
                    for i in range(B):
                        P = fasterrcnn.Proposals(mode, p[i:i + 1], b[i:i + 1], image_shape=IMAGE, nms_threshold=0.7)
                        out.append((P, fasterrcnn.roi_pool(fm[i:i + 1], P.get_proposals(), IMAGE)))
                    return out

                for _ in range(args.warmup):
                    batched()
                    single()
                Pb, pooled_b = batched()
                singles = single()
                torch.cuda.synchronize()
                got = Pb.get_proposals().cpu()
                ref = torch.cat([torch.cat([torch.full((P.get_proposals().shape[0], 1), float(i)), P.get_proposals().cpu()[:, 1:]], 1)
                                 for i, (P, _) in enumerate(singles)])
                same_rows = bool(torch.equal(got.view(torch.int32), ref.view(torch.int32)))
                same_pool = bool(torch.equal(pooled_b.view(torch.int32), torch.cat([x for _, x in singles]).view(torch.int32)))
                del Pb, pooled_b, singles
                tb, ts = [], []
                for _ in range(args.iters):
                    tb.append(event_ms(batched))
                    ts.append(event_ms(single))
                r = {"repeat": rep, "mode": mode, "post_n": MODES[mode], "B": B, "rows": int(got.shape[0]),
                     "batched_ms": float(np.median(tb)), "single_calls_ms": float(np.median(ts)),
                     "batched_ms_minmax": [float(min(tb)), float(max(tb))],
                     "single_calls_ms_minmax": [float(min(ts)), float(max(ts))],
                     "same_rows": same_rows, "same_pooled": same_pool}
                r["single_over_batched"] = r["single_calls_ms"] / r["batched_ms"]
                rows.append(r)
                print(json.dumps(r), flush=True)
    print(f"\n{info['device']} ({info['nvidia_smi']}); medians of {args.iters} CUDA-event runs, Proposals + roi_pool 7x7 "
          f"D={D}, 600x1000 fp32, thr 0.7\n")
    print("| repeat | mode | B | rows | one batched call ms | B single calls ms | single / batched | rows equal |")
    print("|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['repeat']} | {r['mode']} | {r['B']} | {r['rows']} | {r['batched_ms']:.3f} | {r['single_calls_ms']:.3f} "
              f"| {r['single_over_batched']:.2f} | {r['same_rows'] and r['same_pooled']} |")
    if not all(r["same_rows"] and r["same_pooled"] for r in rows):
        raise SystemExit("a batched result differs from the single-image calls")


if __name__ == "__main__":
    main()
