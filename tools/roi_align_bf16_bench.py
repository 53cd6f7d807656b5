"""Times PyramidROIAlign (7x7 and 14x14, bench.rois_log_uniform(1234, 2, 1000), P2..P5 of 2 images, D = 256) for the
four (maps, pooled) dtype pairs, and today's route for bf16 maps: ``[f.float() for f in maps]`` followed by fp32
pooling. One GPU, one process:

    python tools/roi_align_bf16_bench.py [--reps 20]

The pairs alternate within every repetition, each launch after the same read-pass L2 flush as
bench.run_standalone_roialign, timed with CUDA events. Algorithmic bytes are bench.roialign_algorithmic_bytes with the
4-byte element replaced by each tensor's element size; the fraction of peak is over bench.measured_peaks()."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import bench
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip() or "nvidia-smi unavailable"
    peak, peak_src = bench.measured_peaks()
    image = [1024, 1024]
    rois_np = bench.rois_log_uniform(1234, 2, 1000)
    rois = torch.from_numpy(rois_np).to(dev)
    rs = np.random.RandomState(1234 + 7919)
    maps32 = [torch.from_numpy(rs.random_sample((2, s, s, 256)).astype(np.float32)).to(dev) for s in (256, 128, 64, 32)]
    maps = {torch.float32: maps32, torch.bfloat16: [f.to(torch.bfloat16) for f in maps32]}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    f32, bf16 = torch.float32, torch.bfloat16
    routes = {"f32->f32": (f32, f32, False), "bf16->f32": (bf16, f32, False), "f32->bf16": (f32, bf16, False),
              "bf16->bf16": (bf16, bf16, False), "bf16 upcast->f32": (bf16, f32, True)}
    size = {f32: 4, bf16: 2}
    print(f"card: {card}")
    print(f"peak: {peak:.0f} GB/s, {peak_src}")
    res = {}
    for P in (7, 14):
        _, lv = pyramid_roi_align(maps32, rois, image, [P, P], return_levels=True)
        ab = bench.roialign_algorithmic_bytes(rois_np, lv.cpu().numpy(), P, 256)
        outs = {dt: torch.empty((1, 2000, P, P, 256), dtype=dt, device=dev) for dt in (f32, bf16)}

        def call(route):
            md, od, upcast = routes[route]
            m = [f.float() for f in maps[md]] if upcast else maps[md]
            pyramid_roi_align(m, rois, image, [P, P], out=outs[od])

        times = {r: [] for r in routes}
        for r in routes:                                     # warm-up of every route
            call(r)
        for it in range(args.reps):
            for r in routes:
                flush.fill_(float(it))
                flush.sum()                                  # read pass: leaves clean lines in L2
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                call(r)
                b.record()
                torch.cuda.synchronize()
                times[r].append(a.elapsed_time(b))
        print(f"\n{P}x{P} pooling, 2 x 1000 ROIs, D = 256, {args.reps} alternating repetitions")
        print(f"{'maps -> pooled':18s} {'ms median':>9s} {'ms min':>8s} {'ms max':>8s} {'alg. MB':>8s} {'GB/s':>7s} {'frac':>6s}")
        for r, (md, od, upcast) in routes.items():
            t = np.array(times[r])
            byts = ab["unique_in_bytes"] // 4 * size[f32 if upcast else md] + ab["out_bytes"] // 4 * size[od]
            ms = float(np.median(t))
            gbs = byts / ms / 1e6
            res[f"p{P}/{r}"] = {"ms_median": ms, "ms_min": float(t.min()), "ms_max": float(t.max()),
                                "algorithmic_bytes": int(byts), "GBps": gbs, "frac": gbs / peak}
            note = "  (bytes of the fp32 pooling only; the conversion is extra)" if upcast else ""
            print(f"{r:18s} {ms:9.4f} {t.min():8.4f} {t.max():8.4f} {byts / 1e6:8.1f} {gbs:7.0f} {gbs / peak:6.3f}{note}")
    print(json.dumps({"card": card, "peak_GBps": peak, "peak_source": peak_src, "results": res}))


if __name__ == "__main__":
    main()
