"""Times BuildDetectionTargets with bool GT masks read as they are against the float32 masks callers passed before the
library took bytes (``masks.float()`` first, then the float32 call), at BASELINE config 3 (B = 8, N = 2000 proposals,
G = 100 GT boxes, R = 200 training ROIs, 28x28 mask targets). One GPU, one process:

    python tools/mask_targets_u8_bench.py [--reps 30] [--warmup 5] [--h2d-reps 10]

Two mask sizes:
  * mini masks, 56x56 (USE_MINI_MASK, the reference's setting): 2.5 MB of bool masks, 10 MB in float32;
  * full-size masks, 1024x1024 (USE_MINI_MASK = False): 839 MB of bool masks, 3.36 GB in float32.

For each, three routes of the same call on the device, alternating within every repetition after a warm-up of each:
``bool`` (the masks as they are), ``bool -> f32`` (the conversion a caller made before, inside the timed region, then
the float32 call) and ``f32`` (float32 masks that already exist: the kernel's own read of 4-byte taps). Each timing is a
pair of CUDA events around the whole call. The targets of the three routes are compared bit for bit. Then the
host-to-device copy of the same masks as host bool and host float32 arrays, from pageable memory (what
BuildDetectionTargets does with a numpy array) and from pinned memory. The mini masks fit in L2 (126 MB) and are read
from there after the first repetition; the full-size masks do not. The card name and power limit are read in the same
run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


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
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--h2d-reps", type=int, default=10)
    args = ap.parse_args()
    import torch
    import _synth
    from objectdetection_b200 import BuildDetectionTargets
    from objectdetection_b200.config import config as Conf
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip() or "nvidia-smi unavailable"
    B, N, G = 8, 2000, 100
    rs = np.random.RandomState(1234)
    props, cls, gt, pp, pn = _synth.target_inputs(rs, B, N, G)
    P, C, Gb, PP, PN = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (props, cls, gt, pp, pn))
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    res, h2d, meta = {}, {}, {}
    for label, mini, M in (("mini 56x56", True, 56), ("full 1024x1024", False, 1024)):
        class Cf(Conf):
            USE_MINI_MASK = mini
        conf = Cf()
        R = conf.MRCNN_TRAIN_ROIS_PER_IMAGE
        m8 = torch.empty((B, M, M, G), dtype=torch.bool, device=dev)
        for b in range(B):                                   # [B,Mh,Mw,G]: random 0/1 pixels, one image at a time
            m8[b] = torch.rand((M, M, G), device=dev, generator=gen) < 0.5
        m32 = m8.float()

        def call(m):
            return BuildDetectionTargets(conf, P, C, Gb, perm_pos=PP, perm_neg=PN, gt_masks=m).get_target_masks()
        outs = [call(m8), call(m8.float()), call(m32)]
        same = all(torch.equal(outs[0].view(torch.int32), o.view(torch.int32)) for o in outs[1:])
        meta[label] = {"bool_bytes": m8.numel(), "f32_bytes": 4 * m8.numel(), "R": R, "targets_equal": bool(same)}
        res[label] = _time({"bool": lambda: call(m8), "bool -> f32": lambda: call(m8.float()), "f32": lambda: call(m32)},
                           args.reps, args.warmup)
        del outs, m32
        torch.cuda.empty_cache()

        host8 = m8.cpu().numpy()
        host32 = host8.astype(np.float32)
        pin8 = torch.from_numpy(host8).pin_memory()
        pin32 = torch.from_numpy(host32).pin_memory()
        h2d[label] = _time({"pageable bool": lambda: torch.from_numpy(host8).to(dev, non_blocking=True),
                            "pageable f32": lambda: torch.from_numpy(host32).to(dev, non_blocking=True),
                            "pinned bool": lambda: pin8.to(dev, non_blocking=True),
                            "pinned f32": lambda: pin32.to(dev, non_blocking=True)}, args.h2d_reps, 2)
        for r, v in h2d[label].items():
            v["GB_per_s"] = (host8.nbytes if "bool" in r else host32.nbytes) / (v["ms_median"] * 1e6)
        del m8, host8, host32, pin8, pin32
        torch.cuda.empty_cache()

    print(f"card: {card}")
    print(f"BASELINE config 3: B = {B}, N = {N}, G = {G}, R = 200, 28x28 mask targets; {args.reps} alternating "
          f"repetitions after {args.warmup} warm-up rounds; CUDA events around each whole BuildDetectionTargets call")
    print(f"{'masks':15s} {'route':12s} {'ms median':>9s} {'ms min':>8s} {'ms max':>8s}")
    for label, routes in res.items():
        for r, v in routes.items():
            print(f"{label:15s} {r:12s} {v['ms_median']:9.4f} {v['ms_min']:8.4f} {v['ms_max']:8.4f}")
        print(f"{label:15s} {meta[label]['bool_bytes'] / 1e6:.1f} MB bool, {meta[label]['f32_bytes'] / 1e6:.1f} MB f32; "
              f"targets of the three routes equal bit for bit: {meta[label]['targets_equal']}")
    print(f"host-to-device copy of the masks, {args.h2d_reps} alternating repetitions")
    print(f"{'masks':15s} {'copy':14s} {'ms median':>9s} {'ms min':>8s} {'GB/s':>7s}")
    for label, routes in h2d.items():
        for r, v in routes.items():
            print(f"{label:15s} {r:14s} {v['ms_median']:9.3f} {v['ms_min']:8.3f} {v['GB_per_s']:7.1f}")
    print(json.dumps({"card": card, "reps": args.reps, "h2d_reps": args.h2d_reps, "results": res, "h2d": h2d,
                      "masks": meta}))


if __name__ == "__main__":
    main()
