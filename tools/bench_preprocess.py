"""Row f-3 measurement: B raw scans (dataset wire format, resident in HBM) -> [B, 4, N] + labels.

    python tools/bench_preprocess.py [--scans 8 --raw 120000 --npoints 24000 --steps 50 --warmup 5]

Prints one JSON line: raw points/s through filter + sample (CUDA events, median of --steps, 256 MiB written between
iterations), the algorithmic HBM traffic (every raw point and label read twice -- count pass and scatter pass -- plus the
kept-index list and the outputs) against the measured copy peak, the host-to-device staging time of the raw scans, and
(when launched through `python bench.py --workload preprocess`, whose CPU leg may execute oracle/) the numpy oracle on one scan.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(argv=None, cpu_baseline=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=8)
    ap.add_argument("--raw", type=int, default=120000)
    ap.add_argument("--npoints", type=int, default=24000)
    ap.add_argument("--steps", type=int, default=50, help="timed iterations")
    ap.add_argument("--warmup", type=int, default=5, help="untimed iterations before them")
    args = ap.parse_args(argv)
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.preprocess import ScanPreprocessor

    dev = torch.device("cuda", 0)
    scans = [syn.raw_scan(args.raw, 7300 + i) for i in range(args.scans)]
    pre = ScanPreprocessor(syn.SEMANTIC_KITTI_LEARNING_MAP, "inview", dev)
    ups = []
    for _ in range(4):                                   # the first call allocates the pinned staging buffers
        t0 = time.perf_counter()
        batch = pre.upload([p for p, _ in scans], [l for _, l in scans])
        torch.cuda.synchronize()
        ups.append((time.perf_counter() - t0) * 1e3)
    upload_ms = float(np.median(ups[1:]))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    times = []
    for it in range(args.warmup + args.steps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out, lab = pre(batch, args.npoints, train=True, check_empty=False)   # (synthetic scans: never empty; no read-back per batch)
        b.record()
        torch.cuda.synchronize()
        if it >= args.warmup:
            times.append(a.elapsed_time(b))
    ms = float(np.median(times))
    raw_total = args.scans * args.raw
    kept = int(pre.filter(batch)[1].sum().item())
    algo = raw_total * 20 * 2 + kept * 4 * 2 + args.scans * args.npoints * (4 + 20 + 16 + 8)
    peak = None
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    cpu = cpu_baseline(scans[0], args.npoints, args.scans) if cpu_baseline is not None else None
    print(json.dumps({"metric": "scan_preprocess_raw_points_per_sec", "value": raw_total / (ms * 1e-3), "unit": "points/s",
                      "ms_per_batch": ms, "steps": args.steps, "warmup": args.warmup, "config": {"workload": f"{args.scans} raw scans x {args.raw} points -> [{args.scans}, 4, {args.npoints}] "
                                                     "+ labels (train: jitter on), inputs resident", "kept_points": kept},
                      "algorithmic_bytes": algo, "achieved_GBps": algo / (ms * 1e-3) / 1e9, "measured_peaks": peak,
                      "upload_ms_numpy_to_device": upload_ms, "upload_ms_first_call": ups[0],
                      "cpu_baseline": cpu}))


if __name__ == "__main__":
    main()
