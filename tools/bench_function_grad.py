"""Cost of the function-level gradients: the square_distance backward (pn_square_distance_bwd_f32) and chamfer forward +
backward (pn_chamfer_argmin_f32 + pn_chamfer_bwd_f32).

    python tools/bench_function_grad.py [--reps 30] [--out FILE]

Prints one JSON line (and writes it to --out) with the card's name and power limit, read in the same run, and:
  - square_distance backward (both sides) at (B, N, M) = (8, 1024, 24000) -- the reference's level-1 ball-query shape -- and
    (8, 4096, 4096): median over --reps launches, each timed with CUDA events, alternating between two upstream gradients g
    larger than the 126 MB L2 (786 MB and 537 MB each), so g comes from HBM every time.  Effective GB/s counts the
    algorithmic bytes (g read once, src / dst read, dsrc / ddst written), next to a device-to-device copy of g timed the
    same way in the same run (read + write bytes), and torch's own autograd of the reference's expression
    (-2 src dst^T + |src|^2 + |dst|^2, pointnet_util.py:19-40) on the same GPU as a reference point, and the kernel asked for
    one side only (src / dst) to show which half of it costs the time;
  - chamfer_batch forward + backward at B = 8, N = M = 8192 (D = 3): median over --reps steps.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    name = torch.cuda.get_device_name()
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def _median_us(fn, reps, warmup=3):
    """fn(i) is called with the repetition number (to rotate buffers); each call timed with its own events."""
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    times = []
    for i in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(i)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) * 1000.0)
    return float(np.median(times))


def _sqdist_case(B, N, M, reps, dev):
    from pointnet12_b200 import ops

    gen = torch.Generator(device=dev).manual_seed(B * N + M)
    src = torch.rand((B, N, 3), device=dev, generator=gen)
    dst = torch.rand((B, M, 3), device=dev, generator=gen)
    gs = [torch.randn((B, N, M), device=dev, generator=gen) for _ in range(2)]
    g_bytes = 4 * B * N * M
    algo_bytes = g_bytes + 2 * 12 * B * (N + M)        # g once; src, dst read; dsrc, ddst written
    ours = _median_us(lambda i: ops.square_distance_backward(gs[i % 2], src, dst), reps)
    # one side at a time: dsrc alone keeps its sums in registers (no barrier, no column atomics); ddst alone is the
    # shared-memory column reduction with one barrier per 128-column step and a vector red per column and CTA
    src_only = _median_us(lambda i: ops.square_distance_backward(gs[i % 2], src, dst, need_dst=False), reps)
    dst_only = _median_us(lambda i: ops.square_distance_backward(gs[i % 2], src, dst, need_src=False), reps)
    copy_dst = torch.empty_like(gs[0])
    copy = _median_us(lambda i: copy_dst.copy_(gs[i % 2]), reps)
    del copy_dst
    # torch's autograd of the reference expression: backward only, on a graph built once
    s = src.clone().requires_grad_(True)
    d = dst.clone().requires_grad_(True)
    dist = -2 * torch.matmul(s, d.permute(0, 2, 1))
    dist = dist + torch.sum(s ** 2, -1).view(B, N, 1)
    dist = dist + torch.sum(d ** 2, -1).view(B, 1, M)
    ref = _median_us(lambda i: torch.autograd.grad(dist, (s, d), gs[i % 2], retain_graph=True), reps)
    del dist
    ours_gbps = algo_bytes / ours / 1e3
    copy_gbps = 2 * g_bytes / copy / 1e3
    return {"B": B, "N": N, "M": M, "g_MB": round(g_bytes / 1e6, 1), "algorithmic_MB": round(algo_bytes / 1e6, 1),
            "ours_us": round(ours, 1), "ours_GBps": round(ours_gbps, 1),
            "ours_src_only_us": round(src_only, 1), "ours_dst_only_us": round(dst_only, 1),
            "copy_us": round(copy, 1), "copy_GBps": round(copy_gbps, 1), "ours_over_copy_rate": round(ours_gbps / copy_gbps, 3),
            "torch_autograd_us": round(ref, 1), "speedup_vs_torch_autograd": round(ref / ours, 2)}


def _chamfer_case(B, N, M, reps, dev):
    from pointnet12_b200.model.chamfer import chamfer_batch

    gen = torch.Generator(device=dev).manual_seed(7)
    p1s = [torch.rand((B, N, 3), device=dev, generator=gen).requires_grad_(True) for _ in range(2)]
    p2s = [torch.rand((B, M, 3), device=dev, generator=gen).requires_grad_(True) for _ in range(2)]

    def step(i):
        p1, p2 = p1s[i % 2], p2s[i % 2]
        p1.grad = p2.grad = None
        chamfer_batch(p1, p2).backward()

    def forward_only(i):
        with torch.no_grad():
            chamfer_batch(p1s[i % 2], p2s[i % 2])

    return {"B": B, "N": N, "M": M, "D": 3, "forward_backward_us": round(_median_us(step, reps), 1),
            "forward_only_us": round(_median_us(forward_only, reps), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_function_grad.py needs a CUDA device")
    if args.reps < 20:
        raise SystemExit("--reps must be at least 20")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = _card()
    rec = {"card": name, "power_limit": power, "reps": args.reps,
           "square_distance_backward": [_sqdist_case(8, 1024, 24000, args.reps, dev),
                                        _sqdist_case(8, 4096, 4096, args.reps, dev)],
           "chamfer": _chamfer_case(8, 8192, 8192, args.reps, dev)}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
