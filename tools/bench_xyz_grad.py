"""Cost of the coordinate gradient at the C5 shape (PointNet2SemSeg training, 8 x 8000 points).

    python tools/bench_xyz_grad.py [--steps 20 --warmup 5 --batch 8 --points 8000]

Prints one JSON line with the card's name and power limit and:
  - step_ms: one eager train()-mode forward + backward of PointNet2SemSeg(19, 1), without and with points.requires_grad_()
    (CUDA events around each step, median over --steps after --warmup);
  - fp1_bwd_us: pn_three_interpolate_bwd_f32 against pn_three_interpolate_bwd_xyz_f32 at fp1's size (B x N fine rows,
    S = 1024 coarse points, D2 = 128 channels), each timed over --reps launches (including the zero-fill of the outputs the
    kernels accumulate into), alternating the two.
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


def _median_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--points", type=int, default=8000)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_xyz_grad.py needs a CUDA device")

    from pointnet12_b200 import ops, synthetic as syn
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import cross_entropy, semseg_forward_train

    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(1234)
    net = PointNet2SemSeg(19, feature_dims=1).to(dev).train()
    B, N = args.batch, args.points
    pts = torch.from_numpy(syn.kitti_batch(B, N, config=5)).to(dev)
    target = torch.from_numpy(np.random.default_rng(5000).integers(0, 19, size=(B, N))).to(dev)

    def step(wants_grad):
        x = pts.detach().requires_grad_(wants_grad)

        def run():
            net.zero_grad(set_to_none=True)
            cross_entropy(semseg_forward_train(net, x), target).backward()
        return run

    step_ms = {}
    for _ in range(2):                      # alternate, twice
        for wants in (False, True):
            step_ms.setdefault(wants, []).append(_median_ms(step(wants), args.steps, args.warmup))

    # the fp1 backward at its real geometry: fine level 0, coarse level 1 of this batch
    rng = np.random.default_rng(7)
    S, D2 = net.sa1.npoint, 128
    x1 = pts[:, :3, :].permute(0, 2, 1)
    with torch.no_grad():
        x2, _ = net.sa1.geometry(x1.contiguous(), torch.from_numpy(rng.integers(0, N, B)).to(dev))
        idx, w = net.fp1.geometry(x1, x2)
    p2 = torch.randn((B, S, D2), device=dev)
    dx = torch.randn((B * N, D2), device=dev)
    old = lambda: ops.three_interpolate_backward(dx, 0, D2, idx, w, S)                       # noqa: E731
    new = lambda: ops.three_interpolate_backward_xyz(dx, 0, D2, idx, w, p2, x1, x2)          # noqa: E731
    us = {"three_interpolate_bwd": [], "three_interpolate_bwd_xyz": []}
    for _ in range(3):
        for key, fn in (("three_interpolate_bwd", old), ("three_interpolate_bwd_xyz", new)):
            us[key].append(_median_ms(lambda: [fn() for _ in range(args.reps)], 5, 2) * 1000.0 / args.reps)

    name, power = _card()
    print(json.dumps({
        "card": name, "power_limit": power, "batch": B, "points": N,
        "step_ms_no_xyz_grad": [round(v, 3) for v in step_ms[False]],
        "step_ms_xyz_grad": [round(v, 3) for v in step_ms[True]],
        "fp1_bwd_us": {k: [round(v, 2) for v in vals] for k, vals in us.items()},
        "fp1_shape": {"rows": B * N, "S": S, "D2": D2},
    }))


if __name__ == "__main__":
    main()
