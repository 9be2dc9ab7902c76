"""Training iteration of the nets that sample or drop out -- eager autograd vs one CUDA-graph replay (train.GraphedStep).

    python tools/bench_train_nets.py [--steps 60 --warmup 5 --window 10] [--nets PointNet2ClsMsg,...] [--out FILE]

An iteration is the reference drivers' loop (clf.py: ModelNet40 classification, partseg.py: ShapeNet parts) on the package's
training API: forward in train() mode (batch-statistics BatchNorm, dropout, FPS start indices drawn on the CPU generator),
the loss, backward, FlatAdam (lr 1e-3, weight decay 1e-4).  Shapes and losses:

    PointNet2ClsMsg, PointNet2ClsSsg                 32 x 1024 (synthetic.modelnet_batch)   F.nll_loss
    PointNet2PartSegSsg, PointNet2PartSegMsg_one_hot 16 x 2048                              NLL over the points
    PointNetCls(40, feature_transform=True)          32 x 1024                              NLL + 0.001 * feature_transform_reguliarzer

Eager and graphed iterations run on the same net and optimizer in the same call, in alternating windows of --window
iterations (which of the two goes first alternates too).  Each window starts from an idle device (synchronise), is timed with
CUDA events around its iterations, and reports ms per iteration; --steps iterations per mode after --warmup of each (the
graphed warm-up includes the capture).  Inputs are resident on the device: a pool of batches (rotated copies of eight
synthetic batches) larger than the 126 MB L2 that the iterations walk through, so no batch is read from L2 left by its last
use.  Entry-point calls per iteration come from _native.launch_count (a replay counts the calls it captured).  The card's name
and power limit are read in the same run (read-only nvidia-smi query).  Prints one JSON line and writes it to --out.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

POOL_BYTES = 160 << 20          # more than the B200's 126 MB L2
NETS = ["PointNet2ClsMsg", "PointNet2ClsSsg", "PointNet2PartSegSsg", "PointNet2PartSegMsg_one_hot", "PointNetCls"]


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
    except (OSError, subprocess.SubprocessError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def _rotations(n, gen, dev):
    """n random rotations about the z axis [n, 3, 3]."""
    a = torch.rand((n,), generator=gen, device=dev) * (2 * math.pi)
    c, s, z, o = torch.cos(a), torch.sin(a), torch.zeros_like(a), torch.ones_like(a)
    return torch.stack([c, -s, z, s, c, z, z, z, o], 1).view(n, 3, 3)


def _workload(name, dev):
    """(net factory, batch size, points, loss_fn(net, inputs, target), make_pool() -> [(inputs, target)])."""
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model import pointnet as pn, pointnet2 as pn2
    from pointnet12_b200.model.pointnet import feature_transform_reguliarzer

    seg = "PartSeg" in name
    B, N = (16, 2048) if seg else (32, 1024)
    classes = 50 if seg else 40
    gen = torch.Generator(device=dev).manual_seed(99)
    base = torch.from_numpy(np.stack([syn.modelnet_batch(B, N, seed=6000 + i) for i in range(8)])).to(dev)    # [8,B,3,N]
    one_hot = name == "PointNet2PartSegMsg_one_hot"

    def make_pool():
        per_batch = 4 * 3 * B * N * (2 if one_hot else 1) + 8 * B * (N if seg else 1)
        pool = []
        for i in range(-(-POOL_BYTES // per_batch)):
            rot = _rotations(B, gen, dev)
            xyz = torch.bmm(rot, base[i % 8]).contiguous()
            target = torch.randint(0, classes, (B, N) if seg else (B,), generator=gen, device=dev)
            if one_hot:
                nrm = torch.randn((B, 3, N), generator=gen, device=dev)
                nrm = nrm / nrm.norm(dim=1, keepdim=True)
                label = F.one_hot(torch.randint(0, 16, (B,), generator=gen, device=dev), 16).float()
                pool.append(((xyz, nrm, label), target))
            else:
                pool.append((xyz, target))
        return pool

    def seg_nll(logp, t):
        return F.nll_loss(logp.reshape(-1, logp.shape[-1]), t.reshape(-1))

    if name == "PointNet2ClsMsg":
        return pn2.PointNet2ClsMsg, B, N, lambda net, x, t: F.nll_loss(net(x)[0], t), make_pool
    if name == "PointNet2ClsSsg":
        return pn2.PointNet2ClsSsg, B, N, lambda net, x, t: F.nll_loss(net(x), t), make_pool
    if name == "PointNet2PartSegSsg":
        return lambda: pn2.PointNet2PartSegSsg(50), B, N, lambda net, x, t: seg_nll(net(x)[0], t), make_pool
    if name == "PointNet2PartSegMsg_one_hot":
        return lambda: pn2.PointNet2PartSegMsg_one_hot(50), B, N, lambda net, x, t: seg_nll(net(*x), t), make_pool
    if name == "PointNetCls":
        def loss(net, x, t):
            logp, tf = net(x)
            return F.nll_loss(logp, t) + feature_transform_reguliarzer(tf) * 0.001
        return lambda: pn.PointNetCls(40, feature_transform=True), B, N, loss, make_pool
    raise SystemExit(f"unknown net {name}")


def _bench_net(name, args, dev):
    from pointnet12_b200 import _native as nv
    from pointnet12_b200.train import FlatAdam, GraphedStep

    make, B, N, loss_fn, make_pool = _workload(name, dev)
    torch.manual_seed(1234)
    net = make().to(dev).train()
    opt = FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)
    pool = make_pool()
    runner = GraphedStep(net, opt, loss_fn)
    last = {}

    def eager(x, t):
        loss = loss_fn(net, x, t)
        opt.zero_grad()
        loss.backward()
        opt.step(opt.all_reduce())
        return loss.detach()          # (a kept loss would keep its autograd graph alive into the next iterations)

    modes = {"eager": eager, "graphed": runner}
    k = 0
    for mode in ("eager", "graphed"):
        for _ in range(args.warmup):
            modes[mode](*pool[k % len(pool)])
            k += 1
    torch.cuda.synchronize()
    times = {"eager": [], "graphed": []}
    launches = {"eager": [], "graphed": []}
    for w in range(args.steps // args.window):
        for mode in (("eager", "graphed") if w % 2 == 0 else ("graphed", "eager")):
            torch.cuda.synchronize()
            n0 = nv.launch_count
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.window):
                last[mode] = modes[mode](*pool[k % len(pool)])
                k += 1
            b.record()
            torch.cuda.synchronize()
            times[mode].append(a.elapsed_time(b) / args.window)
            launches[mode].append((nv.launch_count - n0) / args.window)
    pool_mb = sum(sum(t.numel() * t.element_size() for t in ((x if isinstance(x, tuple) else (x,)) + (t_,)))
                  for x, t_ in pool) / 1e6
    out = {"net": name, "clouds": B, "points": N, "pool_batches": len(pool), "pool_MB": round(pool_mb, 1)}
    for mode in ("eager", "graphed"):
        ms = np.array(times[mode])
        out[mode] = {"ms_per_iter_median": round(float(np.median(ms)), 4), "ms_per_iter_min": round(float(ms.min()), 4),
                     "ms_per_iter_max": round(float(ms.max()), 4), "entry_point_calls_per_iter": float(np.mean(launches[mode])),
                     "last_loss": float(last[mode].item())}
    out["speedup_median"] = round(out["eager"]["ms_per_iter_median"] / out["graphed"]["ms_per_iter_median"], 3)
    out["graphed_draws_per_iter"] = [e for st in runner._graphs.values() for e in st["draws"].log]
    del runner, net, opt, pool
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60, help="timed iterations per mode and net")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--window", type=int, default=10, help="iterations per timed window")
    ap.add_argument("--nets", default=",".join(NETS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_nets.py needs a CUDA device")
    if args.steps < args.window or args.window < 1:
        raise SystemExit("--steps must be at least --window (>= 1)")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = _card()
    rec = {"card": name, "power_limit": power, "steps_per_mode": args.steps // args.window * args.window, "warmup": args.warmup,
           "window": args.window, "timing": "CUDA events around windows of iterations started from an idle device, "
                                             "eager and graphed windows alternating",
           "nets": [_bench_net(n, args, dev) for n in args.nets.split(",")]}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
