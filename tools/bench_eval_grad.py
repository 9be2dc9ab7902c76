"""Cost of gradients in eval() mode at the C2 shape (PointNet2SemSeg(19, 1), shipped checkpoint, 8 x 24000 points).

    python tools/bench_eval_grad.py [--steps 20 --warmup 5 --batches 48] [--out FILE]

Prints one JSON line (and writes it to --out) with the card's name and power limit and, per step (CUDA events around
each step, median over --steps after --warmup, the three arms alternated twice):
  - attack: eval() net, points.requires_grad_(), forward, NLL of the net's own arg-max labels, backward to points.grad;
  - eval_forward: the fast eval forward alone (no gradient);
  - train_step: a C5-style train() forward + cross-entropy + backward at the same size (no optimizer step).
The batches rotate through --batches device batches (48 x 3.1 MB = 147 MB, more than the 126 MB of L2): eight synthetic
KITTI-shaped clouds, each batch rotated about z by its own angle.
Per layer on C2's shapes: "GEMM + (a)" -- the input-gradient GEMM (pn_train_gemm_bf16x3, transposed weight) followed by the
one-pass eval-mode BatchNorm backward of the layer below (pn_bn_eval_bwd_f32) -- against "(b)", the same in the GEMM's
epilogue (pn_train_gemm_bneval_bf16x3); each timed over --reps launches on rotating buffers (> 150 MB), alternating.
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
CKPT = os.path.join(ROOT, "tests", "golden", "pointnet2-inview-0.55884-0001.pth")


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
    ap.add_argument("--points", type=int, default=24000)
    ap.add_argument("--batches", type=int, default=48)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval_grad.py needs a CUDA device")

    from pointnet12_b200 import ops, synthetic as syn
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import cross_entropy

    dev = torch.device("cuda", torch.cuda.current_device())
    sd = torch.load(CKPT, map_location="cpu")
    sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}
    net = PointNet2SemSeg(19, feature_dims=1)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    trainee = PointNet2SemSeg(19, feature_dims=1)
    trainee.load_state_dict(sd, strict=True)
    trainee = trainee.to(dev).train()
    B, N = args.batch, args.points
    base = torch.from_numpy(syn.kitti_batch(B, N, config=2)).to(dev)
    batches = []
    for i in range(args.batches):
        a = 2 * np.pi * i / args.batches
        rot = torch.tensor([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], dtype=torch.float32, device=dev)
        x = base.clone()
        x[:, :3] = torch.einsum("ij,bjn->bin", rot, base[:, :3])
        batches.append(x)
    target = torch.from_numpy(np.random.default_rng(5000).integers(0, 19, size=(B, N))).to(dev)
    turn = {"i": 0}

    def next_batch():
        turn["i"] = (turn["i"] + 1) % len(batches)
        return batches[turn["i"]]

    def attack():
        x = next_batch().detach().requires_grad_(True)
        logp = net(x)
        labels = ops.argmax_labels(logp.detach())
        torch.nn.functional.nll_loss(logp.reshape(B * N, -1), labels.reshape(-1).long()).backward()
        return x.grad

    def eval_forward():
        with torch.no_grad():
            net(next_batch())

    def train_step():
        trainee.zero_grad(set_to_none=True)
        cross_entropy(trainee(next_batch()), target).backward()

    arms = {"attack": attack, "eval_forward": eval_forward, "train_step": train_step}
    step_ms = {k: [] for k in arms}
    for _ in range(2):
        for k, fn in arms.items():
            step_ms[k].append(_median_ms(fn, args.steps, args.warmup))

    # per layer, C2's shapes: the input-gradient GEMM of a layer (weight [cout, cin]) whose input comes from an inner BatchNorm
    # with running statistics: "GEMM + (a)" (pn_train_gemm_bf16x3 on W^T, then pn_bn_eval_bwd_f32 over the layer below) against
    # "(b)" (pn_train_gemm_bneval_bf16x3: the same BatchNorm backward in the GEMM's epilogue).  Each arm rotates through buffer
    # sets of more than 150 MB in all, so its operands come from HBM, not from the 126 MB L2.
    S1, S2, S3 = net.sa1.npoint, net.sa2.npoint, net.sa3.npoint
    shapes = [("sa1.conv2", B * S1 * 32, 32, 32), ("sa1.conv3", B * S1 * 32, 32, 64),
              ("sa2.conv2", B * S2 * 32, 64, 64), ("sa2.conv3", B * S2 * 32, 64, 128),
              ("sa3.conv2", B * S3 * 32, 128, 128), ("sa3.conv3", B * S3 * 32, 128, 256),
              ("fp1.conv2", B * N, 128, 128), ("fp1.conv3", B * N, 128, 128)]
    layers = {}
    torch.manual_seed(3)
    for name, rows, cin, cout in shapes:
        bn = torch.nn.BatchNorm1d(cin).to(dev).eval()
        with torch.no_grad():
            bn.running_mean.normal_(0, 0.3)
            bn.running_var.uniform_(0.5, 2.0)
        st = ops.running_stats(bn)
        w = torch.randn((cout, cin), device=dev) * 0.1
        per_set = rows * (cout + 3 * cin) * 4
        sets = [(torch.randn((rows, cout), device=dev), torch.randn((rows, cin), device=dev))
                for _ in range(max(2, -(-150_000_000 // per_set)))]
        dg, db = torch.zeros(cin, device=dev), torch.zeros(cin, device=dev)
        acc = torch.zeros((2, cin), dtype=torch.float64, device=dev)
        k = {"i": 0}

        def pick():
            k["i"] = (k["i"] + 1) % len(sets)
            return sets[k["i"]]

        def gemm_a():
            dy, py = pick()
            dz = ops.train_gemm(dy, w, None, transposed=True)
            ops.bn_eval_backward(py, st, dz, True, dgamma=dg, dbeta=db, acc=acc)

        def fused_b():
            dy, py = pick()
            ops.train_gemm_bneval(dy, w, py, st, acc, dgamma=dg, dbeta=db)

        fns = {"gemm_plus_a": gemm_a, "fused_b": fused_b}
        us = {k2: [] for k2 in fns}
        for _ in range(3):
            for k2, fn in fns.items():
                us[k2].append(_median_ms(lambda: [fn() for _ in range(args.reps)], 5, 2) * 1000.0 / args.reps)
        layers[name] = {"rows": rows, "cin": cin, "cout": cout, "buffer_sets": len(sets),
                        **{k2 + "_us": [round(v, 2) for v in vals] for k2, vals in us.items()}}
        del sets
    name, power = _card()
    rec = {
        "card": name, "power_limit": power, "batch": B, "points": N, "device_batches": len(batches),
        "step_ms": {k: [round(v, 3) for v in vals] for k, vals in step_ms.items()},
        "attack_points_per_s": round(B * N / (min(step_ms["attack"]) / 1000.0)),
        "layers": layers,
    }
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
