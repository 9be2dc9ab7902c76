"""Cost of deterministic mode (torch.use_deterministic_algorithms): training iterations and kernels with the flag off and on.

    python tools/bench_deterministic.py [--steps 30 --window 10] [--out FILE]

Iterations: config C5 (PointNet2SemSeg, 8 x 8000 points, one CUDA-graph replay per iteration: train.GraphedTrainStep) and the
graphed nets of tools/bench_train_nets.py at its shapes (train.GraphedStep).  Each workload runs both modes on the same net in
alternating windows of --window iterations (which mode goes first alternates too), timed with CUDA events from an idle
device; inputs rotate through a pool larger than the 126 MB L2.  torch.utils.deterministic.fill_uninitialized_memory is set
False for these numbers (torch's default True fills every torch.empty with NaN in deterministic mode); the C5 iteration is also
reported once with it True.

Kernels, at C5 sizes: each deterministic entry point against its atomic counterpart (the scatter-adds of the grouping and
3-NN backwards including the inverse-index build, the weight gradient per layer shape, the BatchNorm statistics), timed with
CUDA events over repeated launches on inputs that rotate past L2.  The card's name and power limit are read in the same run.
Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

POOL_BYTES = 160 << 20


def _set(det: bool):
    torch.use_deterministic_algorithms(det)


def _windows(step, n_steps, window):
    """{False: ms, True: ms} per iteration, alternating windows."""
    times = {False: [], True: []}
    order = [False, True]
    done = 0
    while done < n_steps:
        for mode in order:
            _set(mode)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(window):
                step()
            b.record()
            torch.cuda.synchronize()
            times[mode].append(a.elapsed_time(b) / window)
        order.reverse()
        done += window
    _set(False)
    return {("on" if k else "off"): float(np.median(v)) for k, v in times.items()}


def bench_c5(dev, steps, window):
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import FlatAdam, GraphedTrainStep

    base = [torch.from_numpy(syn.kitti_batch(8, 8000, config=5, first=8 * i)).to(dev) for i in range(4)]
    n_pool = max(8, POOL_BYTES // base[0].nbytes)
    pool = [base[i % 4].roll(i // 4, dims=1).contiguous() for i in range(n_pool)]
    target = torch.from_numpy(np.random.default_rng(1).integers(0, 19, (8, 8000))).to(dev)
    torch.manual_seed(3)
    net = PointNet2SemSeg(19, feature_dims=1).to(dev).train()
    opt = FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)
    runner = GraphedTrainStep(net, opt)
    it = [0]

    def step():
        runner(pool[it[0] % n_pool], target)
        it[0] += 1

    for mode in (False, True):
        _set(mode)
        for _ in range(3):
            step()
    return _windows(step, steps, window)


def bench_nets(dev, steps, window):
    import bench_train_nets as btn

    from pointnet12_b200.train import FlatAdam, GraphedStep

    out = {}
    for name in btn.NETS:
        make, _, _, loss_fn, make_pool = btn._workload(name, dev)
        torch.manual_seed(7)
        net = make().to(dev).train()
        opt = FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)
        runner = GraphedStep(net, opt, loss_fn)
        pool = make_pool()
        it = [0]

        def step():
            inputs, target = pool[it[0] % len(pool)]
            runner(inputs, target)
            it[0] += 1

        for mode in (False, True):
            _set(mode)
            for _ in range(3):
                step()
        out[name] = _windows(step, steps, window)
    return out


def _time(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / reps


def _pair(make_call, copies):
    """us per call of the atomic and the deterministic variant over `copies` rotating input sets."""
    res = {}
    for mode in (False, True):
        _set(mode)
        res["on" if mode else "off"] = _time(lambda i=0: make_call(copies[i % len(copies)]))
    _set(False)
    return res


def bench_kernels(dev):
    from pointnet12_b200 import ops

    g = torch.Generator(device=dev).manual_seed(0)
    out = {}

    def copies(make, nbytes):
        return [make() for _ in range(max(2, POOL_BYTES // max(nbytes, 1)))][:16]

    # sa1 grouping backward at C5: 8 x 2048 groups x 32 of 8000 points, 32 feature channels (+3 xyz)
    B, N, S, K, D = 8, 8000, 2048, 32, 32
    xyz = torch.rand((B, N, 3), generator=g, device=dev)
    new_xyz = xyz[:, :S].contiguous()
    idx = ops.ball_query(0.1, K, xyz, new_xyz)
    mk = lambda: torch.randn((B * S * K, 3 + D), generator=g, device=dev)          # noqa: E731
    cs = copies(mk, B * S * K * (3 + D) * 4)
    out["group_backward sa1 (incl. inverse index)"] = _pair(lambda dg: ops.group_backward(dg, 3, D, idx, N), cs)
    out["group_backward_xyz sa1 (incl. inverse index)"] = _pair(lambda dg: ops.group_backward_xyz(dg, 0, idx, N), cs)
    inv = ops.csr(idx, N)
    _set(True)
    out["csr build sa1"] = {"on": _time(lambda i=0: ops.csr(idx, N))}
    out["group_backward sa1 (pull only)"] = {"on": _time(lambda i=0: ops.group_backward(cs[i % len(cs)], 3, D, idx, N, inv=inv))}
    _set(False)
    # fp1 3-NN backward: 8 x 8000 fine points from 2048 coarse ones, 128 interpolated channels
    S2, D2 = 2048, 128
    idx3, w3 = ops.three_nn(xyz, new_xyz)
    cs3 = copies(lambda: torch.randn((B * N, D2), generator=g, device=dev), B * N * D2 * 4)
    out["three_interpolate_backward fp1 (incl. inverse index)"] = _pair(
        lambda dx: ops.three_interpolate_backward(dx, 0, D2, idx3, w3, S2), cs3)
    # weight gradients of C5's layer shapes (rows, cout, cin)
    for rows, co, ci in ((524288, 32, 35), (524288, 64, 32), (131072, 128, 131), (64000, 128, 256), (64000, 19, 128)):
        dy = copies(lambda: torch.randn((rows, co), generator=g, device=dev), rows * co * 4)
        x = torch.randn((rows, ci), generator=g, device=dev)
        dw = torch.zeros((co, ci), device=dev)
        db = torch.zeros((co,), device=dev)
        out[f"grad_weight {rows}x{co}x{ci}"] = _pair(lambda d: ops.grad_weight(d, x, dw, db), dy)
    # BatchNorm statistics and their backward reductions
    bn = torch.nn.BatchNorm1d(64).to(dev).train()
    ys = copies(lambda: torch.randn((524288, 64), generator=g, device=dev), 524288 * 64 * 4)
    out["bn_batch_stats 524288x64"] = _pair(lambda y: ops.bn_batch_stats(y, bn, momentum_update=False), ys)
    st = ops.bn_batch_stats(ys[0], bn, momentum_update=False)
    dz = torch.randn((524288, 64), generator=g, device=dev)
    out["bn_act_backward 524288x64"] = _pair(lambda y: ops.bn_act_backward(y, st, dz), ys)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--window", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_deterministic.py needs a CUDA device")
    import torch.utils.deterministic as tud

    import bench_train_nets as btn

    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    dev = torch.device("cuda", 0)
    name, power = btn._card()
    tud.fill_uninitialized_memory = False
    res = {"card": name, "power_limit": power, "fill_uninitialized_memory": False,
           "c5_graphed_train_step_ms": bench_c5(dev, args.steps, args.window),
           "graphed_nets_ms": bench_nets(dev, args.steps, args.window),
           "kernels_us": bench_kernels(dev)}
    tud.fill_uninitialized_memory = True
    res["c5_graphed_train_step_ms_fill_uninitialized_memory_true"] = bench_c5(dev, args.steps, args.window)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
