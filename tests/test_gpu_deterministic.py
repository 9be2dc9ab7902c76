"""Deterministic mode (torch.use_deterministic_algorithms): the deterministic kernel variants against numpy's ordered
scatter-add bit for bit, run-to-run equality of every deterministic kernel and of whole training iterations (eager,
GraphedTrainStep with and without next_points, GraphedStep on every net), and the default path left unchanged with the flag off."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

STEPS = 5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture
def det(monkeypatch):
    """Deterministic mode for one test; the flag and fill_uninitialized_memory are restored afterwards.  torch.bmm of the
    feature-transform regulariser goes through cuBLAS, which torch only accepts in this mode with a fixed workspace config."""
    import torch.utils.deterministic as tud

    old, warn, fill = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
                       tud.fill_uninitialized_memory)
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(old, warn_only=warn)
    tud.fill_uninitialized_memory = fill


def _seed(seed):
    """torch.manual_seed and the dropout counter (train.dropout_seed's call count): the two host draws of an iteration."""
    from pointnet12_b200 import train

    torch.manual_seed(seed)
    train._SEED["next"] = 1000


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def bits_equal(a: torch.Tensor, b) -> bool:
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else b
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32 if a.itemsize == 4 else np.uint64),
                                                                        b.view(np.uint32 if b.itemsize == 4 else np.uint64))


def rl2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ------------------------------------------------------------------------------------------------ 1. the order is pinned
def _colliding_indices(kind, rng):
    """(idx int64 [B, S, K], N) built to collide heavily."""
    if kind == "padded":         # most balls hold one or two hits, the rest of the ball repeats the first
        B, S, K, N = 2, 512, 32, 300
        idx = rng.integers(0, N, (B, S, 1)).repeat(K, axis=2)
        idx[:, :, 1] = rng.integers(0, N, (B, S))
        return idx, N
    if kind == "every_group":    # point 0 sits in every group, the other slots are random
        B, S, K, N = 2, 1024, 16, 2000
        idx = rng.integers(0, N, (B, S, K))
        idx[:, :, rng.integers(0, K)] = 0
        return idx, N
    if kind == "repeats":        # few distinct points, repeated inside each group
        B, S, K, N = 4, 256, 32, 40
        return rng.integers(0, N, (B, S, K)), N
    assert kind == "262k"        # 262 144 rows into 8000 points of two clouds
    B, S, K, N = 2, 4096, 32, 8000
    idx = rng.integers(0, N, (B, S, K))
    idx[:, :, 16:] = idx[:, :, :1]
    return idx, N


@pytest.mark.parametrize("kind", ["padded", "every_group", "repeats", "262k"])
def test_group_backward_equals_np_add_at(dev, det, kind):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(5)
    idx, N = _colliding_indices(kind, rng)
    B, S, K = idx.shape
    D, col0, ld = (16, 3, 20) if kind == "262k" else (37, 3, 44)
    dg = rng.normal(size=(B * S * K, ld)).astype(np.float32)
    want = np.zeros((B, N, D), np.float32)
    for b in range(B):
        np.add.at(want[b], idx[b].reshape(-1), dg[b * S * K:(b + 1) * S * K, col0:col0 + D])
    got = ops.group_backward(T(dg, dev), col0, D, T(idx, dev), N)
    assert bits_equal(got, want)
    # the coordinate gradient through the same inverse index
    inv = ops.csr(T(idx, dev), N)
    dxyz, dnew = ops.group_backward_xyz(T(dg, dev), 0, T(idx, dev), N, inv=inv)
    wx = np.zeros((B, N, 3), np.float32)
    for b in range(B):
        np.add.at(wx[b], idx[b].reshape(-1), dg[b * S * K:(b + 1) * S * K, :3])
    assert bits_equal(dxyz, wx)
    assert torch.equal(dnew, ops.group_backward_xyz(T(dg, dev), 0, T(idx, dev), N)[1])


def test_index_points_backward_equals_np_add_at(dev, det):
    from pointnet12_b200.model import pointnet_util as U

    rng = np.random.default_rng(6)
    B, N, C = 2, 3000, 24
    idx = rng.integers(0, N, (B, 700, 9))
    idx[:, :, 4:] = 17
    pts = T(rng.normal(size=(B, N, C)).astype(np.float32), dev).requires_grad_()
    g = rng.normal(size=(B, 700, 9, C)).astype(np.float32)
    U.index_points(pts, T(idx, dev)).backward(T(g, dev))
    want = np.zeros((B, N, C), np.float32)
    for b in range(B):
        np.add.at(want[b], idx[b].reshape(-1), g[b].reshape(-1, C))
    assert bits_equal(pts.grad, want)


def test_three_interpolate_backward_dp2_equals_np_add_at(dev, det):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(7)
    B, N, S, D1, D2 = 2, 6000, 64, 8, 48
    idx = rng.integers(0, S, (B, N, 3))
    idx[:, ::3, 1] = idx[:, ::3, 0]
    w = rng.random((B, N, 3)).astype(np.float32)
    dx = rng.normal(size=(B * N, D1 + D2)).astype(np.float32)
    dp1, dp2 = ops.three_interpolate_backward(T(dx, dev), D1, D2, T(idx, dev), T(w, dev), S)
    want = np.zeros((B, S, D2), np.float32)
    for b in range(B):
        g = dx[b * N:(b + 1) * N, D1:]
        slots = idx[b].reshape(-1)                                     # slot order: row-major over (n, k)
        prod = (g[:, None, :] * w[b][:, :, None]).reshape(-1, D2)       # fp32 products w * g
        np.add.at(want[b], slots, prod)
    assert bits_equal(dp2, want)
    assert bits_equal(dp1, dx[:, :D1].reshape(B, N, D1))


# ------------------------------------------------------------------------------------------------ 2. run to run
def _twice(fn):
    a = fn()
    b = fn()
    return a, b


def _assert_all_equal(a, b):
    for x, y in zip(a if isinstance(a, (tuple, list)) else (a,), b if isinstance(b, (tuple, list)) else (b,)):
        if x is None:
            assert y is None
            continue
        assert bits_equal(x, y)


@pytest.mark.parametrize("rows", [65536, 262144])
def test_bn_statistics_run_to_run_and_oracle(dev, det, rows):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(8)
    C = 96
    y = (rng.normal(size=(rows, C)) * 0.5 + rng.uniform(-300, 300, C)).astype(np.float32)    # offset channels
    dz = rng.normal(size=(rows, C)).astype(np.float32)
    bn = torch.nn.BatchNorm1d(C).to(dev).train()
    yt, dzt = T(y, dev), T(dz, dev)

    def stats():
        acc = torch.zeros((2, C), dtype=torch.float64, device=dev)
        with ops._on_device(yt):
            ops._col_stats(yt, acc)
        return acc

    a, b = _twice(stats)
    _assert_all_equal(a, b)
    y64 = y.astype(np.float64)
    assert np.allclose(a.cpu().numpy(), [y64.sum(0), (y64 * y64).sum(0)], rtol=1e-12)
    st = ops.bn_batch_stats(yt, bn, momentum_update=False)
    r1, r2 = _twice(lambda: ops.bn_act_backward(yt, st, dzt, True))
    _assert_all_equal(r1, r2)
    run = ops.running_stats(torch.nn.BatchNorm1d(C).to(dev).eval())
    e1, e2 = _twice(lambda: ops.bn_eval_backward(yt, run, dzt, True))
    _assert_all_equal(e1, e2)
    g = dz * (y > 0)
    assert rl2(e1[2].cpu().numpy(), g.astype(np.float64).sum(0)) < 1e-6


@pytest.mark.parametrize("engine,cout,cin,rows", [("tc", 128, 128, 65536), ("tc", 256, 131, 262144), ("fp32", 64, 35, 65536),
                                                  ("fp32", 19, 128, 262144)])
def test_grad_weight_run_to_run_and_oracle(dev, det, engine, cout, cin, rows):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(9)
    dy = rng.normal(size=(rows, cout)).astype(np.float32)
    x = rng.normal(size=(rows, cin)).astype(np.float32)
    dyt, xt = T(dy, dev), T(x, dev)

    def run():
        dw = torch.zeros((cout, cin), dtype=torch.float32, device=dev)
        db = torch.zeros((cout,), dtype=torch.float32, device=dev)
        ops.grad_weight(dyt, xt, dw, db, engine=engine)
        return dw, db

    a, b = _twice(run)
    _assert_all_equal(a, b)
    assert rl2(a[0].cpu().numpy(), dy.astype(np.float64).T @ x) < 1e-4
    assert rl2(a[1].cpu().numpy(), dy.astype(np.float64).sum(0)) < 1e-5
    if engine == "tc":           # the variant with the previous layer's normalise + ReLU applied on load
        st = ops.bn_batch_stats(xt, torch.nn.BatchNorm1d(cin).to(dev).train(), momentum_update=False)

        def run_bn():
            dw = torch.zeros((cout, cin), dtype=torch.float32, device=dev)
            ops.grad_weight(dyt, xt, dw, None, x_stats=st)
            return dw

        _assert_all_equal(*_twice(run_bn))


def test_losses_and_function_gradients_run_to_run(dev, det):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(10)
    rows, C = 64000, 19
    x = T(rng.normal(size=(rows, C)).astype(np.float32), dev)
    t = rng.integers(0, C, rows)
    t[::7] = -100
    tt = T(t, dev)
    _assert_all_equal(*_twice(lambda: ops.cross_entropy(x, tt)))
    l64 = torch.log_softmax(x.double(), 1)
    keep = tt != -100
    assert abs(float(ops.cross_entropy(x, tt)[0]) - float(-l64[keep].gather(1, tt[keep][:, None]).mean())) < 1e-5
    # square_distance, chamfer: 8 x 8000 points
    src = T(rng.normal(size=(8, 1024, 3)).astype(np.float32), dev)
    dst = T(rng.normal(size=(8, 8000, 3)).astype(np.float32), dev)
    g = T(rng.normal(size=(8, 1024, 8000)).astype(np.float32), dev)
    _assert_all_equal(*_twice(lambda: ops.square_distance_backward(g, src, dst)))
    p1 = T(rng.normal(size=(8, 8000, 3)).astype(np.float32), dev)
    p2 = T(rng.normal(size=(8, 6000, 3)).astype(np.float32), dev)
    (tot, am), (tot2, am2) = _twice(lambda: ops.chamfer_argmin(p1, p2))
    assert bits_equal(tot, tot2) and torch.equal(am, am2)
    one = torch.ones((1,), device=dev)
    _assert_all_equal(*_twice(lambda: ops.chamfer_backward(p1, p2, am, one, 0.125)))
    # 3-NN coordinate gradient
    B, N, S, D1, D2 = 8, 8000, 512, 16, 64
    xyz1 = T(rng.normal(size=(B, N, 3)).astype(np.float32), dev)
    xyz2 = T(rng.normal(size=(B, S, 3)).astype(np.float32), dev)
    p2f = T(rng.normal(size=(B, S, D2)).astype(np.float32), dev)
    idx, w = ops.three_nn(xyz1, xyz2)
    dx = T(rng.normal(size=(B * N, D1 + D2)).astype(np.float32), dev)
    _assert_all_equal(*_twice(lambda: ops.three_interpolate_backward_xyz(dx, D1, D2, idx, w, p2f, xyz1, xyz2)))
    torch.use_deterministic_algorithms(False)
    ref = ops.three_interpolate_backward_xyz(dx, D1, D2, idx, w, p2f, xyz1, xyz2)
    torch.use_deterministic_algorithms(True)
    got = ops.three_interpolate_backward_xyz(dx, D1, D2, idx, w, p2f, xyz1, xyz2)
    for a, b in zip(got[1:], ref[1:]):
        assert rl2(a.cpu().numpy(), b.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------ 3. whole iterations
def _bn_buffers(net):
    return [b.detach().clone() for b in net.buffers()]


def _state(net, opt):
    return [opt.flat.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone()] + _bn_buffers(net)


def _assert_loops_equal(run_a, run_b):
    for (la, sa), (lb, sb) in zip(run_a, run_b):
        assert bits_equal(la, lb), (float(la), float(lb))
        for x, y in zip(sa, sb):
            assert torch.equal(x, y)


def _semseg(dev, seed=3):
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import FlatAdam

    torch.manual_seed(seed)
    net = PointNet2SemSeg(19, feature_dims=1).to(dev).train()
    return net, FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)


@pytest.mark.parametrize("mode", ["eager", "graphed", "graphed_next"])
def test_semseg_iterations_bitwise_repeatable(dev, det, mode):
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.train import GraphedTrainStep, cross_entropy

    batches = [T(syn.kitti_batch(8, 8000, config=5, first=8 * i), dev) for i in range(STEPS + 1)]
    target = T(np.random.default_rng(1).integers(0, 19, (8, 8000)), dev)

    def loop():
        net, opt = _semseg(dev)
        _seed(11)
        runner = GraphedTrainStep(net, opt) if mode != "eager" else None
        out = []
        for i in range(STEPS):
            if runner is None:
                loss = cross_entropy(net(batches[i]), target)
                opt.zero_grad()
                loss.backward()
                opt.step()
                loss = loss.detach()
            elif mode == "graphed":
                loss = runner(batches[i], target)
            else:
                loss = runner(batches[i], target, next_points=batches[i + 1])
            out.append((loss.clone(), _state(net, opt)))
        return out

    _assert_loops_equal(loop(), loop())


def _spec(name, dev):
    """(net factory, inputs, target, loss_fn): the shapes and specs of tests/test_gpu_graphed_nets.py."""
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model import pointnet as pn, pointnet2 as pn2
    from pointnet12_b200.model.pointnet import feature_transform_reguliarzer as reg
    from pointnet12_b200.train import cross_entropy

    rng = np.random.default_rng(31)

    def one_hot(B):
        lab = np.zeros((B, 16), np.float32)
        lab[np.arange(B), rng.integers(0, 16, B)] = 1.0
        return T(lab, dev)

    if name in ("PointNet2ClsSsg", "PointNet2ClsMsg", "PointNetCls"):
        B, N = 8, 1024
        xyz = T(syn.modelnet_batch(B, N, seed=5100), dev)
        target = T(rng.integers(0, 40, B), dev)
        if name == "PointNetCls":
            def loss(net, x, t):
                logp, tf = net(x)
                return F.nll_loss(logp, t) + reg(tf) * 0.001
            return (lambda: pn.PointNetCls(40, feature_transform=True)), xyz, target, loss
        msg = name == "PointNet2ClsMsg"
        return (getattr(pn2, name)), xyz, target, lambda net, x, t: F.nll_loss(net(x)[0] if msg else net(x), t)
    if name == "PointNetSeg":
        pts = T(syn.kitti_batch(4, 1024, config=7), dev)
        target = T(rng.integers(0, 19, (4, 1024)), dev)

        def seg_loss(n, x, t):
            out, tf = n(x)
            return cross_entropy(out, t) + reg(tf) * 0.001
        return (lambda: pn.PointNetSeg(19, 4, True)), pts, target, seg_loss
    B, N = 4, 1024
    xyz = T(syn.modelnet_batch(B, N, seed=5200), dev)
    target = T(rng.integers(0, 50, (B, N)), dev)

    def seg_nll(logp, t):
        return F.nll_loss(logp.reshape(-1, logp.shape[-1]), t.reshape(-1))

    if name == "PointNet2PartSegSsg":
        return (lambda: pn2.PointNet2PartSegSsg(50)), xyz, target, lambda net, x, t: seg_nll(net(x)[0], t)
    if name == "PointNet2PartSegMsg_one_hot":
        normals = rng.normal(size=(B, 3, N)).astype(np.float32)
        normals /= np.linalg.norm(normals, axis=1, keepdims=True)
        inputs = (xyz, T(normals, dev), one_hot(B))
        return (lambda: pn2.PointNet2PartSegMsg_one_hot(50)), inputs, target, lambda net, x, t: seg_nll(net(*x), t)
    assert name == "PointNetDenseCls"
    B = 8

    def dense_loss(net, x, t):
        cls_logits, seg_logp, tf = net(*x)
        return seg_nll(seg_logp, t) + F.cross_entropy(cls_logits, x[1].argmax(1)) + reg(tf) * 0.001

    xyz = T(syn.modelnet_batch(B, N, seed=5300), dev)
    target = T(rng.integers(0, 50, (B, N)), dev)
    return (lambda: pn.PointNetDenseCls(16, 50)), (xyz, one_hot(B)), target, dense_loss


NETS = ["PointNet2ClsSsg", "PointNet2ClsMsg", "PointNet2PartSegSsg", "PointNet2PartSegMsg_one_hot", "PointNetCls",
        "PointNetDenseCls", "PointNetSeg"]


@pytest.mark.parametrize("name", NETS)
def test_graphed_step_nets_bitwise_repeatable(dev, det, name):
    from pointnet12_b200.train import FlatAdam, GraphedStep

    make, inputs, target, loss_fn = _spec(name, dev)

    def loop():
        torch.manual_seed(7)
        net = make().to(dev).train()
        opt = FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)
        _seed(12)
        runner = GraphedStep(net, opt, loss_fn)
        out = []
        for _ in range(STEPS):
            loss = runner(inputs, target)
            out.append((loss.clone(), _state(net, opt)))
        return out

    _assert_loops_equal(loop(), loop())


def test_coordinate_eval_and_function_gradients_bitwise_repeatable(dev, det):
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model import pointnet_util as U
    from pointnet12_b200.model.chamfer import chamfer_batch
    from pointnet12_b200.train import cross_entropy

    pts0 = T(syn.kitti_batch(2, 4096, config=5), dev)
    target = T(np.random.default_rng(1).integers(0, 19, (2, 4096)), dev)

    def train_xyz():          # train() step with coordinate gradients
        net, opt = _semseg(dev)
        _seed(5)
        pts = pts0.clone().requires_grad_()
        loss = cross_entropy(net(pts), target)
        opt.zero_grad()
        loss.backward()
        return loss.detach(), pts.grad.clone(), opt.grad.clone()

    _assert_all_equal(*_twice(train_xyz))

    def eval_grad():          # eval() with an input that requires a gradient
        net, opt = _semseg(dev)
        net.eval()
        _seed(5)
        pts = pts0.clone().requires_grad_()
        loss = cross_entropy(net(pts), target)
        opt.zero_grad()
        loss.backward()
        return loss.detach(), pts.grad.clone(), opt.grad.clone()

    _assert_all_equal(*_twice(eval_grad))

    rng = np.random.default_rng(3)
    xyz0 = T(rng.normal(size=(4, 2048, 3)).astype(np.float32), dev)
    feat0 = T(rng.normal(size=(4, 2048, 16)).astype(np.float32), dev)
    ref = T(rng.normal(size=(4, 1500, 3)).astype(np.float32), dev)

    def functions():
        _seed(5)
        xyz, feat = xyz0.clone().requires_grad_(), feat0.clone().requires_grad_()
        d = U.square_distance(xyz, ref)
        g = U.index_points(feat, T(rng_idx, dev))
        new_xyz, new_pts = U.sample_and_group(256, 0.3, 32, xyz, feat, start_idx=torch.zeros(4, dtype=torch.long, device=dev))
        loss = d.mean() + g.square().mean() + new_pts.square().mean() + chamfer_batch(new_xyz, ref)
        loss.backward()
        return loss.detach(), xyz.grad.clone(), feat.grad.clone()

    rng_idx = rng.integers(0, 2048, (4, 3000))
    rng_idx[:, 1000:] = 3
    _assert_all_equal(*_twice(functions))


# ------------------------------------------------------------------------------------------------ 4. the flag off
def _call_log(monkeypatch):
    from pointnet12_b200 import _native as nv

    log = []
    real = nv.call

    def rec(name, *args, **kw):
        log.append(name)
        return real(name, *args, **kw)

    monkeypatch.setattr(nv, "call", rec)
    return log


def test_flag_off_keeps_default_launches_and_eval_forward_is_unchanged(dev, monkeypatch):
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.train import FlatAdam, GraphedStep

    assert not torch.are_deterministic_algorithms_enabled()
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")      # one cuBLAS workspace size for both captures
    log = _call_log(monkeypatch)
    make, inputs, target, loss_fn = _spec("PointNetSeg", dev)
    torch.manual_seed(7)
    net = make().to(dev).train()
    opt = FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4)
    loss = loss_fn(net, inputs, target)
    opt.zero_grad()
    loss.backward()
    opt.step(opt.all_reduce())
    assert log and not [n for n in log if "_det_" in n or n.startswith("pn_csr")]
    # a capture with the flag off, then the flag on: captured again, with the deterministic kernels (GraphedStep on a net
    # whose loss uses no cuBLAS call, and GraphedTrainStep)
    from pointnet12_b200.train import GraphedTrainStep

    make, inputs, target, loss_fn = _spec("PointNet2ClsSsg", dev)
    net = make().to(dev).train()
    runner = GraphedStep(net, FlatAdam(net.parameters(), lr=1e-3), loss_fn)
    runner(inputs, target)
    semseg, sopt = _semseg(dev)
    pts = T(syn.kitti_batch(2, 4096, config=5), dev)
    seg_target = T(np.random.default_rng(1).integers(0, 19, (2, 4096)), dev)
    train_runner = GraphedTrainStep(semseg, sopt)
    train_runner(pts, seg_target)
    old = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        del log[:]
        runner(inputs, target)
        assert len(runner._graphs) == 2 and any("_det_" in n for n in log)
        del log[:]
        train_runner(pts, seg_target)
        assert len(train_runner._graphs) == 2 and any("_det_" in n for n in log)
    finally:
        torch.use_deterministic_algorithms(old)
    # the eval forward of PointNet2SemSeg makes the same calls and gives the same bits with the flag on
    net2, _ = _semseg(dev)
    net2.eval()
    pts = T(syn.kitti_batch(2, 8000, config=5), dev)
    starts = [torch.zeros(2, dtype=torch.long, device=dev) for _ in range(4)]
    with torch.no_grad():
        net2(pts, fps_starts=starts)          # (the first eval forward folds and packs the weights)
        del log[:]
        off = net2(pts, fps_starts=starts)
        calls_off = list(log)
        try:
            torch.use_deterministic_algorithms(True)
            del log[:]
            on = net2(pts, fps_starts=starts)
            calls_on = list(log)
        finally:
            torch.use_deterministic_algorithms(old)
    assert calls_on == calls_off and torch.equal(on, off)
