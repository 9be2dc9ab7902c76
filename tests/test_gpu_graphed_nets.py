"""train.GraphedStep on the nets whose train-mode forward draws on the host: PointNet2ClsSsg, PointNet2ClsMsg,
PointNet2PartSegSsg, PointNet2PartSegMsg_one_hot (FPS start indices and dropout seeds), PointNetCls and PointNetDenseCls
(dropout seeds).  Each net runs as two copies with the same state and their own FlatAdam, one eagerly and one graphed, after
the same torch.manual_seed: the graph must be fed exactly the eager loop's draws, anew on every replay, and every replay must
compute what an eager iteration computes from the same state.  PointNetSeg, which draws nothing, must replay as many entry-point calls as its eager iteration makes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ITERS = 4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def rl2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


def _one_hot(B, rng, dev):
    lab = np.zeros((B, 16), np.float32)
    lab[np.arange(B), rng.integers(0, 16, B)] = 1.0
    return T(lab, dev)


def _spec(name, dev, B=None, N=None):
    """(net factory, inputs, target, loss_fn) of one net at a small shape; inputs is a tuple for the nets with several."""
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model import pointnet as pn, pointnet2 as pn2
    from pointnet12_b200.model.pointnet import feature_transform_reguliarzer as reg

    rng = np.random.default_rng(31)
    if name in ("PointNet2ClsSsg", "PointNet2ClsMsg", "PointNetCls"):
        B, N = B or 8, N or 1024
        xyz = T(syn.modelnet_batch(B, N, seed=5100), dev)
        target = T(rng.integers(0, 40, B), dev)
        if name == "PointNetCls":
            def loss(net, x, t):
                logp, tf = net(x)
                return F.nll_loss(logp, t) + reg(tf) * 0.001
            return (lambda: pn.PointNetCls(40, feature_transform=True)), xyz, target, loss
        msg = name == "PointNet2ClsMsg"
        return (getattr(pn2, name)), xyz, target, lambda net, x, t: F.nll_loss(net(x)[0] if msg else net(x), t)
    B, N = B or 4, N or 1024
    xyz = T(syn.modelnet_batch(B, N, seed=5200), dev)
    target = T(rng.integers(0, 50, (B, N)), dev)

    def seg_nll(logp, t):
        return F.nll_loss(logp.reshape(-1, logp.shape[-1]), t.reshape(-1))

    if name == "PointNet2PartSegSsg":
        return (lambda: pn2.PointNet2PartSegSsg(50)), xyz, target, lambda net, x, t: seg_nll(net(x)[0], t)
    if name == "PointNet2PartSegMsg_one_hot":
        normals = rng.normal(size=(B, 3, N)).astype(np.float32)
        normals /= np.linalg.norm(normals, axis=1, keepdims=True)
        inputs = (xyz, T(normals, dev), _one_hot(B, rng, dev))
        return (lambda: pn2.PointNet2PartSegMsg_one_hot(50)), inputs, target, lambda net, x, t: seg_nll(net(*x), t)
    assert name == "PointNetDenseCls"
    B = 8 if B is None else B                 # the STN's batch-normalised fc layers want more than a few clouds

    def dense_loss(net, x, t):                # PointNetLoss's terms; the category is the one-hot label input
        cls_logits, seg_logp, tf = net(*x)
        return seg_nll(seg_logp, t) + F.cross_entropy(cls_logits, x[1].argmax(1)) + reg(tf) * 0.001

    xyz = T(syn.modelnet_batch(B, N, seed=5300), dev)
    target = T(rng.integers(0, 50, (B, N)), dev)
    return (lambda: pn.PointNetDenseCls(16, 50)), (xyz, _one_hot(B, rng, dev)), target, dense_loss


def _twins(make, dev, seed=7):
    from pointnet12_b200.train import FlatAdam

    torch.manual_seed(seed)
    a = make().to(dev).train()
    b = make().to(dev).train()
    b.load_state_dict(a.state_dict())
    return (a, FlatAdam(a.parameters(), lr=1e-3, weight_decay=1e-4)), (b, FlatAdam(b.parameters(), lr=1e-3, weight_decay=1e-4))


def _copy_state(dst, opt_dst, src, opt_src):
    """Parameters, Adam moments and step count, and BatchNorm buffers of src -> dst (same architecture)."""
    with torch.no_grad():
        for d, s in ((opt_dst.flat, opt_src.flat), (opt_dst.exp_avg, opt_src.exp_avg),
                     (opt_dst.exp_avg_sq, opt_src.exp_avg_sq), (opt_dst.step_dev, opt_src.step_dev)):
            d.copy_(s)
        for d, s in zip(dst.buffers(), src.buffers()):
            d.copy_(s)


def _entries(log):
    """(entry, offset, length) of every logged draw in the control buffer."""
    out, o = [], 0
    for e in log:
        n = e[1] * len(e[2]) if e[0] == "fps" else 2
        out.append((e, o, n))
        o += n
    return out


NETS = ["PointNet2ClsSsg", "PointNet2ClsMsg", "PointNet2PartSegSsg", "PointNet2PartSegMsg_one_hot", "PointNetCls",
        "PointNetDenseCls"]


@pytest.mark.parametrize("name", NETS)
def test_graphed_step_draws_and_numerics_match_eager(dev, monkeypatch, name):
    from pointnet12_b200 import ops, train
    from pointnet12_b200.model import pointnet2
    from pointnet12_b200.train import FlatAdam, GraphedStep

    make, inputs, target, loss_fn = _spec(name, dev)
    (a, opt_a), (b, opt_b) = _twins(make, dev)
    call = (lambda net, x: loss_fn(net, x, target))

    # eager: the draws are recorded by wrapping the two draw functions
    drawn, per_iter = [], []
    fps, seed = pointnet2.draw_fps_starts, train.dropout_seed

    def fps_spy(B, sizes, device):
        out = fps(B, sizes, device)
        drawn.append(torch.stack(out).reshape(-1).cpu())
        return out

    def seed_spy(device):
        out = seed(device)
        drawn.append(out.cpu())
        return out

    la = []
    with monkeypatch.context() as m:
        m.setattr(pointnet2, "draw_fps_starts", fps_spy)
        m.setattr(train, "dropout_seed", seed_spy)
        train._SEED["next"] = 1000
        torch.manual_seed(11)
        for it in range(ITERS):
            drawn.clear()
            loss = call(a, inputs)
            opt_a.zero_grad()
            loss.backward()
            if it == 0:
                grad_a = opt_a.grad.clone()
            opt_a.step(opt_a.all_reduce())
            la.append(loss.item())
            per_iter.append(torch.cat(drawn))
    rng_a, seed_a = torch.get_rng_state(), train._SEED["next"]

    # graphed; beside every replay an eager iteration of a third copy from the same state (parameters, Adam moments,
    # BatchNorm buffers, generator, dropout counter): its loss and gradient must be the replay's at EVERY iteration.  (The
    # two free-running loops agree at iteration 1 only: from there the fp32 atomics of the backward, amplified by Adam and
    # by the feature transforms' BatchNorm over a few clouds, make even two eager runs of PointNetCls drift apart by several
    # per cent in loss within four iterations.)
    c = make().to(dev).train()
    opt_c = FlatAdam(c.parameters(), lr=1e-3, weight_decay=1e-4)
    train._SEED["next"] = 1000
    torch.manual_seed(11)
    runner = GraphedStep(b, opt_b, loss_fn)
    lb, ctl = [], []
    for it in range(ITERS):
        _copy_state(c, opt_c, b, opt_b)
        rng, nxt = torch.get_rng_state(), train._SEED["next"]
        loss = runner(inputs, target)
        (st,) = runner._graphs.values()
        ctl.append(st["draws"].ctl.clone())
        grad_b = opt_b.grad.clone()
        if it == 0:
            grad_b0 = grad_b
        lb.append(loss.item())
        rng_b, nxt_b = torch.get_rng_state(), train._SEED["next"]
        torch.set_rng_state(rng)
        train._SEED["next"] = nxt
        loss_c = call(c, inputs)
        opt_c.zero_grad()
        loss_c.backward()
        assert torch.equal(torch.get_rng_state(), rng_b) and train._SEED["next"] == nxt_b
        assert abs(loss_c.item() - lb[-1]) <= 1e-5 * abs(loss_c.item()), (it, loss_c.item(), lb[-1])
        assert rl2(grad_b, opt_c.grad) < 1e-4, (it, rl2(grad_b, opt_c.grad))
    assert torch.equal(torch.get_rng_state(), rng_a) and train._SEED["next"] == seed_a

    # same draws: the control buffer at every replay holds exactly what the eager iteration drew
    log = st["draws"].log
    fps_entries = [e for e in _entries(log) if e[0][0] == "fps"]
    drop_entries = [e for e in _entries(log) if e[0][0] == "dropout"]
    assert len(drop_entries) == 1 and len(fps_entries) == (1 if name.startswith("PointNet2") else 0)
    for it in range(ITERS):
        assert torch.equal(ctl[it].cpu(), per_iter[it]), (it, ctl[it].cpu(), per_iter[it])
    # not frozen: new FPS starts and a new dropout mask on every replay
    for it in range(ITERS - 1):
        for _, o, n in fps_entries:
            assert not torch.equal(ctl[it][o:o + n], ctl[it + 1][o:o + n])
        (_, o, _), = drop_entries
        ones = torch.ones((256, 128), device=dev)
        masks = [ops.dropout(ones, 0.5, seed_offset=c[o:o + 2])[1] for c in (ctl[it], ctl[it + 1])]
        assert not torch.equal(masks[0], masks[1])

    # numerics of the free-running loops: the first iteration is the same computation, and both train
    assert abs(la[0] - lb[0]) <= 1e-5 * abs(la[0]), (la, lb)
    assert rl2(grad_b0, grad_a) < 1e-4, rl2(grad_b0, grad_a)
    assert la[-1] < la[0] and lb[-1] < lb[0], (la, lb)
    for net in (a, b):
        for mod in net.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                assert int(mod.num_batches_tracked) == ITERS


def test_graphed_step_recaptures_per_mode_and_shape(dev):
    """A dropout set to .eval() after capture captures again, and that graph draws no seed; a second input shape gets its own
    graph whose FPS draws are sized to it."""
    from pointnet12_b200.train import GraphedStep

    make, inputs, target, loss_fn = _spec("PointNet2PartSegSsg", dev)
    (_, _), (b, opt_b) = _twins(make, dev)
    runner = GraphedStep(b, opt_b, loss_fn)
    runner(inputs, target)
    (first,) = runner._graphs.values()
    assert first["draws"].log == [("fps", 4, (1024, 512)), ("dropout",)]
    b.drop1.eval()
    l_eval = runner(inputs, target)
    assert len(runner._graphs) == 2
    second = [st for st in runner._graphs.values() if st is not first][0]
    assert second["draws"].log == [("fps", 4, (1024, 512))] and second["draws"].ctl.numel() == 8
    assert np.isfinite(l_eval.item())
    b.drop1.train()
    _, small, small_target, _ = _spec("PointNet2PartSegSsg", dev, B=2, N=512)
    l_small = runner(small, small_target)
    assert len(runner._graphs) == 3 and np.isfinite(l_small.item())
    third = [st for st in runner._graphs.values() if st is not first and st is not second][0]
    assert third["draws"].log == [("fps", 2, (512, 512)), ("dropout",)] and third["draws"].ctl.numel() == 6
    assert tuple(third["x"][0].shape) == (2, 3, 512)
    runner(inputs, target)                   # back to the first shape and modes: no new capture
    assert len(runner._graphs) == 3


def test_graphed_step_pointnet_seg_launches_unchanged(dev):
    """PointNetSeg draws nothing: an empty log, no staging, and a replay accounts for exactly the entry-point calls of the
    eager iteration it captured."""
    from pointnet12_b200 import _native as nv, synthetic as syn
    from pointnet12_b200.model.pointnet import PointNetSeg, feature_transform_reguliarzer
    from pointnet12_b200.train import GraphedStep, cross_entropy

    pts = T(syn.kitti_batch(4, 1024, config=7), dev)
    target = T(np.random.default_rng(2).integers(0, 19, (4, 1024)), dev)

    def loss_fn(n, x, t):
        out, tf = n(x)
        return cross_entropy(out, t) + feature_transform_reguliarzer(tf) * 0.001

    (a, opt_a), (b, opt_b) = _twins(lambda: PointNetSeg(19, 4, True), dev)
    for _ in range(2):                       # (the second eager iteration is counted)
        n0 = nv.launch_count
        loss = loss_fn(a, pts, target)
        opt_a.zero_grad()
        loss.backward()
        opt_a.step(opt_a.all_reduce())
        eager = nv.launch_count - n0
    runner = GraphedStep(b, opt_b, loss_fn)
    runner(pts, target)
    (st,) = runner._graphs.values()
    assert st["draws"].log == [] and st["ring"] is None
    n0 = nv.launch_count
    runner(pts, target)
    assert nv.launch_count - n0 == eager, (nv.launch_count - n0, eager)
