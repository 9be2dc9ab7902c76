"""Gradients in eval() mode and with frozen BatchNorm, against float64.

In eval() mode a module whose floating-point input requires a gradient runs on the autograd blocks of train.py with
BatchNorm normalising by its running statistics (which stay untouched) and dropout as the identity -- what the reference's
torch modules do.  In train() mode a BatchNorm set to .eval() is frozen the same way.  The yardstick is the float64
restatement of tests/test_gpu_xyz_grad.py (imported, with its ref_mlp replaced by `ref_mlp_modes`, which follows each
BatchNorm's mode) differentiated by torch autograd on the CPU, with the discrete decisions (sampling, ball query, 3-NN)
taken from our forward.

Bounds that hold: the fixed-statistics backward kernel element by element, (4 E32 + 1e-6) * scale as in
tests/test_gpu_train_edges.py.  Blocks: with the exact-fp32 engine a relative L2 error below 1e-4 (no batch coupling: an
arg-max or ReLU flip moves one entry, not a channel); with the tensor-core engine the flip-tolerant comparison of
test_gpu_xyz_grad.py for outputs and input gradients, direction and size for parameter gradients.  Whole nets: direction and size of every gradient, as _net_close, with the tighter fp32 bounds
cos > 0.9999 and size within 1 %.
"""
import numpy as np
import pytest
import torch

import test_gpu_xyz_grad as xg
from test_gpu_xyz_grad import T, _leaf, _np, close_but_for_flips, cosine, rl2, within

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture(params=["bf16x3", "fp32"])
def gemm_mode(request, dev):
    from pointnet12_b200 import ops

    old = ops.set_mlp_mode(request.param)
    yield request.param
    ops.set_mlp_mode(old)


# ------------------------------------------------------------------------------------------------ restatement
LEAVES = {}          # (id(param), dtype) -> float64 / float32 leaf of a parameter in the restatement


def _param(p, dt):
    key = (id(p), dt)
    if key not in LEAVES:
        LEAVES[key] = p.detach().cpu().to(dt).requires_grad_(True)
    return LEAVES[key]


def ref_mlp_modes(x, convs, bns, dt, taps=None):
    """ref_mlp of test_gpu_xyz_grad.py with each BatchNorm's own rule: batch statistics in training mode, its running
    statistics in eval mode; parameters are leaves (LEAVES) so that their gradients can be compared too."""
    from pointnet12_b200 import ops

    for li, (conv, bn) in enumerate(zip(convs, bns)):
        W = _param(conv.weight, dt).reshape(conv.weight.shape[0], -1)
        y = x @ W.T + _param(conv.bias, dt)
        if li == 0 and taps is not None:
            y.retain_grad()
            taps.append((y, W))
        if ops.uses_running_stats(bn):
            mu, var = bn.running_mean.detach().cpu().to(dt), bn.running_var.detach().cpu().to(dt)
        else:
            flat = y.reshape(-1, y.shape[-1])
            mu = flat.mean(0)
            var = ((flat - mu) ** 2).mean(0)
        y = (y - mu) / torch.sqrt(var + bn.eps) * _param(bn.weight, dt) + _param(bn.bias, dt)
        x = torch.relu(y)
    return x


@pytest.fixture
def restate(monkeypatch):
    """The float64 restatement of test_gpu_xyz_grad.py with ref_mlp_modes in place of its batch-statistics ref_mlp."""
    LEAVES.clear()
    monkeypatch.setattr(xg, "ref_mlp", ref_mlp_modes)
    yield
    LEAVES.clear()


def _perturbed(make, seed, dev, train=False):
    """A module with BatchNorm affine parameters and running statistics away from their defaults: means of the size of
    the pre-activations, variances 0.3 .. 3 and one channel per layer with running_var = 0 (1/sqrt(eps) = 316)."""
    torch.manual_seed(seed)
    m = make()
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.normal_(0, 0.2)
                mod.running_mean.normal_(0, 0.2)
                mod.running_var.uniform_(0.3, 3.0)
                mod.running_var[1] = 0.0
                mod.num_batches_tracked.fill_(7)
    return m.to(dev).train(train)


def _bn_state(net):
    return [t.clone() for m in net.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)
            for t in (m.running_mean, m.running_var, m.num_batches_tracked)]


def _same_state(a, b):
    return len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))


def _param_grads_close(net, dt, mode, what, strict=False):
    """Every parameter's .grad against the restatement's leaf gradient.  A parameter gradient sums its rows, so with the
    tensor-core engine the arg-max / ReLU flips of many rows reach most entries of a short vector: direction and size then."""
    strict = strict and mode == "fp32"
    n = 0
    for name, p in net.named_parameters():
        leaf = LEAVES.get((id(p), dt))
        if leaf is None or leaf.grad is None:
            continue
        assert p.grad is not None, (what, name)
        _close(f"{what} {name}.grad", p.grad, leaf.grad, mode, strict)
        n += 1
    assert n > 0


def _close(what, got, want, mode, strict=True):
    """strict (a block): fp32 -> relative L2 below 1e-4, tensor cores -> flip-tolerant.  Not strict (a net): direction and
    size (fp32: cos > 0.9999, size within 1 %; tensor cores: cos > 0.99, size within 5 %)."""
    if float(np.abs(_np(want)).max()) == 0.0:
        assert float(np.abs(_np(got)).max()) == 0.0, what
        return
    if strict:
        if mode == "fp32":
            assert rl2(got, want) < 1e-4, (what, rl2(got, want))
        else:
            close_but_for_flips(what, got, want)
        return
    cos = cosine(got, want)
    ratio = np.linalg.norm(_np(got)) / np.linalg.norm(_np(want))
    fp32 = mode == "fp32"
    assert cos > (0.9999 if fp32 else 0.99) and abs(ratio - 1) < (0.01 if fp32 else 0.05), (what, cos, ratio)


# ------------------------------------------------------------------------------------------------ 1. the kernel
@pytest.mark.parametrize("layout,relu,rows,C", [("rows", True, 1000, 64), ("rows", False, 777, 37), ("grouped", True, 96 * 32, 128),
                                                ("grouped", False, 33 * 16, 19), ("tall", True, 2 * 1000, 1024),
                                                ("tall", False, 3 * 300, 65)])
def test_bn_eval_backward_kernel(dev, layout, relu, rows, C):
    """pn_bn_eval_bwd_f32 against float64: dy = scale * g with g = dz * [y*scale+shift > 0] (pooled: routed by the arg-max
    of bn_act_max, grouped K = 32 / 16 and the tall K >= 256 layout), dgamma / dbeta ADDED to the buffers' contents; y, dz
    and dy with leading dimensions above C."""
    from pointnet12_b200 import ops

    rng = np.random.default_rng(rows + C)
    K = {"rows": 1, "grouped": 32 if C == 128 else 16, "tall": 1000 if C == 1024 else 300}[layout]
    bn = torch.nn.BatchNorm1d(C).eval()
    with torch.no_grad():
        bn.weight.uniform_(-1.5, 1.5)
        bn.bias.normal_(0, 0.3)
        bn.running_mean.copy_(torch.from_numpy(rng.normal(0, 0.5, C)))
        bn.running_var.copy_(torch.from_numpy(rng.uniform(0.1, 4.0, C)))
        bn.running_var[0] = 0.0
    bn = bn.to(dev)
    st = ops.running_stats(bn)
    ybig = torch.zeros((rows, C + 5), device=dev)
    ybig[:, :C] = T(rng.normal(0, 1.5, (rows, C)).astype(np.float32), dev)
    y = ybig[:, :C]
    am = None
    if layout == "rows":
        dzn = rng.standard_normal((rows, C)).astype(np.float32)
    else:
        _, am = ops.bn_act_max(y, st, K, relu)
        dzn = rng.standard_normal((rows // K, C)).astype(np.float32)
    dzbig = torch.zeros((dzn.shape[0], C + 3), device=dev)
    dzbig[:, :C] = T(dzn, dev)
    dg0, db0 = rng.standard_normal(C).astype(np.float32), rng.standard_normal(C).astype(np.float32)
    dgamma, dbeta = T(dg0.copy(), dev), T(db0.copy(), dev)
    dy = ops.bn_eval_backward(y, st, dzbig[:, :C], relu, argmax=am, K=K, dgamma=dgamma, dbeta=dbeta)
    # restatement
    yv = y.cpu().numpy()
    sc, sh, mu, isd = (t.cpu().numpy() for t in (st.scale, st.shift, st.mean, st.invstd))
    if am is None:
        g = dzn.astype(np.float64)
    else:
        amn = am.cpu().numpy()
        sel = (np.arange(rows) % K)[:, None] == np.repeat(amn, K, axis=0)
        g = np.where(sel, np.repeat(dzn, K, axis=0), 0.0).astype(np.float64)
    if relu:
        g = g * ((yv.astype(np.float64) * sc + sh) > 0)
    xh = (yv.astype(np.float64) - mu) * isd
    out = {}
    for dt in (torch.float64, torch.float32):
        gg, xx, s = (torch.from_numpy(a).to(dt) for a in (g, xh, sc.astype(np.float64)))
        out[dt] = (gg * s, (gg * xx).sum(0), gg.sum(0))
    within("dy", dy, out[torch.float64][0], out[torch.float32][0], np.abs(g * sc))
    gx = np.abs(g * xh)
    within("dgamma", dgamma, dg0 + _np(out[torch.float64][1]), dg0 + _np(out[torch.float32][1]), gx.sum(0) + np.abs(dg0),
           4 * rows * xg.U32 * gx.sum(0))
    within("dbeta", dbeta, db0 + _np(out[torch.float64][2]), db0 + _np(out[torch.float32][2]), np.abs(g).sum(0) + np.abs(db0))
    assert (g != 0).any() and ((g == 0).any() or (layout == "rows" and not relu))


@pytest.mark.parametrize("rows,cin,cout", [(1000, 32, 64), (4099, 64, 64), (777, 96, 128), (2048, 128, 256)])
def test_bneval_gemm_equals_gemm_plus_pass(dev, rows, cin, cout):
    """pn_train_gemm_bneval_bf16x3 (the eval-mode BatchNorm backward of the layer below in the epilogue of the input-gradient
    GEMM) against "GEMM + (a)": pn_train_gemm_bf16x3 on W^T followed by pn_bn_eval_bwd_f32.  dy is bit-identical; dgamma /
    dbeta agree to the fp64 summation order, ADDED to the buffers' contents; prev_y with a leading dimension above C."""
    from pointnet12_b200 import ops

    torch.manual_seed(rows)
    bn = torch.nn.BatchNorm1d(cin).eval()
    with torch.no_grad():
        bn.weight.uniform_(-1.5, 1.5)
        bn.bias.normal_(0, 0.3)
        bn.running_mean.normal_(0, 0.5)
        bn.running_var.uniform_(0.1, 4.0)
        bn.running_var[0] = 0.0
    st = ops.running_stats(bn.to(dev))
    dy = torch.randn((rows, cout), device=dev)
    w = torch.randn((cout, cin), device=dev) * 0.2
    pbig = torch.randn((rows, cin + 4), device=dev)
    py = pbig[:, :cin]
    g0, b0 = torch.randn(cin, device=dev), torch.randn(cin, device=dev)
    dg_a, db_a, dg_b, db_b = g0.clone(), b0.clone(), g0.clone(), b0.clone()
    dz = ops.train_gemm(dy, w, None, transposed=True)
    want = ops.bn_eval_backward(py, st, dz, True, dgamma=dg_a, dbeta=db_a)
    acc = torch.zeros((2, cin), dtype=torch.float64, device=dev)
    got = ops.train_gemm_bneval(dy, w, py, st, acc, dgamma=dg_b, dbeta=db_b)
    assert torch.equal(got, want)
    g = torch.where(py * st.scale + st.shift > 0, dz, torch.zeros_like(dz)).double()
    xh = ((py - st.mean) * st.invstd).double()
    for what, a, b, terms in (("dgamma", dg_b, dg_a, (g * xh).abs().sum(0)), ("dbeta", db_b, db_a, g.abs().sum(0))):
        assert ((a - b).double().abs() <= 2 ** -22 * (terms + (g0 if what == "dgamma" else b0).double().abs()) + 1e-30).all(), what
    assert (g == 0).any() and (g != 0).any()


# ------------------------------------------------------------------------------------------------ 2. blocks in eval()
@pytest.mark.parametrize("kind", ["ssg", "msg", "all"])
def test_sa_block_eval_grads(dev, gemm_mode, restate, kind):
    """Set abstraction in eval() with xyz and points requiring a gradient: a grad_fn, xyz.grad, points.grad and every
    parameter gradient against float64; running statistics untouched."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model import pointnet_util as pu

    rng = np.random.default_rng({"ssg": 1, "msg": 2, "all": 3}[kind])
    B, N, D = 2, 512, 16
    if kind == "ssg":
        mod = _perturbed(lambda: pu.PointNetSetAbstraction(128, 0.3, 32, D + 3, [32, 32, 64], False), 11, dev)
    elif kind == "msg":
        mod = _perturbed(lambda: pu.PointNetSetAbstractionMsg(128, [0.2, 0.3, 0.5], [16, 32, 64], D,
                                                               [[16, 16, 32], [32, 32, 64], [32, 48, 64]]), 12, dev)
    else:
        mod = _perturbed(lambda: pu.PointNetSetAbstraction(None, None, None, D + 3, [32, 64, 128], True), 13, dev)
    state = _bn_state(mod)
    xyz_np = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    pts_np = rng.standard_normal((B, N, D)).astype(np.float32)
    start = rng.integers(0, N, B)
    xyz = T(xyz_np.transpose(0, 2, 1), dev).requires_grad_(True)
    pts = T(pts_np.transpose(0, 2, 1), dev).requires_grad_(True)
    new_xyz, out = mod(xyz, pts, start_idx=T(start, dev))
    assert out.grad_fn is not None
    # the forward is the fast path's up to rounding
    with torch.no_grad():
        fx, fo = mod(xyz.detach(), pts.detach(), start_idx=T(start, dev))
    assert torch.equal(fx, new_xyz.detach()) and rl2(out, fo) < 1e-4
    G = rng.standard_normal(out.shape).astype(np.float32)
    Gn = rng.standard_normal(new_xyz.shape).astype(np.float32) if kind != "all" else None
    loss = (out * T(G, dev)).sum() + ((new_xyz * T(Gn, dev)).sum() if Gn is not None else 0)
    loss.backward()
    assert _same_state(state, _bn_state(mod))
    xpm = T(xyz_np, dev)
    fps = ops.fps(xpm, mod.npoint, T(start, dev)) if kind != "all" else None
    if kind == "ssg":
        balls = [ops.ball_query(mod.radius, mod.nsample, xpm, ops.index_points(xpm, fps))]
        blocks = [(mod.mlp_convs, mod.mlp_bns)]
    elif kind == "msg":
        balls = [ops.ball_query(r, k, xpm, ops.index_points(xpm, fps)) for r, k in zip(mod.radius_list, mod.nsample_list)]
        blocks = list(zip(mod.conv_blocks, mod.bn_blocks))
    else:
        balls, blocks = [None], [(mod.mlp_convs, mod.mlp_bns)]
    dt = torch.float64
    a, p = _leaf(xyz_np, dt), _leaf(pts_np, dt)
    outs = []
    for ball, (convs, bns) in zip(balls, blocks):
        nx, o = xg.ref_sa(a, p, torch.from_numpy(fps.cpu().numpy()) if fps is not None else None,
                          torch.from_numpy(ball.cpu().numpy()) if ball is not None else None, convs, bns, dt, msg=kind == "msg")
        outs.append(o)
    o = torch.cat(outs, -1).permute(0, 2, 1)
    ref_loss = (o * torch.from_numpy(G).to(dt)).sum()
    if Gn is not None:
        ref_loss = ref_loss + (nx.permute(0, 2, 1) * torch.from_numpy(Gn).to(dt)).sum()
    ref_loss.backward()
    _close("out", out.detach(), o.detach(), gemm_mode)
    _close("xyz.grad", xyz.grad.permute(0, 2, 1), a.grad, gemm_mode)
    _close("points.grad", pts.grad.permute(0, 2, 1), p.grad, gemm_mode)
    _param_grads_close(mod, dt, gemm_mode, kind, strict=True)


@pytest.mark.parametrize("S,skip", [(1, True), (128, True), (128, False)])
def test_fp_block_eval_grads(dev, gemm_mode, restate, S, skip):
    """Feature propagation in eval(): S = 1 (broadcast) and S > 1 (3-NN interpolation), with and without skip features."""
    rng = np.random.default_rng(S + int(skip))
    from pointnet12_b200.model import pointnet_util as pu

    B, N, D1, D2 = 2, 1024, (32 if skip else 0), 64
    mod = _perturbed(lambda: pu.PointNetFeaturePropagation(D1 + D2, [64, 64]), 21, dev)
    state = _bn_state(mod)
    x1_np, x2_np = xg._fp_clouds(B, N, S, rng) if S > 1 else (rng.uniform(-1, 1, (B, N, 3)).astype(np.float32),
                                                              np.zeros((B, 1, 3), np.float32))
    p1_np = rng.standard_normal((B, N, D1)).astype(np.float32) if skip else None
    p2_np = rng.standard_normal((B, S, D2)).astype(np.float32)
    leaves = [T(a.transpose(0, 2, 1), dev).requires_grad_(True) if a is not None else None for a in (x1_np, x2_np, p1_np, p2_np)]
    out = mod(*leaves)
    assert out.grad_fn is not None
    G = rng.standard_normal(out.shape).astype(np.float32)
    (out * T(G, dev)).sum().backward()
    assert _same_state(state, _bn_state(mod))
    idx, d32 = xg._nn_geometry(T(x1_np, dev), T(x2_np, dev))
    dt = torch.float64
    refs = [_leaf(v, dt) if v is not None else None for v in (x1_np, x2_np, p1_np, p2_np)]
    o = xg.ref_fp(refs[0], refs[1], refs[2], refs[3], torch.from_numpy(idx), d32, mod.mlp_convs, mod.mlp_bns, dt)
    (o.permute(0, 2, 1) * torch.from_numpy(G).to(dt)).sum().backward()
    _close("out", out.detach().permute(0, 2, 1), o.detach(), gemm_mode)
    if skip:
        _close("points1.grad", leaves[2].grad.permute(0, 2, 1), refs[2].grad, gemm_mode)
    _close("points2.grad", leaves[3].grad.permute(0, 2, 1), refs[3].grad, gemm_mode)
    if S > 1:
        # the interpolation weights' 1/d^2 amplifies rounding near coincident points: direction and size
        _close("xyz1.grad", leaves[0].grad.permute(0, 2, 1), refs[0].grad, gemm_mode, strict=False)
    else:
        assert torch.count_nonzero(leaves[0].grad) == 0 and torch.count_nonzero(leaves[1].grad) == 0
    _param_grads_close(mod, dt, gemm_mode, "fp", strict=True)


# ------------------------------------------------------------------------------------------------ 3. PointNet2SemSeg
def _semseg(ckpt_state, dev):
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg

    net = PointNet2SemSeg(19, 1)
    net.load_state_dict({k: torch.as_tensor(v) for k, v in ckpt_state.items()}, strict=True)
    return net.to(dev).eval()


def _semseg_restated(net, pts_np, starts, keep, dev, dt=torch.float64):
    """PointNet2SemSeg in float64 with our forward's decisions -> (points leaf, log-probabilities [B,N,19])."""
    pl = _leaf(pts_np, dt)
    pm = pl.permute(0, 2, 1)
    xs, fs, xds = [pm[:, :, :3]], [pm[:, :, 3:]], [T(pts_np[:, :3].transpose(0, 2, 1), dev)]
    for i, m in enumerate((net.sa1, net.sa2, net.sa3, net.sa4)):
        nx, nf, nxd = xg._sa_level(m, xs[-1], fs[-1], T(starts[i], dev), dt, xds[-1])
        xs.append(nx)
        fs.append(nf)
        xds.append(nxd)
    up = fs[4]
    for i, m in ((3, net.fp4), (2, net.fp3), (1, net.fp2), (0, net.fp1)):
        up = xg._fp_level(m, xs[i], xs[i + 1], fs[i] if i > 0 else None, up, xds[i], xds[i + 1], dt)
    z = ref_mlp_modes(up, [net.conv1], [net.bn1], dt)
    if keep is not None:
        z = xg._dropout(z, keep, float(net.drop1.p))
    W2 = _param(net.conv2.weight, dt).reshape(net.conv2.weight.shape[0], -1)
    return pl, torch.log_softmax(z @ W2.T + _param(net.conv2.bias, dt), -1)


def _cloud(rng, B, N):
    return np.concatenate([rng.uniform(-8, 8, (B, 2, N)), rng.uniform(-1.5, 1, (B, 1, N)), rng.uniform(0, 1, (B, 1, N))],
                          1).astype(np.float32)


def test_semseg_eval_grads(dev, gemm_mode, restate, ckpt_state):
    """The shipped checkpoint in eval(): points.grad and every parameter's .grad against float64, running statistics and
    num_batches_tracked bit-identical afterwards, no dropout kernel launched, no dropout seed drawn."""
    from pointnet12_b200 import train

    net = _semseg(ckpt_state, dev)
    rng = np.random.default_rng(71)
    B, N = 2, 2048
    pts_np = _cloud(rng, B, N)
    starts = [rng.integers(0, n, B) for n in (N, 1024, 256, 64)]
    state = _bn_state(net)
    seed_before = train._SEED["next"]
    points = T(pts_np, dev).requires_grad_(True)
    G = rng.standard_normal((B, N, 19)).astype(np.float32)

    def step():
        points.grad = None
        net.zero_grad()
        logp = net(points, fps_starts=[T(s, dev) for s in starts])
        (logp * T(G, dev)).sum().backward()
        return logp

    logp = step()
    names = xg._kernel_names(step)
    assert not any("dropout" in n for n in names), sorted(n for n in names if "dropout" in n)
    assert any("bn_eval_bwd" in n for n in names)
    assert train._SEED["next"] == seed_before
    assert _same_state(state, _bn_state(net))
    pl, lp = _semseg_restated(net, pts_np, starts, None, dev)
    (lp * torch.from_numpy(G).to(torch.float64)).sum().backward()
    assert (logp.detach().cpu().double() - lp.detach()).abs().max() < 1e-2
    for c, what in ((slice(0, 3), "xyz"), (slice(3, 4), "reflectance")):
        _close(f"points.grad {what}", points.grad[:, c], pl.grad[:, c], gemm_mode, strict=False)
    _param_grads_close(net, torch.float64, gemm_mode, "semseg")


def test_semseg_eval_autograd_forward_matches_fast_path(dev, ckpt_state):
    """Same seed, same draws: the eval autograd forward samples, groups and interpolates with the fast path's indices
    (equal log-probabilities within 1e-3, equal labels outside a 2e-3 top-2 margin) and leaves the CPU generator in the
    same state; without a gradient-requiring input, or under no_grad, the fast path runs unchanged (same kernels, equal
    output)."""
    from pointnet12_b200 import ops

    net = _semseg(ckpt_state, dev)
    rng = np.random.default_rng(72)
    B, N = 2, 24000
    x = T(_cloud(rng, B, N), dev)
    torch.manual_seed(5)
    fast = net(x)
    gen_fast = torch.get_rng_state()
    torch.manual_seed(5)
    slow = net(x.clone().requires_grad_(True))
    gen_slow = torch.get_rng_state()
    assert torch.equal(gen_fast, gen_slow)
    assert slow.grad_fn is not None and fast.grad_fn is None
    assert (slow.detach() - fast).abs().max() < 1e-3
    top2 = fast.topk(2, -1).values
    sure = (top2[..., 0] - top2[..., 1]) > 2e-3
    assert torch.equal(ops.argmax_labels(slow.detach())[sure], ops.argmax_labels(fast)[sure])
    # the sampling / grouping / 3-NN decisions: the levels' geometry of both paths from the same draws
    from pointnet12_b200.train import semseg_geometry
    from pointnet12_b200.model.pointnet_util import draw_fps_starts

    torch.manual_seed(9)
    st = draw_fps_starts(B, [N, 1024, 256, 64], dev)
    sa_geo, fp_geo = semseg_geometry(net, x, st)
    xpm = x[:, :3].permute(0, 2, 1).contiguous()
    for lvl, m in enumerate((net.sa1, net.sa2, net.sa3, net.sa4)):
        fps = ops.fps(xpm, m.npoint, st[lvl])
        nx = ops.index_points(xpm, fps)
        assert torch.equal(nx, sa_geo[lvl][0]) and torch.equal(ops.ball_query(m.radius, m.nsample, xpm, nx), sa_geo[lvl][1])
        xpm = nx
    # the 3-NN neighbours of every level: the search the fast path runs (pn_three_nn) on the same clouds
    levels = [x[:, :3].permute(0, 2, 1).contiguous()] + [g[0] for g in sa_geo]
    for i in range(4):
        idx, w = ops.three_nn(levels[i], levels[i + 1])
        assert torch.equal(idx, fp_geo[i][0]) and torch.equal(w, fp_geo[i][1])
    # no change without a gradient: the same kernels and the same output with and without no_grad
    torch.manual_seed(5)
    names_plain = xg._kernel_names(lambda: net(x))
    torch.manual_seed(5)
    again = net(x)
    xr = x.clone().requires_grad_(True)
    with torch.no_grad():
        torch.manual_seed(5)
        names_nograd = xg._kernel_names(lambda: net(xr))
        torch.manual_seed(5)
        nog = net(xr)
    assert torch.equal(again, fast) and torch.equal(nog, fast)
    assert names_plain == names_nograd and not any("bn_eval_bwd" in n or "bn_stats" in n for n in names_plain)


# ------------------------------------------------------------------------------------------------ 4. other nets in eval()
def test_cls_msg_eval_grads(dev, gemm_mode, restate):
    """PointNet2ClsMsg in eval(): MSG levels, group-all and the fc head (dropout = identity) against float64."""
    from pointnet12_b200.model.pointnet2 import PointNet2ClsMsg

    rng = np.random.default_rng(81)
    net = _perturbed(PointNet2ClsMsg, 81, dev)
    state = _bn_state(net)
    B, N = 4, 1024
    xyz_np = rng.uniform(-1, 1, (B, 3, N)).astype(np.float32)
    starts = [rng.integers(0, n, B) for n in (N, 512)]
    xyz = T(xyz_np, dev).requires_grad_(True)
    logp, _ = net(xyz, dropout_masks=[torch.zeros((B, 512), dtype=torch.uint8, device=dev)] * 2,   # ignored in eval
                  fps_starts=[T(s, dev) for s in starts])
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    assert _same_state(state, _bn_state(net))
    dt = torch.float64
    xl = _leaf(xyz_np, dt)
    x, f, xd = xl.permute(0, 2, 1), None, T(xyz_np.transpose(0, 2, 1), dev)
    for i, m in enumerate((net.sa1, net.sa2, net.sa3)):
        x, f, xd = xg._sa_level(m, x, f, T(starts[i], dev) if i < 2 else None, dt, xd)
    h = f.reshape(B, 1024)
    for fc, bn in ((net.fc1, net.bn1), (net.fc2, net.bn2)):
        h = ref_mlp_modes(h, [fc], [bn], dt)
    lp = torch.log_softmax(h @ _param(net.fc3.weight, dt).T + _param(net.fc3.bias, dt), -1)
    (lp * torch.from_numpy(G).to(dt)).sum().backward()
    _close("xyz.grad", xyz.grad, xl.grad, gemm_mode, strict=False)
    _param_grads_close(net, dt, gemm_mode, "cls_msg")


@pytest.mark.parametrize("which", ["ssg", "partseg_ssg", "partseg_msg"])
def test_pointnet2_nets_eval_grads(dev, gemm_mode, restate, which):
    """PointNet2ClsSsg, PointNet2PartSegSsg and PointNet2PartSegMsg_one_hot in eval(): the input gradients (xyz; for the
    one-hot net also cls_label, which reaches the loss only through fp1's skip features) and every parameter's .grad
    against the float64 restatement, for direction and size; running statistics untouched."""
    from pointnet12_b200.model import pointnet2 as P2

    rng = np.random.default_rng(91)
    B, N = 2, 1024
    make = {"ssg": P2.PointNet2ClsSsg, "partseg_ssg": lambda: P2.PointNet2PartSegSsg(50),
            "partseg_msg": lambda: P2.PointNet2PartSegMsg_one_hot(50)}[which]
    net = _perturbed(make, 91, dev)
    state = _bn_state(net)
    xyz_np = rng.uniform(-1, 1, (B, 3, N)).astype(np.float32)
    nrm_np = rng.standard_normal((B, 3, N)).astype(np.float32)
    lab_np = np.zeros((B, 16), np.float32)
    lab_np[np.arange(B), rng.integers(0, 16, B)] = 1
    starts = [rng.integers(0, n, B) for n in (N, 512)]
    xyz = T(xyz_np, dev).requires_grad_(True)
    label = T(lab_np, dev).requires_grad_(True)
    fs_dev = [T(s, dev) for s in starts]
    if which == "partseg_msg":
        out = net(xyz, T(nrm_np, dev), label, fps_starts=fs_dev)
    else:
        out = net(xyz, fps_starts=fs_dev)
    logp = out[0] if isinstance(out, tuple) else out
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    assert _same_state(state, _bn_state(net))
    dt = torch.float64
    xl, ll = _leaf(xyz_np, dt), _leaf(lab_np, dt)
    x0 = xl.permute(0, 2, 1)
    nrm = torch.from_numpy(nrm_np.transpose(0, 2, 1).astype(np.float64))
    xs, fs, xds = [x0], [nrm if which == "partseg_msg" else None], [T(xyz_np.transpose(0, 2, 1), dev)]
    for i, m in enumerate((net.sa1, net.sa2, net.sa3)):
        nx, nf, nxd = xg._sa_level(m, xs[-1], fs[-1], T(starts[i], dev) if i < 2 else None, dt, xds[-1])
        xs.append(nx)
        fs.append(nf)
        xds.append(nxd)
    if which == "ssg":
        h = fs[3].reshape(B, 1024)
        for fc, bn in ((net.fc1, net.bn1), (net.fc2, net.bn2)):
            h = ref_mlp_modes(h, [fc], [bn], dt)
        lp = torch.log_softmax(h @ _param(net.fc3.weight, dt).T + _param(net.fc3.bias, dt), -1)
    else:
        f2 = xg._fp_level(net.fp3, xs[2], xs[3], fs[2], fs[3], xds[2], xds[3], dt)
        f1 = xg._fp_level(net.fp2, xs[1], xs[2], fs[1], f2, xds[1], xds[2], dt)
        skip = None
        if which == "partseg_msg":
            skip = torch.cat([ll[:, None, :].expand(B, N, 16), x0, nrm], -1)
        f0 = xg._fp_level(net.fp1, xs[0], xs[1], skip, f1, xds[0], xds[1], dt)
        z = ref_mlp_modes(f0, [net.conv1], [net.bn1], dt)
        W2 = _param(net.conv2.weight, dt).reshape(net.conv2.weight.shape[0], -1)
        lp = torch.log_softmax(z @ W2.T + _param(net.conv2.bias, dt), -1)
    (lp * torch.from_numpy(G).to(dt)).sum().backward()
    _close("xyz.grad", xyz.grad, xl.grad, gemm_mode, strict=False)
    if which == "partseg_msg":
        _close("cls_label.grad", label.grad, ll.grad, gemm_mode, strict=False)
    _param_grads_close(net, dt, gemm_mode, which)


# float64 restatement of model/pointnet.py on point-major rows [B, N, C] (eval-mode BatchNorm via ref_mlp_modes' rule)
def _lin(x, mod, dt):
    W = _param(mod.weight, dt).reshape(mod.weight.shape[0], -1)
    return x @ W.T + _param(mod.bias, dt)


def _bn(x, bn, dt, relu=True):
    from pointnet12_b200 import ops

    assert ops.uses_running_stats(bn)
    mu, var = bn.running_mean.detach().cpu().to(dt), bn.running_var.detach().cpu().to(dt)
    y = (x - mu) / torch.sqrt(var + bn.eps) * _param(bn.weight, dt) + _param(bn.bias, dt)
    return torch.relu(y) if relu else y


def ref_stn(stn, x, dt):
    h = _bn(_lin(x, stn.conv1, dt), stn.bn1, dt)
    h = _bn(_lin(h, stn.conv2, dt), stn.bn2, dt)
    g = _bn(_lin(h, stn.conv3, dt), stn.bn3, dt).max(1)[0]
    g = _bn(_lin(g, stn.fc1, dt), stn.bn4, dt)
    g = _bn(_lin(g, stn.fc2, dt), stn.bn5, dt)
    return (_lin(g, stn.fc3, dt) + torch.eye(stn.k, dtype=dt).flatten()).view(-1, stn.k, stn.k)


def ref_encoder(enc, x, dt):
    """-> (global [B,1024], pointfeat [B,N,64], trans_feat)."""
    x = torch.bmm(x, ref_stn(enc.stn, x, dt))
    x = _bn(_lin(x, enc.conv1, dt), enc.bn1, dt)
    tf = None
    if enc.feature_transform:
        tf = ref_stn(enc.fstn, x, dt)
        x = torch.bmm(x, tf)
    h = _bn(_lin(x, enc.conv2, dt), enc.bn2, dt)
    return _bn(_lin(h, enc.conv3, dt), enc.bn3, dt, relu=False).max(1)[0], x, tf


def ref_pointnet(which, net, x, label, dt):
    """The outputs of each net as a list of tensors (point-major where the net's own output is)."""
    B, N = x.shape[0], x.shape[1]
    if which == "stn":
        return [ref_stn(net, x, dt)]
    if which == "encoder":
        g, pf, _ = ref_encoder(net, x, dt)
        return [torch.cat([g[:, None, :].expand(B, N, 1024), pf], -1)]
    if which == "cls":
        g, _, _ = ref_encoder(net.feat, x, dt)
        h = _bn(_lin(g, net.fc1, dt), net.bn1, dt)
        h = _bn(_lin(h, net.fc2, dt), net.bn2, dt)          # dropout is the identity in eval()
        return [torch.log_softmax(_lin(h, net.fc3, dt), -1)]
    if which == "seg":
        g, pf, _ = ref_encoder(net.feat, x, dt)
        h = torch.cat([g[:, None, :].expand(B, N, 1024), pf], -1)
        for conv, bn in ((net.conv1, net.bn1), (net.conv2, net.bn2), (net.conv3, net.bn3)):
            h = _bn(_lin(h, conv, dt), bn, dt)
        return [torch.log_softmax(_lin(h, net.conv4, dt), -1)]
    x = torch.bmm(x, ref_stn(net.stn, x, dt))                # PointNetDenseCls
    o1 = _bn(_lin(x, net.conv1, dt), net.bn1, dt)
    o2 = _bn(_lin(o1, net.conv2, dt), net.bn2, dt)
    o3 = _bn(_lin(o2, net.conv3, dt), net.bn3, dt)
    t = torch.bmm(o3, ref_stn(net.fstn, o3, dt))
    o4 = _bn(_lin(t, net.conv4, dt), net.bn4, dt)
    o5 = _bn(_lin(o4, net.conv5, dt), net.bn5, dt, relu=False)
    om = o5.max(1)[0]
    h = _bn(_lin(om, net.fc1, dt), net.bnc1, dt)
    h = _bn(_lin(h, net.fc2, dt), net.bnc2, dt)
    cls = _lin(h, net.fc3, dt)
    cat = torch.cat([torch.cat([om, label], 1)[:, None, :].expand(B, N, 2048 + label.shape[1]), o1, o2, o3, o4, o5], -1)
    for conv, bn in ((net.convs1, net.bns1), (net.convs2, net.bns2), (net.convs3, net.bns3)):
        cat = _bn(_lin(cat, conv, dt), bn, dt)
    return [cls, torch.log_softmax(_lin(cat, net.convs4, dt), -1)]


@pytest.mark.parametrize("which", ["seg", "cls", "dense", "stn", "encoder"])
def test_pointnet_nets_eval_grads(dev, gemm_mode, restate, which):
    """PointNetSeg(19, 4, True), PointNetCls, PointNetDenseCls, STN3d and PointNetEncoder in eval(): a grad_fn, the fast
    eval output up to rounding, and the input gradient and every parameter's .grad against the float64 restatement of
    model/pointnet.py (direction and size); running statistics untouched."""
    from pointnet12_b200.model import pointnet as PN

    rng = np.random.default_rng(101)
    B, N = 2, 512
    D = {"seg": 4, "cls": 3, "dense": 3, "stn": 3, "encoder": 3}[which]
    make = {"seg": lambda: PN.PointNetSeg(19, 4, True), "cls": lambda: PN.PointNetCls(5),
            "dense": lambda: PN.PointNetDenseCls(16, 50), "stn": PN.STN3d,
            "encoder": lambda: PN.PointNetEncoder(global_feat=False, input_dims=3)}[which]
    net = _perturbed(make, 101, dev)
    state = _bn_state(net)
    x_np = rng.uniform(-1, 1, (B, D, N)).astype(np.float32)
    lab_np = np.eye(16, dtype=np.float32)[:B]
    args = (T(lab_np, dev),) if which == "dense" else ()
    with torch.no_grad():
        fast = net(T(x_np, dev), *args)
    xr = T(x_np, dev).requires_grad_(True)
    out = net(xr, *args)
    pick = {"seg": [0], "cls": [0], "dense": [0, 1], "stn": [None], "encoder": [0]}[which]
    got = [out if i is None else out[i] for i in pick]
    fast = [fast if i is None else fast[i] for i in pick]
    for o, f in zip(got, fast):
        assert o.grad_fn is not None and rl2(o.detach(), f) < 1e-3
    Gs = [rng.standard_normal(o.shape).astype(np.float32) for o in got]
    sum((o * T(g, dev)).sum() for o, g in zip(got, Gs)).backward()
    assert _same_state(state, _bn_state(net))
    dt = torch.float64
    xl = _leaf(x_np, dt)
    refs = ref_pointnet(which, net, xl.permute(0, 2, 1), torch.from_numpy(lab_np.astype(np.float64)), dt)
    if which == "encoder":
        refs = [refs[0].permute(0, 2, 1)]                    # the encoder returns [B, 1088, N]
    sum((r * torch.from_numpy(g).to(dt)).sum() for r, g in zip(refs, Gs)).backward()
    _close("x.grad", xr.grad, xl.grad, gemm_mode, strict=False)
    _param_grads_close(net, dt, gemm_mode, which)

# ------------------------------------------------------------------------------------------------ 5. frozen BatchNorm
@pytest.mark.parametrize("frozen", ["all", "half"])
def test_semseg_train_step_frozen_bn(dev, gemm_mode, restate, ckpt_state, frozen):
    """A PointNet2SemSeg train step with every BatchNorm (or every other one) in eval(): frozen layers normalise with their
    running statistics, which stay bit-identical; the other layers update theirs; gradients against float64."""
    from pointnet12_b200.train import semseg_forward_train

    net = _semseg(ckpt_state, dev).train()
    bns = [m for m in net.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
    frozen_bns = bns if frozen == "all" else bns[::2]
    for m in frozen_bns:
        m.eval()
    before = {id(m): [t.clone() for t in (m.running_mean, m.running_var, m.num_batches_tracked)] for m in bns}
    rng = np.random.default_rng(111)
    B, N = 2, 2048
    pts_np = _cloud(rng, B, N)
    starts = [rng.integers(0, n, B) for n in (N, 1024, 256, 64)]
    keep = (rng.random((B * N, 128)) > 0.5).astype(np.uint8)
    points = T(pts_np, dev).requires_grad_(True)
    logp = semseg_forward_train(net, points, fps_starts=[T(s, dev) for s in starts], dropout_mask=T(keep, dev))
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    for m in bns:
        same = all(torch.equal(a, b) for a, b in zip(before[id(m)], (m.running_mean, m.running_var, m.num_batches_tracked)))
        assert same == (m in frozen_bns)
    # the restatement reads the running statistics the frozen layers used (unchanged) and batch statistics elsewhere
    pl, lp = _semseg_restated(net, pts_np, starts, keep, dev)
    (lp * torch.from_numpy(G).to(torch.float64)).sum().backward()
    if frozen == "all":
        _close("points.grad", points.grad, pl.grad, gemm_mode, strict=False)
        _param_grads_close(net, torch.float64, gemm_mode, "frozen")
        return
    # batch coupling through the live layers: the train-mode bounds of test_gpu_xyz_grad.py (a conv bias ahead of a live
    # BatchNorm has a gradient of rounding noise only, so the weights are compared)
    xg._net_close("points.grad", points.grad, pl.grad, gemm_mode)
    for name, p in net.named_parameters():
        leaf = LEAVES.get((id(p), torch.float64))
        if name.endswith("weight") and leaf is not None and leaf.grad is not None:
            xg._net_close(f"{name}.grad", p.grad, leaf.grad, gemm_mode)


def test_graphed_train_step_frozen_bn_and_mode_toggle(dev, ckpt_state):
    """GraphedTrainStep with frozen BatchNorm matches the eager step; toggling a BatchNorm's mode after capture makes the
    runner capture again instead of replaying a graph of the other mode."""
    from pointnet12_b200.train import FlatAdam, GraphedTrainStep, cross_entropy, semseg_forward_train

    rng = np.random.default_rng(121)
    B, N = 2, 4096
    x = T(_cloud(rng, B, N), dev)
    target = T(rng.integers(0, 19, (B, N)), dev)

    def make():
        net = _semseg(ckpt_state, dev).train()
        for m in net.modules():
            if isinstance(m, (torch.nn.modules.batchnorm._BatchNorm, torch.nn.Dropout)):
                m.eval()          # (dropout off too: the graph and the eager step draw their masks from other streams)
        return net

    a, b = make(), make()
    opt_a, opt_b = FlatAdam(a.parameters(), lr=1e-3), FlatAdam(b.parameters(), lr=1e-3)
    step = GraphedTrainStep(a, opt_a)
    for i in range(3):
        torch.manual_seed(100 + i)
        la = step(x, target)
        torch.manual_seed(100 + i)
        from pointnet12_b200.model.pointnet_util import draw_fps_starts

        st = draw_fps_starts(B, [N, 1024, 256, 64], dev)
        lb = cross_entropy(semseg_forward_train(b, x, fps_starts=st), target)
        opt_b.zero_grad()
        lb.backward()
        opt_b.step()
        assert abs(float(la) - float(lb)) < 1e-3 * max(1.0, abs(float(lb))), (i, float(la), float(lb))
    assert rl2(opt_a.flat, opt_b.flat) < 1e-4
    assert len(step._graphs) == 1
    a.bn1.train()
    step(x, target)
    assert len(step._graphs) == 2
    a.bn1.eval()
    step(x, target)
    assert len(step._graphs) == 2


def test_graphed_step_recaptures_on_mode_toggle(dev):
    """GraphedStep (PointNetSeg) with frozen BatchNorm: a graph per set of BatchNorm / dropout modes -- a toggle after capture
    captures again, toggling back replays the first graph -- and the frozen statistics do not move."""
    from pointnet12_b200.model.pointnet import PointNetSeg
    from pointnet12_b200.train import FlatAdam, GraphedStep, cross_entropy

    torch.manual_seed(131)
    net = PointNetSeg(19, 4, False).to(dev).train()
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.eval()
    frozen = _bn_state(net)
    step = GraphedStep(net, FlatAdam(net.parameters(), lr=1e-4), lambda n, x, t: cross_entropy(n(x)[0], t))
    x = torch.rand((2, 4, 1024), device=dev)
    t = torch.randint(0, 19, (2, 1024), device=dev)
    l0 = float(step(x, t))
    assert len(step._graphs) == 1 and np.isfinite(l0)
    assert _same_state(frozen, _bn_state(net))
    net.bn1.train()
    step(x, t)
    assert len(step._graphs) == 2
    net.bn1.eval()
    step(x, t)
    assert len(step._graphs) == 2
