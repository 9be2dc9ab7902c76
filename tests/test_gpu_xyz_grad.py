"""Gradients with respect to the point coordinates through the PointNet++ blocks in train() mode, against float64.

The reference builds its blocks from torch expressions, so autograd differentiates them in the coordinates too: through the
sampled centroids (new_xyz = xyz[fps_idx]), the grouping (xyz[idx] - new_xyz, or xyz itself for group-all) and the 3-NN
interpolation weights (1 / square_distance).  The yardstick is a float64 restatement of those expressions in torch on the
CPU, differentiated by torch autograd, with two rules that keep the comparison deterministic:

  - the discrete decisions come from our forward: FPS indices, ball-query indices, 3-NN indices and dropout masks (other
    tests show they are bit-exact with the reference), so the float64 run cannot pick other neighbours;
  - the clamp mask of the interpolation and r = 1/max(d, 1e-10) come from the float32 SQDIST values (SURVEY App. B,
    restated in numpy float32): the values the reference's float32 forward uses.  Everything after them is float64.

Elementwise bound, as in tests/test_gpu_train_edges.py:  |got - want| <= (4 * E32 + 1e-6) * scale (+ the float32 atomic
accumulation bound 4 m 2^-24 sum|terms| for values that m scattered terms add up to), where scale is the size of the terms
the value is built from and E32 the largest |ref32 - want| / scale of the same restatement run in float32 by torch's CPU
autograd.  With the tensor-core GEMM engine, max-pool arg-max and ReLU flips move whole gradient rows (DESIGN.md section 9):
those comparisons are flip-tolerant, and whole nets are compared on the direction and size of the gradient.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

K_TORCH = 4.0
FLOOR = 1e-6
U32 = 2.0 ** -24
CLAMP = 1e-10


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


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64) if isinstance(t, torch.Tensor) else np.asarray(t, np.float64)


def within(what, got, want, ref32, scale, extra=0.0):
    """|got - want| <= (K_TORCH * E32 + FLOOR) * scale + extra elementwise (see the module docstring)."""
    got, want, ref32 = _np(got), _np(want), _np(ref32)
    scale = np.broadcast_to(np.maximum(np.asarray(scale, np.float64), 1e-30), want.shape)
    e32 = float(np.max(np.abs(ref32 - want) / scale, initial=0.0))
    bound = (K_TORCH * e32 + FLOOR) * scale + extra
    err = np.abs(got - want)
    bad = ~(err <= bound)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / bound, 0)), want.shape)
        pytest.fail(f"{what}: {int(bad.sum())} of {want.size} elements out of bound; worst at {i}: got {got[i]!r}, "
                    f"want {want[i]!r}, bound {bound[i]:.3g} (E32 {e32:.3g}, scale {scale[i]:.3g})")


def rl2(a, b):
    a, b = _np(a), _np(b)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def close_but_for_flips(what, got, want):
    """tests/test_gpu_train.py::_close_but_for_flips for the tensor-core engine: a max-pool arg-max flip (two activations
    within the engines' ~1e-5 rounding difference) routes a gradient row to another point.  Tiny median error, fewer than 1 %
    of the entries off by more than 1e-4 of the largest, and a loose L2 bound on everything."""
    err = np.abs(_np(got) - _np(want)).reshape(-1)
    scale = np.abs(_np(want)).max()
    assert np.median(err) < 1e-5 * scale and (err > 1e-4 * scale).mean() < 0.01, (what, np.median(err) / scale,
                                                                                 (err > 1e-4 * scale).mean())
    assert rl2(got, want) < 2e-2, (what, rl2(got, want))


# ------------------------------------------------------------------------------------------------ float32 SQDIST
def _fma32(a, b, c):
    # a*b of two float32 is exact in float64; the float64 sum then rounds once more before the float32 rounding (a double
    # rounding that differs from the fused operation for about one input in 2^29)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def sqdist32(a, b):
    """SQDIST of SURVEY App. B in numpy float32: dot = fma(az,bz, fma(ay,by, ax*bx)); ((-2*dot) + |a|^2) + |b|^2."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    dot = _fma32(a[..., 2], b[..., 2], _fma32(a[..., 1], b[..., 1], a[..., 0] * b[..., 0]))
    sa = (a[..., 0] * a[..., 0] + a[..., 1] * a[..., 1]) + a[..., 2] * a[..., 2]
    sb = (b[..., 0] * b[..., 0] + b[..., 1] * b[..., 1]) + b[..., 2] * b[..., 2]
    return ((np.float32(-2.0) * dot) + sa) + sb


def _gather(x, idx):
    """x [B,N,C], idx [B,...] -> [B,...,C] (index_points)."""
    B = x.shape[0]
    bi = torch.arange(B).view((B,) + (1,) * (idx.dim() - 1))
    return x[bi, idx]


# ------------------------------------------------------------------------------------------------ torch restatements
def ref_interp(xyz1, xyz2, p2, idx, d32):
    """interpolated_points of pointnet_util.py:295-307 for S > 1 (xyz1 [B,N,3], xyz2 [B,S,3], p2 [B,S,D2], idx [B,N,3]),
    with the float32 SQDIST values d32 [B,N,3] of the chosen neighbours injected: the clamp decision and r = 1/dc take
    their values from it, the derivative of d is 2 (a - b) in the run's dtype."""
    dt = xyz1.dtype
    d = ((xyz1[:, :, None, :] - _gather(xyz2, idx)) ** 2).sum(-1)
    d = d - d.detach() + torch.from_numpy(d32.astype(np.float64)).to(dt)
    clamped = torch.from_numpy(d32 < np.float32(CLAMP))
    dc = torch.where(clamped, torch.full_like(d, CLAMP), d)            # dists[dists < 1e-10] = 1e-10: no gradient there
    r = 1.0 / dc
    r32 = np.float32(1.0) / np.where(d32 < np.float32(CLAMP), np.float32(CLAMP), d32)
    r = r - r.detach() + torch.from_numpy(r32.astype(np.float64)).to(dt)
    w = r / r.sum(-1, keepdim=True)
    return (_gather(p2, idx) * w[..., None]).sum(2)


def ref_mlp(x, convs, bns, dt, taps=None):
    """conv 1x1 -> BatchNorm with batch statistics (biased variance) -> ReLU per layer on rows [..., cin]; taps (a list)
    receives the first layer's output y (retain_grad) and weight for the scale of the input gradient."""
    for li, (conv, bn) in enumerate(zip(convs, bns)):
        W = conv.weight.detach().cpu().to(dt).reshape(conv.weight.shape[0], -1)
        y = x @ W.T + conv.bias.detach().cpu().to(dt)
        if li == 0 and taps is not None:
            y.retain_grad()
            taps.append((y, W))
        flat = y.reshape(-1, y.shape[-1])
        mu = flat.mean(0)
        var = ((flat - mu) ** 2).mean(0)
        y = (y - mu) / torch.sqrt(var + bn.eps) * bn.weight.detach().cpu().to(dt) + bn.bias.detach().cpu().to(dt)
        x = torch.relu(y)
    return x


def ref_sa(xyz, pts, fps_idx, idx, convs, bns, dt, msg=False, taps=None):
    """sample_and_group (+ the MSG order) / sample_and_group_all + MLP + max: xyz [B,N,3], pts [B,N,D] or None,
    fps_idx [B,S] (None: group-all), idx [B,S,K] -> (new_xyz [B,S,3], pooled [B,S,C'])."""
    if fps_idx is None:
        new_xyz = torch.zeros((xyz.shape[0], 1, 3), dtype=dt)
        gx = xyz[:, None]
        gp = pts[:, None] if pts is not None else None
    else:
        new_xyz = _gather(xyz, fps_idx)
        gx = _gather(xyz, idx) - new_xyz[:, :, None, :]
        gp = _gather(pts, idx) if pts is not None else None
    g = gx if gp is None else (torch.cat([gp, gx], -1) if msg else torch.cat([gx, gp], -1))
    return new_xyz, ref_mlp(g, convs, bns, dt, taps).max(2)[0]


def ref_fp(xyz1, xyz2, p1, p2, idx, d32, convs, bns, dt, taps=None):
    """PointNetFeaturePropagation.forward (:283-312) point-major: -> [B,N,C']."""
    B, N, _ = xyz1.shape
    interp = p2.expand(B, N, p2.shape[2]) if xyz2.shape[1] == 1 else ref_interp(xyz1, xyz2, p2, idx, d32)
    x = interp if p1 is None else torch.cat([p1, interp], -1)
    return ref_mlp(x, convs, bns, dt, taps)


def _nn_geometry(x1, x2):
    """Our 3-NN on the float32 clouds (point-major device tensors) -> (idx [B,N,3] numpy, d32 [B,N,3])."""
    from pointnet12_b200 import ops

    if x2.shape[1] == 1:
        return np.zeros((x1.shape[0], x1.shape[1], 3), np.int64), None
    idx, _ = ops.three_nn(x1, x2)
    idx = idx.cpu().numpy()
    a, b = x1.detach().cpu().numpy(), x2.detach().cpu().numpy()
    return idx, sqdist32(a[:, :, None, :], b[np.arange(b.shape[0])[:, None, None], idx])


def _leaf(a, dt):
    return torch.tensor(np.asarray(a), dtype=dt, requires_grad=True)


# ------------------------------------------------------------------------------------------------ 1. the kernels
def _ball_rows(B, S, K, N, rng):
    """Ball-query rows as the net produces them: u unique hits padded with the first (u = 1, 2, 5, K per quarter)."""
    idx = np.empty((B, S, K), np.int64)
    for b in range(B):
        for s in range(S):
            u = (1, 2, 5, K)[s % 4]
            hits = rng.choice(N, u, replace=False)
            idx[b, s, :u] = hits
            idx[b, s, u:] = hits[0]
        idx[b, 1, 1] = N - 1
    return idx


@pytest.mark.parametrize("order,D", [("ssg", 0), ("ssg", 13), ("msg", 13), ("msg", 64), ("all", 5)])
def test_group_backward_xyz_kernel(dev, order, D):
    """pn_group_bwd_xyz_f32: scatter of the xyz_rel columns and -sum_k for the centroid (none for group-all)."""
    from pointnet12_b200 import ops

    rng = np.random.default_rng(len(order) * 100 + D)
    B, N = 2, 700
    S, K = (1, N) if order == "all" else (64, 32)
    idx = np.broadcast_to(np.arange(N), (B, 1, N)).copy() if order == "all" else _ball_rows(B, S, K, N, rng)
    col0 = D if order == "msg" else 0
    width = D + 3
    dg = torch.zeros((B * S * K, width + 3), device=dev)                # ldg > width
    vals = rng.standard_normal((B * S * K, width)).astype(np.float32)
    dg[:, :width] = T(vals, dev)
    dxyz, dnew = ops.group_backward_xyz(dg[:, :width], col0, T(idx, dev), N, recentred=order != "all")
    # float64 restatement by autograd: grouped_xyz = xyz[idx] - new_xyz (group-all: xyz, not recentred)
    xyz = _leaf(np.zeros((B, N, 3)), torch.float64)
    new = _leaf(np.zeros((B, S, 3)), torch.float64)
    G = torch.from_numpy(vals[:, col0:col0 + 3].astype(np.float64)).view(B, S, K, 3)
    gx = _gather(xyz, torch.from_numpy(idx)) - (0 if order == "all" else new[:, :, None, :])
    (gx * G).sum().backward()
    terms = np.abs(vals[:, col0:col0 + 3].astype(np.float64)).reshape(B, S * K, 3)
    cnt, asum = np.zeros((B, N, 1)), np.zeros((B, N, 3))
    for b in range(B):
        np.add.at(cnt[b], idx[b].reshape(-1), 1.0)
        np.add.at(asum[b], idx[b].reshape(-1), terms[b])
    within("dxyz", dxyz, xyz.grad, xyz.grad, asum, 4 * cnt * U32 * asum)
    if order == "all":
        assert dnew is None
    else:
        within("dnew_xyz", dnew, new.grad, new.grad, terms.reshape(B, S, K, 3).sum(2), 4 * K * U32 * terms.reshape(B, S, K, 3).sum(2))
    if order != "all":
        assert cnt[:, N - 1].min() > 0 and (idx[:, :, 1] == idx[:, :, 0]).any()    # the padding repeats are there


def _fp_clouds(B, N, S, rng):
    """Coarse cloud xyz2 [B,S,3] and fine cloud xyz1 [B,N,3] with the hazards of the interpolation weights: fine points
    that coincide with coarse points, exact duplicates in the fine cloud, pairs at d < 1e-10 and just above it (near the
    origin, where the float32 expansion formula resolves 1e-10), and points equidistant from three coarse points."""
    xyz2 = rng.uniform(-1, 1, (B, S, 3)).astype(np.float32)
    xyz1 = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    q = max(N // 10, 1)
    for b in range(B):
        xyz1[b, :q] = xyz2[b, rng.integers(0, S, q)]                        # coincident with a coarse point
        xyz1[b, q:2 * q] = xyz1[b, rng.integers(2 * q, N, q)]               # exact duplicates of other fine points
        if S == 3:                                                          # every fine point has the same three
            for k in range(3):
                ang = 2 * np.pi * k / 3
                xyz2[b, k] = [0.5 * np.cos(ang), 0.5 * np.sin(ang), 0.1]
            xyz1[b, 2 * q] = [0.0, 0.0, 0.1]                                # equidistant from all three
        elif S >= 8 and N >= 3 * q + 8:
            xyz2[b, 0] = [1e-3, -2e-3, 1.5e-3]
            xyz2[b, 1] = [-3e-3, 1e-3, 2e-3]
            for i, off in enumerate((4e-6, 6e-6, 9e-6, 1.05e-5, 1.2e-5, 2e-5)):   # d from 1.6e-11 to 4e-10
                c = xyz2[b, i % 2]
                u = rng.standard_normal(3)
                xyz1[b, 2 * q + i] = (c + off * u / np.linalg.norm(u)).astype(np.float32)
            for i in range(2):                                              # equidistant from three coarse points
                ctr = rng.uniform(-0.5, 0.5, 3)
                for k in range(3):
                    ang = 2 * np.pi * k / 3
                    xyz2[b, 2 + 3 * i + k] = (ctr + 0.05 * np.array([np.cos(ang), np.sin(ang), 0.0])).astype(np.float32)
                xyz1[b, 2 * q + 6 + i] = ctr.astype(np.float32)
    return xyz1, xyz2


def _interp_scale(x1, x2, idx, d32, w, gabs):
    """Sizes of the terms of dxyz1 / dxyz2: with G_k = sum_c |dinterp_c p2[idx_k]_c| (gabs), M = sum_k w_k G_k,
    t_k = 2 (G_k + M) / R r_k^2 |a - b_k| for the unclamped neighbours."""
    B, N = idx.shape[:2]
    live = d32 >= np.float32(CLAMP)
    r = 1.0 / np.where(live, d32, np.float32(CLAMP)).astype(np.float64)
    R = r.sum(-1, keepdims=True)
    M = (w * gabs).sum(-1, keepdims=True)
    nb = x2[np.arange(B)[:, None, None], idx]
    t = 2 * (live * (gabs + M) / R * r * r)[..., None] * np.abs(x1[:, :, None, :] - nb)      # [B,N,3,3]
    s1 = t.sum(2)
    s2, cnt = np.zeros(x2.shape), np.zeros(x2.shape[:2] + (1,))
    for b in range(B):
        for k in range(3):
            np.add.at(s2[b], idx[b, :, k], t[b, :, k])
            np.add.at(cnt[b], idx[b, :, k], 1.0)
    return s1, s2, cnt


@pytest.mark.parametrize("S,N,D1,D2", [(3, 400, 0, 128), (3, 400, 22, 256), (1024, 6000, 0, 128), (1024, 6000, 64, 256),
                                       (1024, 6000, 22, 128), (1024, 24000, 0, 128)])
def test_three_interpolate_backward_xyz_kernel(dev, S, N, D1, D2):
    """pn_three_interpolate_bwd_xyz_f32 element by element against the float64 restatement (24000 x 1024 is C2's fp1), and
    its dp1 / dp2 against pn_three_interpolate_bwd_f32.  D1 = 22: the unvectorised path."""
    from pointnet12_b200 import ops

    rng = np.random.default_rng(S + N + D1 + D2)
    B = 2
    x1, x2 = _fp_clouds(B, N, S, rng)
    p2 = rng.standard_normal((B, S, D2)).astype(np.float32)
    vals = rng.standard_normal((B * N, D1 + D2)).astype(np.float32)
    dx = torch.zeros((B * N, D1 + D2 + 4), device=dev)
    dx[:, :D1 + D2] = T(vals, dev)
    dx = dx[:, :D1 + D2]
    x1d, x2d = T(x1, dev), T(x2, dev)
    idx_t, w_t = ops.three_nn(x1d, x2d)
    dp1, dp2, dxyz1, dxyz2 = ops.three_interpolate_backward_xyz(dx, D1, D2, idx_t, w_t, T(p2, dev), x1d, x2d)
    ep1, ep2 = ops.three_interpolate_backward(dx, D1, D2, idx_t, w_t, S)
    if D1:
        assert torch.equal(dp1, ep1)
    else:
        assert dp1 is None
    idx, w = idx_t.cpu().numpy(), w_t.cpu().numpy().astype(np.float64)
    d32 = sqdist32(x1[:, :, None, :], x2[np.arange(B)[:, None, None], idx])
    g = vals[:, D1:].astype(np.float64).reshape(B, N, D2)
    asum2, cnt = np.zeros((B, S, D2)), np.zeros((B, S, 1))
    for b in range(B):
        for k in range(3):
            np.add.at(asum2[b], idx[b, :, k], np.abs(g[b] * w[b, :, k:k + 1]))
            np.add.at(cnt[b], idx[b, :, k], 1.0)
    assert (np.abs(_np(dp2) - _np(ep2)) <= 8 * cnt * U32 * asum2 + 1e-30).all()    # the same sums, atomics in another order
    out = {}
    for dt in (torch.float64, torch.float32):
        a, b_, p = _leaf(x1, dt), _leaf(x2, dt), _leaf(p2, dt)
        interp = ref_interp(a, b_, p, torch.from_numpy(idx), d32)
        (interp * torch.from_numpy(g).to(dt)).sum().backward()
        out[dt] = (a.grad, b_.grad)
    gabs = np.abs(g)[:, :, None, :] @ np.abs(p2[np.arange(B)[:, None, None], idx].astype(np.float64)).transpose(0, 1, 3, 2)
    s1, s2, c2 = _interp_scale(x1.astype(np.float64), x2.astype(np.float64), idx, d32, w, gabs[:, :, 0, :])
    within("dxyz1", dxyz1, out[torch.float64][0], out[torch.float32][0], s1)
    within("dxyz2", dxyz2, out[torch.float64][1], out[torch.float32][1], s2, 4 * c2 * U32 * s2)
    live = d32 >= np.float32(CLAMP)
    if S >= 1024:      # the hazards are in the data: clamped and barely unclamped pairs, coincident points
        assert (~live).any() and (live & (d32 < np.float32(1e-9))).any()


# ------------------------------------------------------------------------------------------------ 2. blocks in train() mode
def _seeded(make, seed, dev):
    torch.manual_seed(seed)
    m = make()
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.normal_(0, 0.2)
    return m.to(dev).train()


def _first_layer_scale(taps, cols):
    """|dy1| |W1| for the given input columns of the first layer: the size of the terms of its input gradient."""
    y, W = taps[0]
    return (y.grad.abs().reshape(-1, W.shape[0]) @ W.abs()[:, cols]).reshape(y.shape[:-1] + (len(cols),))


def _check(what, got, want, ref32, scale, mode):
    if mode == "fp32":
        within(what, got, want, ref32, scale)
    else:
        close_but_for_flips(what, got, want)


@pytest.mark.parametrize("kind", ["ssg", "msg", "all"])
def test_sa_block_xyz_grad(dev, gemm_mode, kind):
    """SSG (K = 32), MSG (three scales, [features, xyz_rel]) and group-all set abstraction in train() mode: xyz.grad, with
    gradients arriving through the pooled features AND the returned new_xyz (the centroid path)."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model import pointnet_util as pu

    rng = np.random.default_rng({"ssg": 1, "msg": 2, "all": 3}[kind])
    B, N, D = 2, 512, 16
    if kind == "ssg":
        mod = _seeded(lambda: pu.PointNetSetAbstraction(128, 0.3, 32, D + 3, [32, 32, 64], False), 11, dev)
    elif kind == "msg":
        mod = _seeded(lambda: pu.PointNetSetAbstractionMsg(128, [0.2, 0.3, 0.5], [16, 32, 64], D,
                                                            [[16, 16, 32], [32, 32, 64], [32, 48, 64]]), 12, dev)
    else:
        mod = _seeded(lambda: pu.PointNetSetAbstraction(None, None, None, D + 3, [32, 64, 128], True), 13, dev)
    xyz_np = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    pts_np = rng.standard_normal((B, N, D)).astype(np.float32)
    start = rng.integers(0, N, B)
    xyz = T(xyz_np.transpose(0, 2, 1), dev).requires_grad_(True)
    pts = T(pts_np.transpose(0, 2, 1), dev).requires_grad_(True)
    new_xyz, out = mod(xyz, pts, start_idx=T(start, dev))
    G = rng.standard_normal(out.shape).astype(np.float32)
    Gn = rng.standard_normal(new_xyz.shape).astype(np.float32) if kind != "all" else None
    loss = (out * T(G, dev)).sum() + ((new_xyz * T(Gn, dev)).sum() if Gn is not None else 0)
    loss.backward()
    assert xyz.grad is not None and pts.grad is not None
    # the decisions of our forward
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
    res = {}
    for dt in (torch.float64, torch.float32):
        a, p = _leaf(xyz_np, dt), _leaf(pts_np, dt)
        outs, taps = [], []
        for ball, (convs, bns) in zip(balls, blocks):
            tap = []
            nx, o = ref_sa(a, p, torch.from_numpy(fps.cpu().numpy()) if fps is not None else None,
                           torch.from_numpy(ball.cpu().numpy()) if ball is not None else None, convs, bns, dt,
                           msg=kind == "msg", taps=tap)
            outs.append(o)
            taps.append(tap)
        o = torch.cat(outs, -1).permute(0, 2, 1)
        ref_loss = (o * torch.from_numpy(G).to(dt)).sum()
        if Gn is not None:
            ref_loss = ref_loss + (nx.permute(0, 2, 1) * torch.from_numpy(Gn).to(dt)).sum()
        ref_loss.backward()
        res[dt] = (a.grad, taps)
    want, taps = res[torch.float64]
    # scale: the first-layer input-gradient terms of the xyz_rel columns, scattered to their points with |.|, plus the
    # centroid terms (sum over the group, and the incoming gradient of new_xyz) at the sampled points
    scale = np.zeros((B, N, 3))
    for ball, tap in zip(balls, taps):
        cols = [D, D + 1, D + 2] if kind == "msg" else [0, 1, 2]
        s = _np(_first_layer_scale(tap, cols))
        if ball is None:
            scale += s[:, 0]
            continue
        bi = ball.cpu().numpy()
        f = fps.cpu().numpy()
        for b in range(B):
            np.add.at(scale[b], bi[b].reshape(-1), s[b].reshape(-1, 3))
            np.add.at(scale[b], f[b], s[b].sum(1))
    if Gn is not None:
        for b in range(B):
            np.add.at(scale[b], fps.cpu().numpy()[b], np.abs(Gn[b].T))
    got = xyz.grad.permute(0, 2, 1)
    _check(f"{kind} xyz.grad", got, want, res[torch.float32][0], scale, gemm_mode)


@pytest.mark.parametrize("S", [1, 128])
def test_fp_block_xyz_grad(dev, gemm_mode, S):
    """Feature propagation in train() mode: xyz1.grad and xyz2.grad through the interpolation weights (S > 1), and an
    exactly zero coordinate gradient for the broadcast of a single coarse point (S = 1)."""
    from pointnet12_b200.model import pointnet_util as pu

    rng = np.random.default_rng(S)
    B, N, D1, D2 = 2, 1024, 32, 64
    mod = _seeded(lambda: pu.PointNetFeaturePropagation(D1 + D2, [64, 64]), 21, dev)
    x1_np, x2_np = _fp_clouds(B, N, S, rng) if S > 1 else (rng.uniform(-1, 1, (B, N, 3)).astype(np.float32),
                                                           np.zeros((B, 1, 3), np.float32))
    p1_np = rng.standard_normal((B, N, D1)).astype(np.float32)
    p2_np = rng.standard_normal((B, S, D2)).astype(np.float32)
    leaves = [T(a.transpose(0, 2, 1), dev).requires_grad_(True) for a in (x1_np, x2_np, p1_np, p2_np)]
    out = mod(*leaves)
    G = rng.standard_normal(out.shape).astype(np.float32)
    (out * T(G, dev)).sum().backward()
    if S == 1:
        assert torch.count_nonzero(leaves[0].grad) == 0 and torch.count_nonzero(leaves[1].grad) == 0
        return
    idx, d32 = _nn_geometry(T(x1_np, dev), T(x2_np, dev))
    res = {}
    for dt in (torch.float64, torch.float32):
        a, b_, p1, p2 = (_leaf(v, dt) for v in (x1_np, x2_np, p1_np, p2_np))
        taps = []
        o = ref_fp(a, b_, p1, p2, torch.from_numpy(idx), d32, mod.mlp_convs, mod.mlp_bns, dt, taps)
        (o.permute(0, 2, 1) * torch.from_numpy(G).to(dt)).sum().backward()
        res[dt] = (a.grad, b_.grad, taps)
    dint_scale = _np(_first_layer_scale(res[torch.float64][2], list(range(D1, D1 + D2))))     # [B,N,D2]
    nb = p2_np[np.arange(B)[:, None, None], idx].astype(np.float64)                          # [B,N,3,D2]
    gabs = (dint_scale[:, :, None, :] * np.abs(nb)).sum(-1)
    w = 1.0 / np.where(d32 < np.float32(CLAMP), np.float32(CLAMP), d32).astype(np.float64)
    w /= w.sum(-1, keepdims=True)
    s1, s2, c2 = _interp_scale(x1_np.astype(np.float64), x2_np.astype(np.float64), idx, d32, w, gabs)
    got1, got2 = leaves[0].grad.permute(0, 2, 1), leaves[1].grad.permute(0, 2, 1)
    if gemm_mode == "fp32":
        within("xyz1.grad", got1, res[torch.float64][0], res[torch.float32][0], s1)
        within("xyz2.grad", got2, res[torch.float64][1], res[torch.float32][1], s2, 4 * c2 * U32 * s2)
    else:
        # no max-pool here, but a ReLU of the MLP whose input lies within the engine's rounding of zero gates a whole
        # channel of a row of dinterp: bound the L2 error and the direction
        for what, got, want in (("xyz1.grad", got1, res[torch.float64][0]), ("xyz2.grad", got2, res[torch.float64][1])):
            assert rl2(got, want) < 2e-2 and cosine(got, want) > 0.999, (what, rl2(got, want), cosine(got, want))


# ------------------------------------------------------------------------------------------------ 3. nets in train() mode
def _dropout(x, keep, p):
    return x * torch.from_numpy(keep.astype(np.float64)).to(x.dtype).view(x.shape) / (1.0 - p)


def cosine(a, b):
    a, b = _np(a).reshape(-1), _np(b).reshape(-1)
    return float(a @ b / max(np.linalg.norm(a) * np.linalg.norm(b), 1e-300))


def _net_close(what, got, want, mode):
    """A whole net, as tests/test_gpu_train.py compares its deep parameter gradients: every max-pool and ReLU of the levels
    can flip between float32 and float64, and through the batch statistics of BatchNorm a flip reaches every row of its
    channel, so the comparison is on the direction (cosine > 0.999 with the exact-fp32 engine, > 0.98 with the tensor-core
    engine) and the size (within 5 % / 10 %) of the whole gradient.  The size is dominated by the few points closest to a
    coarse point, where the 1/d^2 of the interpolation weights amplifies every upstream difference."""
    cos = cosine(got, want)
    ratio = np.linalg.norm(_np(got)) / np.linalg.norm(_np(want))
    fp32 = mode == "fp32"
    assert cos > (0.999 if fp32 else 0.98) and abs(ratio - 1) < (0.05 if fp32 else 0.1), (what, cos, ratio)


def _sa_level(mod, x, f, start, dt, xdev):
    """One set-abstraction level of a net in the restatement, with our forward's decisions (computed on xdev, the level's
    float32 coordinates on the device).  -> (new_xyz, features, new_xdev)."""
    from pointnet12_b200 import ops

    if getattr(mod, "group_all", False):
        nx, o = ref_sa(x, f, None, None, mod.mlp_convs, mod.mlp_bns, dt)
        return nx, o, torch.zeros((x.shape[0], 1, 3), device=xdev.device)
    fps = ops.fps(xdev, mod.npoint, start)
    nxd = ops.index_points(xdev, fps)
    fps_c = torch.from_numpy(fps.cpu().numpy())
    if hasattr(mod, "radius_list"):
        outs = []
        for r, k, convs, bns in zip(mod.radius_list, mod.nsample_list, mod.conv_blocks, mod.bn_blocks):
            ball = torch.from_numpy(ops.ball_query(r, k, xdev, nxd).cpu().numpy())
            nx, o = ref_sa(x, f, fps_c, ball, convs, bns, dt, msg=True)
            outs.append(o)
        return nx, torch.cat(outs, -1), nxd
    ball = torch.from_numpy(ops.ball_query(mod.radius, mod.nsample, xdev, nxd).cpu().numpy())
    nx, o = ref_sa(x, f, fps_c, ball, mod.mlp_convs, mod.mlp_bns, dt)
    return nx, o, nxd


def _fp_level(mod, x1, x2, p1, p2, x1d, x2d, dt):
    idx, d32 = _nn_geometry(x1d, x2d)
    return ref_fp(x1, x2, p1, p2, torch.from_numpy(idx), d32, mod.mlp_convs, mod.mlp_bns, dt)


def _seg_head(net, feat, keep, dt):
    """conv1-bn1-relu-drop1-conv2-log_softmax (pointnet2.py:172-175) on point-major rows."""
    z = ref_mlp(feat, [net.conv1], [net.bn1], dt)
    z = _dropout(z, keep, float(net.drop1.p))
    W2 = net.conv2.weight.detach().cpu().to(dt).reshape(net.conv2.weight.shape[0], -1)
    return torch.log_softmax(z @ W2.T + net.conv2.bias.detach().cpu().to(dt), -1)


def test_semseg_net_points_grad(dev, gemm_mode):
    """PointNet2SemSeg(19, 1) at B = 2, N = 2048: all four channels of points.grad (xyz and reflectance)."""
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import semseg_forward_train

    rng = np.random.default_rng(31)
    net = _seeded(lambda: PointNet2SemSeg(19, 1), 31, dev)
    B, N = 2, 2048
    pts_np = np.concatenate([rng.uniform(-4, 4, (B, 3, N)), rng.uniform(0, 1, (B, 1, N))], 1).astype(np.float32)
    sizes = [N, 1024, 256, 64]
    starts = [rng.integers(0, n, B) for n in sizes]
    keep = (rng.random((B * N, 128)) > 0.5).astype(np.uint8)
    points = T(pts_np, dev).requires_grad_(True)
    logp = semseg_forward_train(net, points, fps_starts=[T(s, dev) for s in starts], dropout_mask=T(keep, dev))
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    res = {}
    for dt in (torch.float64,):
        pl = _leaf(pts_np, dt)
        pm = pl.permute(0, 2, 1)
        xs, fs, xds = [pm[:, :, :3]], [pm[:, :, 3:]], [T(pts_np[:, :3].transpose(0, 2, 1), dev)]
        for i, m in enumerate((net.sa1, net.sa2, net.sa3, net.sa4)):
            nx, nf, nxd = _sa_level(m, xs[-1], fs[-1], T(starts[i], dev), dt, xds[-1])
            xs.append(nx)
            fs.append(nf)
            xds.append(nxd)
        up = fs[4]
        for i, m in ((3, net.fp4), (2, net.fp3), (1, net.fp2), (0, net.fp1)):
            up = _fp_level(m, xs[i], xs[i + 1], fs[i] if i > 0 else None, up, xds[i], xds[i + 1], dt)
        lp = _seg_head(net, up, keep, dt)
        (lp * torch.from_numpy(G).to(dt)).sum().backward()
        res[dt] = pl.grad
    got = points.grad
    assert torch.count_nonzero(got[:, :3]) > 0.99 * B * 3 * N
    for c, what in ((slice(0, 3), "xyz"), (slice(3, 4), "reflectance")):
        _net_close(f"points.grad {what}", got[:, c], res[torch.float64][:, c], gemm_mode)


def test_cls_msg_net_xyz_grad(dev, gemm_mode):
    """PointNet2ClsMsg: MSG levels without input features, a group-all level and the fc head with two dropouts."""
    from pointnet12_b200.model.pointnet2 import PointNet2ClsMsg

    rng = np.random.default_rng(41)
    net = _seeded(PointNet2ClsMsg, 41, dev)
    B, N = 4, 1024
    xyz_np = rng.uniform(-1, 1, (B, 3, N)).astype(np.float32)
    starts = [rng.integers(0, n, B) for n in (N, 512)]
    keeps = [(rng.random((B, c)) > 0.4).astype(np.uint8) for c in (512, 256)]
    xyz = T(xyz_np, dev).requires_grad_(True)
    logp, _ = net(xyz, dropout_masks=[T(k, dev) for k in keeps], fps_starts=[T(s, dev) for s in starts])
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    res = {}
    for dt in (torch.float64,):
        xl = _leaf(xyz_np, dt)
        x, f, xd = xl.permute(0, 2, 1), None, T(xyz_np.transpose(0, 2, 1), dev)
        for i, m in enumerate((net.sa1, net.sa2, net.sa3)):
            x, f, xd = _sa_level(m, x, f, T(starts[i], dev) if i < 2 else None, dt, xd)
        h = f.reshape(B, 1024)
        for fc, bn, drop, keep in ((net.fc1, net.bn1, net.drop1, keeps[0]), (net.fc2, net.bn2, net.drop2, keeps[1])):
            h = _dropout(ref_mlp(h, [fc], [bn], dt), keep, float(drop.p))
        lp = torch.log_softmax(h @ net.fc3.weight.detach().cpu().to(dt).T + net.fc3.bias.detach().cpu().to(dt), -1)
        (lp * torch.from_numpy(G).to(dt)).sum().backward()
        res[dt] = xl.grad
    assert torch.count_nonzero(xyz.grad) > 0.9 * xyz.numel()
    _net_close("xyz.grad", xyz.grad, res[torch.float64], gemm_mode)


def test_partseg_msg_one_hot_net_xyz_grad(dev, gemm_mode):
    """PointNet2PartSegMsg_one_hot: xyz reaches the loss through the geometry of every level AND as a skip feature of fp1;
    xyz.grad must hold both parts (fp3 interpolates from the single group-all point: no coordinate gradient there)."""
    from pointnet12_b200.model.pointnet2 import PointNet2PartSegMsg_one_hot

    rng = np.random.default_rng(51)
    net = _seeded(lambda: PointNet2PartSegMsg_one_hot(50), 51, dev)
    B, N = 2, 1024
    xyz_np = rng.uniform(-1, 1, (B, 3, N)).astype(np.float32)
    nrm_np = rng.standard_normal((B, 3, N)).astype(np.float32)
    nrm_np /= np.linalg.norm(nrm_np, axis=1, keepdims=True)
    label = np.zeros((B, 16), np.float32)
    label[np.arange(B), rng.integers(0, 16, B)] = 1
    starts = [rng.integers(0, n, B) for n in (N, 512)]
    keep = (rng.random((B * N, 128)) > 0.5).astype(np.uint8)
    xyz = T(xyz_np, dev).requires_grad_(True)
    logp = net(xyz, T(nrm_np, dev), T(label, dev), dropout_mask=T(keep, dev), fps_starts=[T(s, dev) for s in starts])
    G = rng.standard_normal(logp.shape).astype(np.float32)
    (logp * T(G, dev)).sum().backward()
    res = {}
    for variant, dt in (("all", torch.float64), ("skip", torch.float64)):
        xl = _leaf(xyz_np, dt)
        x0 = xl.permute(0, 2, 1)
        xg = x0 if variant == "all" else x0.detach()          # "skip": xyz only as the skip feature of fp1
        nrm = torch.from_numpy(nrm_np.transpose(0, 2, 1).astype(np.float64)).to(dt)
        xs, fs, xds = [xg], [nrm], [T(xyz_np.transpose(0, 2, 1), dev)]
        for i, m in enumerate((net.sa1, net.sa2, net.sa3)):
            nx, nf, nxd = _sa_level(m, xs[-1], fs[-1], T(starts[i], dev) if i < 2 else None, dt, xds[-1])
            xs.append(nx)
            fs.append(nf)
            xds.append(nxd)
        f2 = _fp_level(net.fp3, xs[2], xs[3], fs[2], fs[3], xds[2], xds[3], dt)
        f1 = _fp_level(net.fp2, xs[1], xs[2], fs[1], f2, xds[1], xds[2], dt)
        lab = torch.from_numpy(label.astype(np.float64)).to(dt)[:, None, :].expand(B, N, 16)
        skip = torch.cat([lab, x0, nrm], -1)
        f0 = _fp_level(net.fp1, xs[0], xs[1], skip, f1, xds[0], xds[1], dt)
        lp = _seg_head(net, f0, keep, dt)
        (lp * torch.from_numpy(G).to(dt)).sum().backward()
        res[(variant, dt)] = xl.grad
    want = res[("all", torch.float64)]
    _net_close("xyz.grad", xyz.grad, want, gemm_mode)
    # both parts are there: the skip-feature part alone is far from the whole gradient, which ours matches
    assert rl2(res[("skip", torch.float64)], want) > 0.1


# ------------------------------------------------------------------------------------------------ 4. no change without it
def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


@pytest.mark.parametrize("wants_grad", [False, True])
def test_coordinate_kernels_run_only_when_asked(dev, wants_grad):
    """A train step whose points do not require a gradient launches neither coordinate kernel; one whose points do,
    launches both."""
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.train import cross_entropy, semseg_forward_train

    rng = np.random.default_rng(61)
    net = _seeded(lambda: PointNet2SemSeg(19, 1), 61, dev)
    B, N = 2, 2048
    points = T(rng.uniform(-4, 4, (B, 4, N)).astype(np.float32), dev).requires_grad_(wants_grad)
    target = T(rng.integers(0, 19, (B, N)), dev)

    def step():
        loss = cross_entropy(semseg_forward_train(net, points), target)
        loss.backward()

    step()
    names = _kernel_names(step)
    new = {n for n in names if "group_bwd_xyz_kernel" in n or "three_interpolate_bwd_xyz_kernel" in n}
    if wants_grad:
        assert any("group_bwd_xyz_kernel" in n for n in new) and any("three_interpolate_bwd_xyz_kernel" in n for n in new)
    else:
        assert not new, new
        assert any("three_interpolate_bwd_kernel" in n for n in names)
