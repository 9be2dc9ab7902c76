"""Gradients through the function-level API -- square_distance, index_points, sample_and_group(_all) and the chamfer losses --
against float64.

The reference writes these functions as torch expressions (pointnet_util.py:19-157, chamfer.py:7-53), so autograd
differentiates them; here each gets a backward of its own.  The yardstick is a float64 restatement of the reference's
expression in torch on the CPU, differentiated by torch autograd, with the conventions of tests/test_gpu_xyz_grad.py:

  - the discrete decisions come from our forward: FPS and ball-query indices and the chamfer arg-min are injected, so the
    float64 run cannot pick other points;
  - |got - want| <= (4 * E32 + 1e-6) * scale elementwise, where E32 is the largest |ref32 - want| / scale of the same
    restatement run in float32, plus the float32 atomic-accumulation bound 4 m 2^-24 sum|terms| for values that m scattered
    terms add up to.  scale and sum|terms| come from a "magnitude run": the same expression on |upstream gradient| with every
    subtraction turned into an addition, so each gradient entry becomes the sum of the sizes of its terms.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

K_TORCH = 4.0
FLOOR = 1e-6
U32 = 2.0 ** -24
F64 = torch.float64


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64) if isinstance(t, torch.Tensor) else np.asarray(t, np.float64)


def within(what, got, want, ref32, scale, extra=0.0):
    """|got - want| <= (K_TORCH * E32 + FLOOR) * scale + extra elementwise (tests/test_gpu_xyz_grad.py::within)."""
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


def _gather(x, idx):
    """x [B,N,C], idx [B,...] -> [B,...,C] (index_points)."""
    B = x.shape[0]
    bi = torch.arange(B).view((B,) + (1,) * (idx.dim() - 1))
    return x[bi, idx]


def _leaves(arrays, dt):
    return [None if a is None else torch.tensor(np.asarray(a), dtype=dt, requires_grad=True) for a in arrays]


def _grads(fn, arrays, grads_out, dt):
    """Gradients of sum(out_i * G_i) with respect to the arrays, for fn(*leaves) -> outputs, in dtype dt on the CPU."""
    leaves = _leaves(arrays, dt)
    outs = fn(*leaves)
    outs = outs if isinstance(outs, (tuple, list)) else (outs,)
    sum(((o * torch.from_numpy(np.asarray(g)).to(dt)).sum() for o, g in zip(outs, grads_out) if g is not None)).backward()
    return [None if t is None else t.grad for t in leaves]


# ------------------------------------------------------------------------------------------------ square_distance
def ref_sqdist(src, dst):
    """pointnet_util.py:34-39."""
    B, N, _ = src.shape
    M = dst.shape[1]
    dist = -2 * torch.matmul(src, dst.permute(0, 2, 1))
    dist = dist + torch.sum(src ** 2, -1).view(B, N, 1)
    return dist + torch.sum(dst ** 2, -1).view(B, 1, M)


@pytest.mark.parametrize("case", ["plain", "n_gt_m", "strided", "g_row_slice", "g_transposed", "src_only", "dst_only"])
def test_square_distance_backward(dev, case):
    from pointnet12_b200.model import pointnet_util as U

    B, N, M = {"plain": (2, 512, 2048), "n_gt_m": (2, 1500, 301)}.get(case, (2, 700, 1000))
    rng = np.random.default_rng(["plain", "n_gt_m", "strided", "g_row_slice", "g_transposed", "src_only", "dst_only"].index(case))
    a = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    b = rng.uniform(-1, 1, (B, M, 3)).astype(np.float32)
    g = rng.standard_normal((B, N, M)).astype(np.float32)
    if case == "strided":          # channel-major storage seen point-major, as the reference's modules pass xyz
        src_leaf, dst_leaf = T(a.transpose(0, 2, 1), dev).requires_grad_(True), T(b.transpose(0, 2, 1), dev).requires_grad_(True)
        src, dst = src_leaf.permute(0, 2, 1), dst_leaf.permute(0, 2, 1)
        assert src.stride() == (3 * N, 1, N)
    else:
        src_leaf = T(a, dev).requires_grad_(case != "dst_only")
        dst_leaf = T(b, dev).requires_grad_(case != "src_only")
        src, dst = src_leaf, dst_leaf
    if case == "g_row_slice":      # row stride M + 3: unaligned rows, the scalar path
        gd = T(np.concatenate([g, np.zeros((B, N, 3), np.float32)], 2), dev)[:, :, :M]
        assert gd.stride(1) == M + 3
    elif case == "g_transposed":   # columns not contiguous: the wrapper copies
        gd = T(g.transpose(0, 2, 1), dev).transpose(1, 2)
        assert gd.stride(2) != 1
    else:
        gd = T(g, dev)
    out = U.square_distance(src, dst)
    assert out.grad_fn is not None
    with torch.no_grad():
        assert torch.equal(out, U.square_distance(src, dst))           # the forward-only launch, same values
    out.backward(gd)
    want = _grads(ref_sqdist, (a, b), (g,), F64)
    ref32 = _grads(ref_sqdist, (a, b), (g,), torch.float32)
    ag, ab_, absg = np.abs(a).astype(np.float64), np.abs(b).astype(np.float64), np.abs(g).astype(np.float64)
    # scale 2 sum |g| (|src| + |dst|) per coordinate; the sums run over M (rows) / N (columns) terms
    s_src = 2 * (absg.sum(2)[..., None] * ag + absg @ ab_)
    s_dst = 2 * (absg.sum(1)[..., None] * ab_ + absg.transpose(0, 2, 1) @ ag)
    if case != "dst_only":
        within("dsrc", src_leaf.grad.permute(0, 2, 1) if case == "strided" else src_leaf.grad, want[0], ref32[0], s_src,
               4 * M * U32 * s_src)
    else:
        assert src_leaf.grad is None
    if case != "src_only":
        within("ddst", dst_leaf.grad.permute(0, 2, 1) if case == "strided" else dst_leaf.grad, want[1], ref32[1], s_dst,
               4 * N * U32 * s_dst)
    else:
        assert dst_leaf.grad is None


# ------------------------------------------------------------------------------------------------ index_points
@pytest.mark.parametrize("C", [1, 3, 67])
@pytest.mark.parametrize("rank", [2, 3])
def test_index_points_backward(dev, rank, C):
    from pointnet12_b200.model import pointnet_util as U

    rng = np.random.default_rng(10 * rank + C)
    B, N, S, K = 2, 300, 64, 8
    pts = rng.standard_normal((B, N, C)).astype(np.float32)
    shape = (B, S) if rank == 2 else (B, S, K)
    idx = rng.integers(0, N // 4, shape)                     # a quarter of the points: many repeats
    idx.reshape(B, -1)[:, :5] = 7                            # and one point hit five times in a row
    g = rng.standard_normal(shape + (C,)).astype(np.float32)
    leaf = T(pts, dev).requires_grad_(True)
    out = U.index_points(leaf, T(idx, dev))
    assert out.grad_fn is not None and out.shape == shape + (C,)
    out.backward(T(g, dev))
    ti = torch.from_numpy(idx)
    want = _grads(lambda p: _gather(p, ti), (pts,), (g,), F64)[0]
    ref32 = _grads(lambda p: _gather(p, ti), (pts,), (g,), torch.float32)[0]
    asum = _grads(lambda p: _gather(p, ti), (pts,), (np.abs(g),), F64)[0].numpy()
    cnt = _grads(lambda p: _gather(p, ti), (pts,), (np.ones_like(g),), F64)[0].numpy()
    assert cnt.max() >= 5
    within("dpoints", leaf.grad, want, ref32, asum, 4 * cnt * U32 * asum)


# ------------------------------------------------------------------------------------------------ sample_and_group
def ref_sample_and_group(xyz, pts, fps_idx, idx, sign=-1.0):
    """pointnet_util.py:122-137 with the indices injected -> (new_xyz, new_points, grouped_xyz); sign=+1: magnitude run."""
    new_xyz = _gather(xyz, fps_idx)
    grouped_xyz = _gather(xyz, idx)
    norm = grouped_xyz + sign * new_xyz[:, :, None, :]
    new_points = norm if pts is None else torch.cat([norm, _gather(pts, idx)], -1)
    return new_xyz, new_points, grouped_xyz


def _cloud(B, N, D, seed):
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    pts = rng.standard_normal((B, N, D)).astype(np.float32) if D else None
    return rng, xyz, pts


def _geometry(xyz_d, npoint, radius, nsample, start):
    from pointnet12_b200.model import pointnet_util as U

    with torch.no_grad():
        fps_idx = U.farthest_point_sample(xyz_d, npoint, start)
        idx = U.query_ball_point(radius, nsample, xyz_d, U.index_points(xyz_d, fps_idx))
    return fps_idx, idx


@pytest.mark.parametrize("D", [0, 13])
@pytest.mark.parametrize("returnfps", [False, True])
def test_sample_and_group_backward(dev, D, returnfps):
    from pointnet12_b200.model import pointnet_util as U

    B, N, S, K, radius = 2, 1024, 128, 32, 0.3
    rng, xyz, pts = _cloud(B, N, D, 100 + D + returnfps)
    start = torch.tensor([5, N - 1])
    xyz_leaf = T(xyz, dev).requires_grad_(True)
    pts_leaf = T(pts, dev).requires_grad_(True) if D else None
    out = U.sample_and_group(S, radius, K, xyz_leaf, pts_leaf, returnfps=returnfps, start_idx=start)
    fps_idx, idx = _geometry(T(xyz, dev), S, radius, K, start)
    assert all(o.grad_fn is not None for o in out[:3 if returnfps else 2])
    with torch.no_grad():                                   # the same values as the forward-only path
        plain = U.sample_and_group(S, radius, K, xyz_leaf, pts_leaf, returnfps=returnfps, start_idx=start)
    for o, p in zip(out, plain):
        assert torch.equal(o, p)
    if returnfps:
        assert torch.equal(out[3], fps_idx)
    gn = rng.standard_normal((B, S, 3)).astype(np.float32)
    gp = rng.standard_normal((B, S, K, 3 + D)).astype(np.float32)
    gg = rng.standard_normal((B, S, K, 3)).astype(np.float32) if returnfps else None
    torch.autograd.backward(list(out[:3 if returnfps else 2]), [T(x, dev) for x in (gn, gp, gg) if x is not None])
    fi, gi = torch.from_numpy(fps_idx.cpu().numpy()), torch.from_numpy(idx.cpu().numpy())
    arrays = (xyz, pts) if D else (xyz,)
    gouts = (gn, gp, gg)

    def fn(sign):
        return lambda x, p=None: ref_sample_and_group(x, p, fi, gi, sign)

    want = _grads(fn(-1.0), arrays, gouts, F64)
    ref32 = _grads(fn(-1.0), arrays, gouts, torch.float32)
    asum = _grads(fn(1.0), arrays, tuple(None if x is None else np.abs(x) for x in gouts), F64)
    cnt = _grads(fn(1.0), arrays, tuple(None if x is None else np.ones_like(x) for x in gouts), F64)
    within("dxyz", xyz_leaf.grad, want[0], ref32[0], asum[0].numpy(), 4 * cnt[0].numpy() * U32 * asum[0].numpy())
    if D:
        within("dpoints", pts_leaf.grad, want[1], ref32[1], asum[1].numpy(), 4 * cnt[1].numpy() * U32 * asum[1].numpy())


@pytest.mark.parametrize("D", [0, 5])
def test_sample_and_group_all_backward(dev, D):
    from pointnet12_b200.model import pointnet_util as U

    B, N = 2, 777
    rng, xyz, pts = _cloud(B, N, D, 200 + D)
    xyz_leaf = T(xyz, dev).requires_grad_(True)
    pts_leaf = T(pts, dev).requires_grad_(True) if D else None
    new_xyz, new_points = U.sample_and_group_all(xyz_leaf, pts_leaf)
    assert new_xyz.grad_fn is None and new_points.grad_fn is not None and new_points.shape == (B, 1, N, 3 + D)
    with torch.no_grad():
        assert torch.equal(new_points, U.sample_and_group_all(xyz_leaf, pts_leaf)[1])
    gp = rng.standard_normal((B, 1, N, 3 + D)).astype(np.float32)
    new_points.backward(T(gp, dev))
    # pointnet_util.py:151-156: new_points = cat([xyz.view(B, 1, N, 3), points.view(B, 1, N, D)], -1) -- each input element
    # receives exactly one upstream value
    assert torch.equal(xyz_leaf.grad.cpu(), torch.from_numpy(gp[:, 0, :, :3]))
    if D:
        assert torch.equal(pts_leaf.grad.cpu(), torch.from_numpy(gp[:, 0, :, 3:]))


# ------------------------------------------------------------------------------------------------ chamfer
def ref_chamfer(p1, p2, argmin, divisor, sign=-1.0):
    """chamfer.py:32-53 (norm -> min -> sum -> / B) with the arg-min injected."""
    return torch.norm(p1 + sign * _gather(p2, argmin), 2, dim=2).sum() / divisor


def _check_chamfer(dev, a, b, p1, p2, leaf1, leaf2, loss, batch, unwrap=lambda t: t):
    from pointnet12_b200 import ops

    B = a.shape[0]
    divisor = B if batch else 1
    _, am = ops.chamfer_argmin(p1.detach(), p2.detach())
    ai = torch.from_numpy(am.cpu().numpy().astype(np.int64))
    # the arg-min is the first minimum of the float32 squared distances (fma order of the kernel restated in float64:
    # products of float32 are exact there, only ties and near-ties matter, and the first index of equal minima is kept)
    d2 = ((a[:, :, None, :].astype(np.float64) - b[:, None, :, :]) ** 2).sum(-1)
    assert (np.take_along_axis(d2, ai.numpy()[..., None], 2)[..., 0] <= d2.min(2) * (1 + 1e-6) + 1e-12).all()
    loss.backward()
    want = _grads(lambda x, y: ref_chamfer(x, y, ai, divisor), (a, b), (np.float32(1.0),), F64)
    ref32 = _grads(lambda x, y: ref_chamfer(x, y, ai, divisor), (a, b), (np.float32(1.0),), torch.float32)
    # |d ||r|| / dr| = 1: every p1 entry is at most 1/divisor, a p2 entry the sum over the p1 points that chose it
    cnt = np.zeros(b.shape[:2] + (1,))
    for bb in range(B):
        np.add.at(cnt[bb], ai[bb].numpy(), 1.0)
    s1 = np.full(a.shape, 1.0 / divisor)
    s2 = np.broadcast_to(cnt / divisor, b.shape)
    g1, g2 = unwrap(leaf1.grad), unwrap(leaf2.grad)
    assert torch.isfinite(g1).all() and torch.isfinite(g2).all()
    within("dp1", g1, want[0], ref32[0], s1)
    within("dp2", g2, want[1], ref32[1], s2, 4 * cnt * U32 * s2)
    return am, g1, g2


def test_chamfer_known_answer_with_backward(dev):
    """model/chamfer.py:55-67 (11.6073 both ways), now with .backward()."""
    from model.chamfer import chamfer_batch, chamfer_non_batch

    a = np.array([[[1., 2, 3], [4, 5, 6], [3, 5, 6], [5, 6, 7]], [[2., 2, 3], [3, 5, 6], [4, 5, 6], [8, 6, 7]]], np.float32)
    b = np.array([[[3., 7, 8], [1, 4, 5]], [[3., 8, 8], [2, 4, 5]]], np.float32)
    l1, l2 = T(a, dev).requires_grad_(True), T(b, dev).requires_grad_(True)
    loss = chamfer_batch(l1, l2)
    assert loss.grad_fn is not None and abs(loss.item() - 11.6073) < 1e-4
    _check_chamfer(dev, a, b, l1, l2, l1, l2, loss, batch=True)
    total = 0.0
    for i in range(2):
        m1, m2 = T(a[i:i + 1], dev).requires_grad_(True), T(b[i:i + 1], dev).requires_grad_(True)
        part = chamfer_non_batch(m1, m2)
        assert part.grad_fn is not None
        total += part.item() / 2
        _check_chamfer(dev, a[i:i + 1], b[i:i + 1], m1, m2, m1, m2, part, batch=False)
    assert abs(total - 11.6073) < 1e-4


@pytest.mark.parametrize("D", [2, 3, 8])
@pytest.mark.parametrize("batch", [True, False])
def test_chamfer_backward(dev, D, batch):
    from pointnet12_b200.model.chamfer import chamfer_batch, chamfer_non_batch

    rng = np.random.default_rng(300 + D + 10 * batch)
    B, N, M = (3, 1000, 700) if batch else (1, 1000, 700)
    a = rng.standard_normal((B, N, D)).astype(np.float32)
    b = rng.standard_normal((B, M, D)).astype(np.float32)
    a[:, 0] = b[:, 5]                            # a p1 point ON a p2 point: d = 0, zero gradient, no NaN
    b[:, 9] = b[:, 8]                            # duplicated p2 points: the first index wins the tie ...
    a[:, 1] = b[:, 8] + np.float32(2.0 ** -10)   # ... for a p1 point that is nearest to them
    fn = chamfer_batch if batch else chamfer_non_batch
    l1, l2 = T(a, dev).requires_grad_(True), T(b, dev).requires_grad_(True)
    loss = fn(l1, l2)
    with torch.no_grad():
        assert torch.equal(loss, fn(l1, l2))
    am, g1, g2 = _check_chamfer(dev, a, b, l1, l2, l1, l2, loss, batch)
    assert (am[:, 0] == 5).all() and (am[:, 1] == 8).all()
    assert (g1[:, 0] == 0).all()
    assert (g2[:, 9] == 0).all() and (g2[:, 8] != 0).any()     # nothing reaches the second copy


def test_chamfer_backward_strided(dev):
    """Channel-major clouds seen point-major (permuted views)."""
    from pointnet12_b200.model.chamfer import chamfer_batch

    rng = np.random.default_rng(400)
    B, N, M, D = 2, 900, 1100, 3
    a = rng.standard_normal((B, N, D)).astype(np.float32)
    b = rng.standard_normal((B, M, D)).astype(np.float32)
    l1, l2 = T(a.transpose(0, 2, 1), dev).requires_grad_(True), T(b.transpose(0, 2, 1), dev).requires_grad_(True)
    p1, p2 = l1.permute(0, 2, 1), l2.permute(0, 2, 1)
    loss = chamfer_batch(p1, p2)
    _check_chamfer(dev, a, b, p1, p2, l1, l2, loss, batch=True, unwrap=lambda t: t.permute(0, 2, 1))


# ------------------------------------------------------------------------------------------------ forward-only paths
def test_no_grad_paths_are_the_forward_only_launches(dev):
    """Under torch.no_grad(), or with inputs that do not require a gradient, every function returns no grad_fn and the
    values of the direct kernel calls the functions made before they were differentiable."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model import pointnet_util as U
    from pointnet12_b200.model.chamfer import _chamfer_sum, chamfer_batch, chamfer_non_batch

    rng, xyz, pts = _cloud(2, 1024, 6, 500)
    start = torch.tensor([3, 9])
    x0, p0 = T(xyz, dev), T(pts, dev)
    idx = T(rng.integers(0, 1024, (2, 50, 4)), dev)
    for mode in ("no_grad", "plain"):
        x, p = (x0.clone().requires_grad_(True), p0.clone().requires_grad_(True)) if mode == "no_grad" else (x0, p0)
        with torch.no_grad() if mode == "no_grad" else torch.enable_grad():
            outs = {
                "square_distance": (U.square_distance(x, x[:, :300]), ops.square_distance(x0, x0[:, :300])),
                "index_points": (U.index_points(p, idx), ops.index_points(p0, idx)),
                "chamfer_batch": (chamfer_batch(x, x[:, ::3]), (_chamfer_sum(x0, x0[:, ::3]) / 2).to(torch.float32)),
                "chamfer_non_batch": (chamfer_non_batch(x[:1], x[1:]), _chamfer_sum(x0[:1], x0[1:]).to(torch.float32)),
            }
            fps_idx = ops.fps(x0, 128, start.to(dev))
            new_xyz = ops.index_points(x0, fps_idx)
            gidx = ops.ball_query(0.3, 32, x0, new_xyz)
            sg = U.sample_and_group(128, 0.3, 32, x, p, returnfps=True, start_idx=start)
            for name, o, w in zip(("new_xyz", "new_points", "grouped_xyz", "fps_idx"), sg,
                                  (new_xyz, ops.group(x0, p0, new_xyz, gidx, msg_order=False), ops.index_points(x0, gidx), fps_idx)):
                outs["sample_and_group." + name] = (o, w)
            everyone = torch.arange(1024, device=dev).expand(2, 1, 1024).contiguous()
            outs["sample_and_group_all"] = (U.sample_and_group_all(x, p)[1],
                                            ops.group(x0, p0, torch.zeros((2, 1, 3), device=dev), everyone, msg_order=False))
        for name, (o, w) in outs.items():
            assert o.grad_fn is None and not o.requires_grad, (mode, name)
            assert torch.equal(o, w), (mode, name)


def test_double_backward_is_refused(dev):
    from pointnet12_b200.model import pointnet_util as U

    x = T(np.random.default_rng(1).uniform(-1, 1, (1, 64, 3)).astype(np.float32), dev).requires_grad_(True)
    (gx,) = torch.autograd.grad(U.square_distance(x, x).sum(), x, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable|does not require grad"):
        gx.sum().backward()


# ------------------------------------------------------------------------------------------------ a user-built layer
def test_user_layer_sample_group_conv_max_chamfer(dev):
    """A layer a user builds from the exported functions: sample_and_group -> one 1x1 conv + max written in torch ->
    chamfer_batch against a target cloud -> .backward().  xyz.grad and points.grad match the float64 restatement (indices
    injected) in direction (cosine >= 0.999) and size."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model import pointnet_util as U
    from pointnet12_b200.model.chamfer import chamfer_batch

    B, N, D, S, K, radius = 2, 2048, 4, 256, 32, 0.25
    rng, xyz, pts = _cloud(B, N, D, 600)
    target = rng.uniform(-1, 1, (B, 500, 3)).astype(np.float32)
    W = (rng.standard_normal((3, 3 + D)) * 0.5).astype(np.float32)
    bias = rng.standard_normal(3).astype(np.float32)
    start = torch.tensor([0, 17])

    def layer(new_points, w, b_):
        return (torch.einsum("bskc,oc->bsko", new_points, w) + b_).max(2)[0]         # [B, S, 3]

    xl, pl = T(xyz, dev).requires_grad_(True), T(pts, dev).requires_grad_(True)
    _, new_points = U.sample_and_group(S, radius, K, xl, pl, start_idx=start)
    feat = layer(new_points, T(W, dev), T(bias, dev))
    chamfer_batch(feat, T(target, dev)).backward()
    fps_idx, idx = _geometry(T(xyz, dev), S, radius, K, start)
    _, am = ops.chamfer_argmin(feat.detach(), T(target, dev))
    fi, gi, ai = (torch.from_numpy(t.cpu().numpy().astype(np.int64)) for t in (fps_idx, idx, am))

    def ref(x, p):
        _, npts, _ = ref_sample_and_group(x, p, fi, gi)
        f = layer(npts, torch.from_numpy(W).to(x.dtype), torch.from_numpy(bias).to(x.dtype))
        return ref_chamfer(f, torch.from_numpy(target).to(x.dtype), ai, B)

    want = _grads(ref, (xyz, pts), (np.float32(1.0),), F64)
    for what, got, w in (("xyz", xl.grad, want[0]), ("points", pl.grad, want[1])):
        g, w = _np(got).ravel(), _np(w).ravel()
        cos = float(g @ w / (np.linalg.norm(g) * np.linalg.norm(w)))
        ratio = float(np.linalg.norm(g) / np.linalg.norm(w))
        assert cos >= 0.999 and abs(ratio - 1) < 1e-2, (what, cos, ratio)
