"""Training kernels against float64 at their numerical edges, element by element.

tests/test_gpu_train.py checks every kernel of csrc/train.cu once on well-conditioned data.  This file goes where such
kernels go wrong: BatchNorm statistics of channels whose mean is large against their spread (or that are exactly constant),
row counts at the kernels' tails, the labels nn.CrossEntropyLoss ignores, the index patterns a ball query really produces
for the scatter-add backward, and hundreds of device-side Adam steps with a learning-rate decay, eager and graph-replayed.

Every check is elementwise and compares with a float64 restatement.  The bounds, stated once:

    |got - want| <= (K_TORCH * E32 + FLOOR) * scale

    scale   the magnitude of the terms the value is formed from (for z = y*scale + shift: |y*gamma*invstd| + |mean*gamma*
            invstd| + |beta|), so that float32 round-off is a fixed fraction of it wherever cancellation happens;
    E32     the largest |ref32 - want| / scale over the tensor, ref32 being the same value in float32 arithmetic:
            torch's CPU BatchNorm (native_batch_norm / native_batch_norm_backward) fed the exact statistics, torch's
            CrossEntropyLoss in float32.  For the statistics themselves ref32 is the float64 value rounded once to float32:
            torch's training-mode statistics on the CPU accumulate the mean in float32 and are no yardstick (a constant
            channel at 27.1 over 70 001 rows: save_invstd 18 % below 1/sqrt(eps)), while the kernels sum in float64;
    K_TORCH = 4, FLOOR = 1e-6 (about 16 float32 ulps of the terms).
"""
import numpy as np
import pytest
import torch

from oracle import train_oracle as tor

pytestmark = pytest.mark.gpu

K_TORCH = 4.0
FLOOR = 1e-6
EPS, MOMENTUM = 1e-5, 0.1
U32 = 2.0 ** -24


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


def within(what, got, want, ref32, scale):
    """|got - want| <= (K_TORCH * E32 + FLOOR) * scale elementwise (see the module docstring)."""
    got, want, ref32 = _np(got), _np(want), _np(ref32)
    scale = np.broadcast_to(np.asarray(scale, np.float64), want.shape)
    e32 = float(np.max(np.abs(ref32 - want) / np.maximum(scale, 1e-300), initial=0.0))
    bound = (K_TORCH * e32 + FLOOR) * scale
    err = np.abs(got - want)
    bad = ~(err <= bound)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(bound, 1e-300), 0)), want.shape)
        pytest.fail(f"{what}: {int(bad.sum())} of {want.size} elements out of bound; worst at {i}: got {got[i]!r}, "
                    f"want {want[i]!r}, bound {bound[i]:.3g} (E32 {e32:.3g}, scale {scale[i]:.3g})")


# ------------------------------------------------------------------------------------------------ 1. BatchNorm
# Channels of one case (C = 37, not a multiple of 32): the offset ones with |mean|/std ~ 1, 30, 300, 3000; an all-zero
# channel; constant channels (std = 0) at 3.7, -12.9, 27.1; then ordinary channels.
RATIOS = (1.0, 30.0, 300.0, 3000.0)
CONSTS = (3.7, -12.9, 27.1)
C_BN, CIN, LDX = 37, 67, 68
ROWS = (2, 7, 9, 33, 127, 129, 70001)       # < one 16-lane stats block, not a multiple of 8, one past a 128-row tile
POOL_K = {2: 2, 7: 7, 9: 3, 33: 33, 127: 127, 129: 43, 70001: 70001}     # (70001 is prime) K >= 256: the tall max-pool kernel


def _layer(route, rows, rng):
    """x [rows, CIN], W [C_BN, CIN], bias: the offset of a channel comes from the bias ("bias") or from an input with a
    large mean ("input": x = 5 + 0.01 * noise, one input column exactly 5)."""
    w = np.zeros((C_BN, CIN))
    b = np.zeros(C_BN)
    g = rng.standard_normal((C_BN, CIN))
    if route == "bias":
        x = rng.standard_normal((rows, CIN))
        g /= np.linalg.norm(g, axis=1, keepdims=True)
        for c, r in enumerate(RATIOS):           # std 1, mean r
            w[c], b[c] = g[c], r
        for c, v in enumerate(CONSTS):           # W row 0: y = bias exactly
            b[5 + c] = v
    else:
        x = 5.0 + 0.01 * rng.standard_normal((rows, CIN))
        x[:, 0] = 5.0
        gn = g[:, 1:] - g[:, 1:].mean(1, keepdims=True)
        gn /= np.linalg.norm(gn, axis=1, keepdims=True)
        for c, r in enumerate(RATIOS):           # mean 5, std 0.01 * sqrt(1/66 + s^2)
            s = np.sqrt(max((500.0 / r) ** 2 - 1.0 / (CIN - 1), 0.0))
            w[c, 1:] = 1.0 / (CIN - 1) + s * gn[c]
        for c, v in enumerate(CONSTS):           # every row computes the same products: a constant channel
            w[5 + c, 0] = v / 5.0
    w[8:] = g[8:] / np.sqrt(CIN)
    b[8:] = rng.standard_normal(C_BN - 8)
    return x.astype(np.float32), w.astype(np.float32), b.astype(np.float32)


def _bn_module(rng, dev):
    bn = torch.nn.BatchNorm1d(C_BN).to(dev)
    with torch.no_grad():
        bn.weight.copy_(T((rng.uniform(0.5, 1.5, C_BN) * rng.choice([-1, 1], C_BN)).astype(np.float32), dev))
        bn.bias.copy_(T(rng.standard_normal(C_BN).astype(np.float32), dev))
        bn.running_mean.copy_(T(rng.standard_normal(C_BN).astype(np.float32), dev))
        bn.running_var.copy_(T(rng.uniform(0.5, 2.0, C_BN).astype(np.float32), dev))
    return bn


def _check_stats(y64, st, bn, rm0, rv0):
    n = y64.shape[0]
    mu, var = y64.mean(0), y64.var(0)
    sd, inv = np.sqrt(var), 1.0 / np.sqrt(var + EPS)
    f32 = lambda a: a.astype(np.float32)                          # noqa: E731 -- the correctly rounded float32 answer
    within("mean", st.mean, mu, f32(mu), np.abs(mu) + sd)
    within("invstd", st.invstd, inv, f32(inv), inv)
    rm = (1 - MOMENTUM) * rm0 + MOMENTUM * mu
    within("running_mean", bn.running_mean, rm, f32(rm), (1 - MOMENTUM) * np.abs(rm0) + MOMENTUM * (np.abs(mu) + sd))
    unb = var * n / (n - 1)
    rv = (1 - MOMENTUM) * rv0 + MOMENTUM * unb
    within("running_var", bn.running_var, rv, f32(rv), (1 - MOMENTUM) * rv0 + MOMENTUM * unb)
    assert int(bn.num_batches_tracked) == 1
    return mu, var, inv


def _check_backward(tag, y32, mu, inv, gam, gz, dy, dg, db):
    """dy / dgamma / dbeta of the BatchNorm backward for the gradient gz that reached its output (ReLU mask applied)."""
    y64 = y32.astype(np.float64)
    xhat = (y64 - mu) * inv
    m1, m2 = gz.mean(0), (gz * xhat).mean(0)
    xterm = (np.abs(y64) + np.abs(mu)) * inv                     # xhat = (y - mean) * invstd: the terms y and mean
    r32 = torch.ops.aten.native_batch_norm_backward(
        torch.from_numpy(gz.astype(np.float32)), torch.from_numpy(y32), torch.from_numpy(gam.astype(np.float32)), None, None,
        torch.from_numpy(mu.astype(np.float32)), torch.from_numpy(inv.astype(np.float32)), True, EPS, [True, True, True])
    within(f"{tag} dy", dy, gam * inv * (gz - m1 - xhat * m2), r32[0],
           np.abs(gam * inv) * (np.abs(gz) + np.abs(m1) + xterm * np.abs(m2)))
    within(f"{tag} dgamma", dg, (gz * xhat).sum(0), r32[1], (np.abs(gz) * xterm).sum(0))
    within(f"{tag} dbeta", db, gz.sum(0), r32[2], np.abs(gz).sum(0))


@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("route", ["bias", "input"])
@pytest.mark.parametrize("path", ["bn_batch_stats", "train_gemm_epilogue"])
def test_bn_statistics_and_normalisation(dev, path, route, rows):
    """Every path that forms BatchNorm batch statistics, then normalise (+ max-pool) and the backward on top of them."""
    from pointnet12_b200 import ops

    rng = np.random.default_rng(1000 * rows + (route == "input"))
    x, w, b = _layer(route, rows, rng)
    bn = _bn_module(rng, dev)
    rm0, rv0 = _np(bn.running_mean), _np(bn.running_var)
    xb = torch.zeros((rows, LDX), device=dev)
    xb[:, :CIN] = T(x, dev)                                       # ld > cin
    if path == "train_gemm_epilogue":
        acc = torch.zeros((2, C_BN), dtype=torch.float64, device=dev)
        yv = ops.train_gemm(xb[:, :CIN], T(w, dev), T(b, dev), stats_acc=acc)
        st = ops.bn_finalize(acc, rows, bn)
    else:
        wide = torch.zeros((rows, C_BN + 3), device=dev)         # ld > C
        wide[:, :C_BN] = ops.train_gemm(xb[:, :CIN], T(w, dev), T(b, dev))
        yv = wide[:, :C_BN]
        st = ops.bn_batch_stats(yv, bn)
    y32 = yv.cpu().numpy()
    y64 = y32.astype(np.float64)
    assert np.all(y64[:, 4] == 0) and all(np.all(y64[:, 5 + c] == y64[0, 5 + c]) for c in range(3))   # the constant channels
    mu, var, inv = _check_stats(y64, st, bn, rm0, rv0)
    gam, bet = _np(bn.weight), _np(bn.bias)

    # normalise + ReLU; torch's float32 transform given the exact statistics is the yardstick
    z = ops.bn_act(yv, st, relu=True)
    z_want = np.maximum((y64 - mu) * inv * gam + bet, 0)
    z32 = torch.relu(torch.ops.aten.native_batch_norm(torch.from_numpy(y32), torch.from_numpy(gam.astype(np.float32)),
                                                      torch.from_numpy(bet.astype(np.float32)), torch.from_numpy(mu.astype(np.float32)),
                                                      torch.from_numpy(var.astype(np.float32)), False, MOMENTUM, EPS)[0])
    # (invstd of the eval-mode call is 1/sqrt(float32(var) + eps): within 2^-24 of the exact one)
    z_scale = np.abs(gam) * inv * (np.abs(y64) + np.abs(mu)) + np.abs(bet)
    within("bn_act", z, z_want, z32, z_scale)
    zk = z.cpu().numpy()

    # max over runs of K rows: within the largest bound of the run
    K = POOL_K[rows]
    G = rows // K
    pooled, am = ops.bn_act_max(yv, st, K, relu=True)
    within("bn_act_max", pooled, z_want.reshape(G, K, -1).max(1), _np(z32).reshape(G, K, -1).max(1),
           z_scale.reshape(G, K, -1).max(1))
    amk = am.cpu().numpy().astype(np.int64)
    assert np.array_equal(amk, zk.reshape(G, K, -1).argmax(1))       # the first maximum of what bn_act computes

    # backward, MODE 1 (a gradient per row) and MODE 2 (the pooled gradient routed through the arg-max)
    mask = zk > 0                                                   # the kernels' own ReLU decisions (fused multiply-add)
    dz = rng.standard_normal((rows, C_BN)).astype(np.float32)
    dy, dg, db = ops.bn_act_backward(yv, st, T(dz, dev), relu=True)
    _check_backward("mode 1", y32, mu, inv, gam, dz * mask, dy, dg, db)
    dpool = rng.standard_normal((G, C_BN)).astype(np.float32)
    dy, dg, db = ops.bn_act_backward(yv, st, T(dpool, dev), relu=True, argmax=am, K=K)
    routed = np.zeros((G, K, C_BN))
    np.put_along_axis(routed, amk[:, None, :], dpool[:, None, :].astype(np.float64), axis=1)
    _check_backward("mode 2", y32, mu, inv, gam, routed.reshape(rows, C_BN) * mask, dy, dg, db)

    # the same reductions in the epilogue of the input-gradient GEMM (dz = dyo W, sums of the layer below's backward)
    co = 48
    dyo = rng.standard_normal((rows, co)).astype(np.float32)
    wo = (rng.standard_normal((co, C_BN)) / np.sqrt(co)).astype(np.float32)
    acc = torch.zeros((2, C_BN), dtype=torch.float64, device=dev)
    dzk = ops.train_gemm_bnbwd(T(dyo, dev), T(wo, dev), yv, st, acc)
    dy, dg, db = ops.bn_act_backward(yv, st, dzk, relu=True, acc=acc, acc_ready=True)
    _check_backward("train_gemm_bnbwd", y32, mu, inv, gam, _np(dzk) * mask, dy, dg, db)


def _oracle_sd(layers):
    sd = {}
    for i, (conv, bn, _) in enumerate(layers):
        for k, v in conv.state_dict().items():
            sd[f"c{i}.{k}"] = _np(v)
        for k, v in bn.state_dict().items():
            sd[f"b{i}.{k}"] = _np(v)
    return sd


def test_block_with_a_constant_channel(dev, gemm_mode):
    """train.mlp_forward / mlp_backward on 13 -> 37 -> 64 -> 19 with channel 5 of layer 1 constant (W row 0, bias 27.1),
    against the float64 oracle: the statistics of that channel decide its BatchNorm gradient, and with it row 5 of dW1.
    Bound per output channel (row of a weight): a row is a sum over the rows of products whose operands carry a relative
    rounding u (2^-24 in fp32, 2^-17 for the split-bf16 operands of the tensor-core engine); through the three layers
    |got - want| <= 64 * u * sqrt(rows) * max|want row|."""
    from pointnet12_b200.train import mlp_backward, mlp_forward

    rows, dims = 999, (13, 37, 64, 19)
    torch.manual_seed(7)
    layers = [(torch.nn.Conv1d(a, b_, 1).to(dev), torch.nn.BatchNorm1d(b_).to(dev), True) for a, b_ in zip(dims[:-1], dims[1:])]
    with torch.no_grad():
        layers[0][0].weight[5].zero_()
        layers[0][0].bias[5] = 27.1
        for _, bn, _ in layers:
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(0.2, 0.6)
    sd = _oracle_sd(layers)
    rng = np.random.default_rng(8)
    x = rng.standard_normal((rows, dims[0])).astype(np.float32)
    dz = rng.standard_normal((rows, dims[-1])).astype(np.float32)
    out, saved = mlp_forward(T(x, dev), layers)
    _, grads = mlp_backward(saved, layers, T(dz, dev), None, need_dx=False)

    h, caches, bufs = x.astype(np.float64), [], {}
    for i in range(3):
        h, c = tor.conv_bn_relu_fwd(sd, f"c{i}", f"b{i}", h, bufs)
        caches.append(c)
    want = {}
    g = dz.astype(np.float64)
    for i in (2, 1, 0):
        g = tor.conv_bn_relu_bwd(sd, f"c{i}", f"b{i}", caches[i], g, want)
    u = 2.0 ** -24 if gemm_mode == "fp32" else 2.0 ** -17
    tol = 64 * u * np.sqrt(rows)

    def rows_within(what, got, ref):
        """per row of a matrix (an output channel), against that row's largest entry; a vector counts as one row"""
        ref = np.asarray(ref, np.float64)
        got, ref = _np(got).reshape(ref.shape[0] if ref.ndim > 1 else 1, -1), ref.reshape(ref.shape[0] if ref.ndim > 1 else 1, -1)
        err = np.abs(got - ref).max(1)
        lim = tol * np.abs(ref).max(1) + 1e-30
        assert np.all(err <= lim), (what, np.flatnonzero(err > lim), (err / lim).max())

    rows_within("output", out.T, h.T)
    for i, (conv, bn, _) in enumerate(layers):
        dw, _, dgam, dbet = grads[i]
        rows_within(f"dW{i}", dw, want[f"c{i}.weight"])
        rows_within(f"dgamma{i}", dgam, want[f"b{i}.weight"])
        rows_within(f"dbeta{i}", dbet, want[f"b{i}.bias"])
        rows_within(f"running_mean{i}", bn.running_mean, bufs[f"b{i}.running_mean"])
        rows_within(f"running_var{i}", bn.running_var, bufs[f"b{i}.running_var"])


# ------------------------------------------------------------------------------------------------ 2. cross-entropy
def _ce_inputs(C, rows, ignored, rng):
    logits = rng.standard_normal((rows, C)) * 3
    x = logits - np.log(np.exp(logits).sum(-1, keepdims=True))
    x[rng.random((rows, C)) < 0.05] = -80.0                      # extreme entries
    x[rng.random((rows, C)) < 0.02] = -1e4
    tie = rng.random(rows) < 0.1                                 # near-ties: the two largest one float32 ulp apart
    top = x.argmax(1)
    other = (top + 1) % C
    x[tie, other[tie]] = np.nextafter(x[tie, top[tie]].astype(np.float32), np.float32(-np.inf))
    t = rng.integers(0, C, rows)
    t[rng.permutation(rows)[:int(round(ignored * rows))]] = -100
    return x.astype(np.float32), t


@pytest.mark.parametrize("C,rows", [(2, 1001), (19, 4099), (50, 777)])
@pytest.mark.parametrize("ignored", [0.0, 0.3, 1.0])
@pytest.mark.parametrize("grad_scale", [1.0, 0.25])
def test_cross_entropy_ignored_labels(dev, C, rows, ignored, grad_scale):
    """ops.cross_entropy / train.cross_entropy == nn.CrossEntropyLoss() (ignore_index -100) in float64: the loss and
    (grad_scale x) its gradient.  Every label ignored: torch's 0/0 = NaN loss and a zero gradient."""
    from pointnet12_b200 import ops
    from pointnet12_b200.train import cross_entropy

    rng = np.random.default_rng(C * 100 + int(ignored * 10))
    x, t = _ce_inputs(C, rows, ignored, rng)
    ref = {}
    for dt in (torch.float64, torch.float32):
        xt = torch.from_numpy(x).to(dt).requires_grad_(True)
        loss = torch.nn.CrossEntropyLoss()(xt, torch.from_numpy(t))
        (loss * grad_scale).backward()
        ref[dt] = (loss.item(), xt.grad.numpy())
    want_loss, want_dx = ref[torch.float64]
    loss, dx = ops.cross_entropy(T(x, dev), T(t, dev), grad_scale=grad_scale)
    xr = torch.from_numpy(x).reshape(1, rows, C).to(dev).requires_grad_(True)
    loss2 = cross_entropy(xr, T(t.reshape(1, rows), dev))
    (loss2 * grad_scale).backward()
    keep = t != -100
    n = int(keep.sum())
    if n == 0:
        assert np.isnan(want_loss) and np.isnan(loss.item()) and np.isnan(loss2.item())
        assert not dx.any() and not xr.grad.any() and not want_dx.any()
        return
    # loss = mean over kept rows of lse(x) - x[t]: terms |lse| + |x[t]| (lse computed as max + log(sum exp(x - max)))
    x64 = x.astype(np.float64)
    lse_terms = np.abs(x64.max(1)) + np.log(np.exp(x64 - x64.max(1, keepdims=True)).sum(1))
    l_scale = (lse_terms + np.abs(x64[np.arange(rows), np.where(keep, t, 0)]))[keep].mean()
    within("loss", loss.item(), want_loss, ref[torch.float32][0], l_scale)
    within("train.cross_entropy loss", loss2.item(), want_loss, ref[torch.float32][0], l_scale)
    # dx = (softmax - onehot) * grad_scale / n on kept rows, 0 on ignored ones
    p = np.exp(x64 - x64.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    onehot = np.zeros_like(p)
    onehot[np.arange(rows)[keep], t[keep]] = 1
    d_scale = (p + onehot) * grad_scale / n * keep[:, None] + 1e-30
    within("dx", dx, want_dx, ref[torch.float32][1], d_scale)
    within("train.cross_entropy dx", xr.grad.reshape(rows, C), want_dx, ref[torch.float32][1], d_scale)
    assert not dx[T(~keep, dev)].any()                             # ignored rows: exactly zero


# ------------------------------------------------------------------------------------------------ 3. scatter-add backward
def _scatter_bound(got, want, count, abs_sum):
    """float32 atomics: each of the m terms on an element adds at most one rounding of the running sum (<= sum |terms|),
    so |got - want| <= 4 m 2^-24 sum|terms| + 1e-30 (and exact where nothing lands)."""
    got = _np(got)
    lim = 4 * count * U32 * abs_sum + 1e-30
    bad = ~(np.abs(got - want) <= lim)
    assert not bad.any(), (int(bad.sum()), np.argwhere(bad)[:5].tolist())


def _ball_rows(B, S, K, N, rng):
    """Ball-query rows as the net produces them: u unique hits, padded with the first (u = 1, 2, 5, K per quarter of the
    balls); 60 % of all balls have the same hot point first; index N-1 is hit."""
    idx = np.empty((B, S, K), np.int64)
    hot = rng.integers(0, N)
    for b in range(B):
        for s in range(S):
            u = (1, 2, 5, K)[s % 4]
            hits = rng.choice(N, u, replace=False)
            if rng.random() < 0.6:
                hits[0] = hot
            idx[b, s, :u] = hits
            idx[b, s, u:] = hits[0]
        idx[b, 1, 1] = N - 1
    return idx


@pytest.mark.parametrize("D", [1, 13, 64, 259])
@pytest.mark.parametrize("xyz_first", [True, False])
def test_group_backward_at_ball_query_patterns(dev, D, xyz_first):
    from pointnet12_b200 import ops

    rng = np.random.default_rng(D * 2 + xyz_first)
    B, S, K, N = 2, 64, 32, 700
    idx = _ball_rows(B, S, K, N, rng)
    width = D + 3
    col0 = 3 if xyz_first else 0                                  # [xyz, feat] or MSG order [feat, xyz]
    dg = torch.zeros((B * S * K, width + 5), device=dev)          # ldg > width
    vals = rng.standard_normal((B * S * K, width)).astype(np.float32)
    dg[:, :width] = T(vals, dev)
    got = ops.group_backward(dg[:, :width], col0, D, T(idx, dev), N)
    terms = vals[:, col0:col0 + D].astype(np.float64).reshape(B, S * K, D)
    want, cnt, asum = np.zeros((B, N, D)), np.zeros((B, N, 1)), np.zeros((B, N, D))
    for b in range(B):
        np.add.at(want[b], idx[b].reshape(-1), terms[b])
        np.add.at(cnt[b], idx[b].reshape(-1), 1.0)
        np.add.at(asum[b], idx[b].reshape(-1), np.abs(terms[b]))
    _scatter_bound(got, want, cnt, asum)
    assert cnt[:, N - 1].min() > 0


@pytest.mark.parametrize("S", [1, 2, 40])
@pytest.mark.parametrize("D1", [0, 7])
def test_three_interpolate_backward_at_real_patterns(dev, S, D1):
    """S = 1: the single coarse point (idx (0,0,0), weight (1,0,0)); S = 2: neighbours repeat; S = 40: random, with rows
    whose three neighbours are one index, and index S-1 always hit."""
    from pointnet12_b200 import ops

    rng = np.random.default_rng(S * 10 + D1)
    B, N, D2 = 2, 1000, 24
    if S == 1:
        idx = np.zeros((B, N, 3), np.int64)
        w = np.tile(np.float32([1, 0, 0]), (B, N, 1))
    else:
        idx = rng.integers(0, S, (B, N, 3))
        idx[:, ::7] = idx[:, ::7, :1]                             # one index three times
        idx[:, 3, 2] = S - 1
        w = rng.dirichlet(np.ones(3), (B, N)).astype(np.float32)
    width = D1 + D2
    dx = torch.zeros((B * N, width + 3), device=dev)              # ldx > width
    vals = rng.standard_normal((B * N, width)).astype(np.float32)
    dx[:, :width] = T(vals, dev)
    dp1, dp2 = ops.three_interpolate_backward(dx[:, :width], D1, D2, T(idx, dev), T(w, dev), S)
    if D1:
        assert np.array_equal(dp1.cpu().numpy(), vals[:, :D1].reshape(B, N, D1))
    else:
        assert dp1 is None
    g = vals[:, D1:].astype(np.float64).reshape(B, N, D2)
    want, cnt, asum = np.zeros((B, S, D2)), np.zeros((B, S, 1)), np.zeros((B, S, D2))
    for b in range(B):
        for k in range(3):
            term = g[b] * w[b, :, k:k + 1].astype(np.float64)
            np.add.at(want[b], idx[b, :, k], term)
            np.add.at(cnt[b], idx[b, :, k], 1.0)
            np.add.at(asum[b], idx[b, :, k], np.abs(term))
    # (the kernel rounds each product g*w to float32 before adding it: one more 2^-24 |term|, inside the factor 4)
    _scatter_bound(dp2, want, cnt, asum)
    assert cnt[:, S - 1].min() > 0


# ------------------------------------------------------------------------------------------------ 4. device-side Adam
SIZES = (1, 7, 64, 1000, 100003)


@pytest.mark.parametrize("graphed", [False, True])
@pytest.mark.parametrize("grad_scale", [1.0, 0.25])
def test_flat_adam_300_steps_vs_torch(dev, graphed, grad_scale):
    """FlatAdam (pn_adam_dev_f32: learning rate and step count in device memory) for 300 steps beside torch.optim.Adam
    (weight_decay 1e-4) on the CPU, the learning rate halved at steps 100 and 200; graphed: the update captured once in a
    CUDA graph and replayed.  After every step: max |ours - float64 Adam| <= 2 * max |torch float32 - float64 Adam| + 1e-7."""
    from pointnet12_b200 import ops
    from pointnet12_b200.train import FlatAdam

    rng = np.random.default_rng(300 + graphed)
    init = [(rng.standard_normal(n) * 0.5).astype(np.float32) for n in SIZES]
    mod = torch.nn.ParameterList([torch.nn.Parameter(T(p, dev)) for p in init])
    opt = FlatAdam(mod.parameters(), lr=1e-3, weight_decay=1e-4)
    ref = [torch.nn.Parameter(torch.from_numpy(p.copy())) for p in init]
    topt = torch.optim.Adam(ref, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)
    p64 = np.concatenate(init).astype(np.float64)
    m64, v64 = np.zeros_like(p64), np.zeros_like(p64)
    offs = np.cumsum((0,) + SIZES)
    g_ = opt.param_groups[0]
    if graphed:
        # (any first launch of the library's kernels outside the capture: its one-time device queries)
        scratch = torch.zeros(4, device=dev)
        ops.adam_step_dev(scratch, scratch, scratch, scratch, torch.ones(1, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ops.adam_step_dev(opt.flat, opt.grad, opt.exp_avg, opt.exp_avg_sq, opt.lr_dev, opt.step_dev, g_["betas"], g_["eps"],
                              g_["weight_decay"], grad_scale)
    lr = 1e-3
    for step in range(1, 301):
        if step in (101, 201):
            lr /= 2
            g_["lr"] = lr                                        # what FlatAdam.step forwards to the device
            topt.param_groups[0]["lr"] = lr
            if graphed:
                opt.lr_dev.fill_(lr)
        g = (rng.standard_normal(p64.size) * 10.0 ** rng.uniform(-6, 0, p64.size)).astype(np.float32)
        opt.grad.copy_(T(g / grad_scale, dev))                   # grad_scale 0.25: 4x the gradient, scaled back in the kernel
        if graphed:
            graph.replay()
        else:
            opt.step(grad_scale=grad_scale)
        for i, p in enumerate(ref):
            p.grad = torch.from_numpy(g[offs[i]:offs[i + 1]].copy())
        topt.step()
        p64, m64, v64 = tor.adam_step(p64, g, m64, v64, step, lr=lr)
        ours = opt.flat.cpu().numpy().astype(np.float64)
        t32 = np.concatenate([p.detach().numpy() for p in ref]).astype(np.float64)
        e_t, e_o = np.abs(t32 - p64).max(), np.abs(ours - p64).max()
        assert e_o <= 2 * e_t + 1e-7, (step, e_o, e_t)
    assert opt.steps == 300
