"""Training step and evaluation metrics on the native kernels (SURVEY.md section 8, rows f-1 and f-2).

Reference: pcdseg.py:157-186 -- `model.train()`, `logits = model(points)`, `nn.CrossEntropyLoss()(logits.transpose(2, 1),
target)`, `loss.backward()`, `optimizer.step()` with torch.optim.Adam(lr, betas (0.9, 0.999), eps 1e-8, weight_decay 1e-4)
under nn.DataParallel -- and pcdseg.py:58-97 (test_kitti_semseg).

The drop-in contract is the reference's own: in train() mode the modules of model/pointnet_util.py, and every net of
model/pointnet2.py and model/pointnet.py (both models pcdseg.py can train among them) return tensors that carry a grad_fn, so the reference's loop (torch loss, loss.backward(), any torch optimizer) runs
unchanged; every kernel underneath -- forward with batch-statistics BatchNorm, dropout, and the whole backward -- is ours
(csrc/train.cu + linear.cu + the sampling / grouping kernels of the inference path).  One torch.autograd.Function per
block (set abstraction, feature propagation, segmentation head): autograd only connects them.  The same blocks serve eval()
mode when an input requires a gradient (model/pointnet_util.autograd_path): every BatchNorm / Dropout module follows its own
mode as in torch -- running statistics, left untouched, for a BatchNorm in .eval() (also frozen layers of a train() net), no
dropout for a Dropout in .eval().

On top of that, the pieces a B200-native training loop uses instead of the torch ones:
    cross_entropy(logp, target)    the reference's loss as one kernel (forward + gradient)
    FlatAdam(params, ...)          parameters and gradients re-pointed into ONE flat buffer each: the data-parallel gradient
                                   exchange is a single all-reduce of 3.9 MB and Adam is a single kernel launch
    SegMetrics(num_classes)        argmax + per-class I/U + accuracy accumulated on the device (no .item() per class)

The forward and input-gradient GEMMs run on the tensor cores (single-layer tcgen05 chains, 3-pass split bf16 = fp32 parity,
weights re-packed every iteration); the weight-gradient GEMM (reduction over the rows) is a CUDA-core kernel with fp32
atomics; `ops.set_mlp_mode("fp32")` puts every GEMM on the CUDA cores.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import torch
from torch.autograd.function import once_differentiable

from . import ops


# ------------------------------------------------------------------------------------------------
# shared MLP with batch-statistics BatchNorm: forward keeps (input, pre-norm output, statistics) per layer
def _w2d(conv) -> torch.Tensor:
    return conv.weight.detach().reshape(conv.weight.shape[0], -1)


class PackedWeights:
    """The conv weights of a network in the fused GEMM's shared-memory layout (bf16 hi + lo), both orientations (W for the
    forward, W^T for the input gradient), converted by ONE launch per training iteration (pn_train_pack_many) instead of one
    small launch in front of every GEMM.  lookup() returns the image of a weight, or None when it is not in the arena or the
    parameter's storage has moved since (the GEMM then converts the weight itself)."""

    def __init__(self, convs):
        import numpy as np

        from . import _native as nv

        items, self.slots, total = [], {}, 0
        for conv in convs:
            co, ci = int(conv.weight.shape[0]), int(conv.weight[0].numel())
            for tr in (False, True):
                cin, cout = (co, ci) if tr else (ci, co)
                if not ops.train_gemm_supported(cin, cout):
                    continue
                nbytes = int(nv.lib().pn_train_gemm_scratch_bytes(cin, cout))
                items.append((conv.weight, total, nbytes, cin, cout, tr))
                total += (nbytes + 127) // 128 * 128
        self.n = len(items)
        if not self.n:
            return
        dev = items[0][0].device
        self.arena = torch.empty((total,), dtype=torch.uint8, device=dev)
        table = np.zeros(self.n, dtype=[("w", "<u8"), ("out", "<u8"), ("cin", "<i4"), ("cout", "<i4"), ("tr", "<i4"), ("res", "<i4")])
        for i, (w, off, nbytes, cin, cout, tr) in enumerate(items):
            table[i] = (w.data_ptr(), self.arena.data_ptr() + off, cin, cout, int(tr), 0)
            self.slots[(w.data_ptr(), tr)] = self.arena[off:off + nbytes]
        self.table = torch.from_numpy(table.view(np.uint8).copy()).to(dev)
        self.max_cin, self.max_cout = max(i[3] for i in items), max(i[4] for i in items)
        self._ptrs = [(w, w.data_ptr()) for w, *_ in items]

    def valid(self) -> bool:
        return self.n > 0 and all(w.data_ptr() == p for w, p in self._ptrs)

    def pack(self) -> None:
        from . import _native as nv

        with ops._on_device(self.arena):
            nv.call("pn_train_pack_many", self.table.data_ptr(), self.n, self.max_cin, self.max_cout, ops._stream())

    def lookup(self, w: torch.Tensor, transposed: bool):
        return self.slots.get((w.data_ptr(), bool(transposed)))


def _net_convs(net):
    convs = []
    for m in (net.sa1, net.sa2, net.sa3, net.sa4, net.fp4, net.fp3, net.fp2, net.fp1):
        convs += list(m.mlp_convs)
    return convs + [net.conv1, net.conv2]


def _gemm(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], transposed: bool = False, arena=None) -> torch.Tensor:
    """x [rows, cin] @ W^T + bias with W = w [cout, cin] (or, transposed=True, W = w^T for w [cin, cout]: the input-
    gradient GEMM dx = dy W of a conv with weight w).  Tensor cores (single-layer tcgen05 chain, 3-pass split bf16 = fp32
    parity; the weight is re-packed on every call because it changes every iteration) unless the MLP mode is 'fp32'."""
    cout, cin = (w.shape[1], w.shape[0]) if transposed else (w.shape[0], w.shape[1])
    if ops.mlp_mode() == "bf16x3" and FUSED_BN and ops.train_gemm_supported(cin, cout):
        return ops.train_gemm(x, w, bias, transposed=transposed, packed=arena.lookup(w, transposed) if arena is not None else None)
    if ops.mlp_mode() == "bf16x3" and ops.PackedChain.supported([(cin, cout)]):
        return ops.mlp_rows_tc(ops.PackedChain([(w, bias, False)], transposed=transposed), x)
    if ops.mlp_mode() == "bf16x3" and cout > 1024 and ops.PackedChain.supported([(cin, 1024)]):
        # wider than one chain takes (PointNetSeg's 1088-channel input gradient): column slabs of <= 1024 outputs
        out = torch.empty((x.shape[0], cout), dtype=torch.float32, device=x.device)
        for c0 in range(0, cout, 1024):
            c1 = min(cout, c0 + 1024)
            wk = (w[:, c0:c1] if transposed else w[c0:c1]).contiguous()
            bk = bias[c0:c1].contiguous() if bias is not None else None
            ops.mlp_rows_tc(ops.PackedChain([(wk, bk, False)], transposed=transposed), x, out=out[:, c0:c1])
        return out
    return ops.linear(x, ops.transpose(w) if transposed else w, bias, relu=False)


def _grad_sink(p: torch.Tensor, shape) -> Tuple[torch.Tensor, bool]:
    """Where the gradient of parameter p is accumulated: straight into p.grad when an optimizer with a flat gradient
    buffer owns it (FlatAdam marks its parameters; the kernels add atomically, so no per-parameter add launch is needed
    and the Function returns None for it), else into a fresh zero tensor that autograd accumulates."""
    if getattr(p, "_pn_direct_grad", False) and p.grad is not None:
        return p.grad.view(shape), True
    return torch.zeros(shape, dtype=torch.float32, device=p.device), False


def _dropout_on(drop, mask: Optional[torch.Tensor] = None) -> bool:
    """nn.Dropout's rule: applied in training mode only, when p > 0 or a keep-mask is given.  When it is not applied, no
    dropout seed is drawn and a given mask is ignored."""
    return drop.training and (float(drop.p) > 0.0 or mask is not None)


FUSED_BN = os.environ.get("PN12_TRAIN_FUSED", "1") != "0"     # BatchNorm fused into the training GEMMs (pn_train_gemm_bf16x3)
PACK_ONCE = os.environ.get("PN12_TRAIN_PACK_ONCE", "1") != "0"      # all weight images converted by one launch per iteration
FUSED_BN_BWD = os.environ.get("PN12_TRAIN_FUSED_BWD", "0") != "0"   # BatchNorm-backward reductions in the input-gradient GEMM's epilogue


# The eval-mode BatchNorm backward goes into the input-gradient GEMM's epilogue when the layer below has fewer channels than
# this.  Measured on C2's layers (NVIDIA B200, profiles/r03_eval_grad_bench.json): the fused epilogue wins at 32 and 64
# channels (sa1, sa2: 7-10 % per layer) and loses at 128 on the 192 000 rows of fp1 (188 vs 170 us: the epilogue, already
# the GEMM's bottleneck at that width, then also reads the layer below's y), so 128-wide layers keep GEMM + one pass.
BNEVAL_EPILOGUE_BELOW = 128


def mlp_forward(x: torch.Tensor, layers: Sequence[Tuple], pool_K: Optional[int] = None, arena=None):
    """x [rows, cin] -> (output, saved).  layers = [(conv, bn or None, relu)]; pool_K: the last layer's activation is
    max-pooled over runs of K rows (set abstraction).

    Fused path (tensor-core mode, layers that fit pn_train_gemm_bf16x3): a layer is ONE kernel -- the GEMM applies the
    previous layer's normalise + ReLU while loading its operand and accumulates this layer's batch statistics in its
    epilogue -- plus the tiny finalize; only the pre-normalisation outputs y exist in memory.  `pending` is the BatchStats
    still to be applied to the current x.  saved[l] = (x, pending-at-input, y, stats, relu, argmax).
    A BatchNorm in eval mode (ops.uses_running_stats) normalises with its running statistics, which it leaves untouched:
    the GEMM accumulates no column sums for it and nothing is finalized."""
    saved = []
    pending = None
    rows = x.shape[0]
    widest = max(c.weight.shape[0] for c, _, _ in layers)
    accs = None
    for li, (conv, bn, relu) in enumerate(layers):
        w = _w2d(conv)
        bias = conv.bias.detach() if conv.bias is not None else None
        fused = (FUSED_BN and bn is not None and ops.mlp_mode() == "bf16x3"
                 and ops.train_gemm_supported(w.shape[1], w.shape[0]))
        running = bn is not None and ops.uses_running_stats(bn)
        st, am = None, None
        if bn is not None and not relu and li != len(layers) - 1:
            # (a BatchNorm without ReLU is supported as the LAST layer of a chain only: PointNetEncoder's bn3 ahead of the max)
            raise NotImplementedError("training path: an inner BatchNorm layer must be followed by ReLU")
        if fused:
            if running:
                y = ops.train_gemm(x, w, bias, in_stats=pending,
                                   packed=arena.lookup(conv.weight, False) if arena is not None else None)
                st = ops.running_stats(bn)
            else:
                if accs is None:          # one fill for the block's statistics
                    accs = torch.zeros((len(layers), 2, widest), dtype=torch.float64, device=x.device)
                acc = accs[li, :, :w.shape[0]]
                y = ops.train_gemm(x, w, bias, in_stats=pending, stats_acc=acc,
                                   packed=arena.lookup(conv.weight, False) if arena is not None else None)
                st = ops.bn_finalize(acc, rows, bn)
            saved.append((x, pending, y, st, relu, None))
            x, pending = y, st
            continue
        if pending is not None:                      # a layer the fused kernel does not take: materialise its input first
            x, pending = ops.bn_act(x, pending, True), None
        y = _gemm(x, w, bias, arena=arena)
        if bn is not None:
            st = ops.running_stats(bn) if running else ops.bn_batch_stats(y, bn)
            saved.append((x, None, y, st, relu, None))
            x, pending = y, st
        else:
            if relu:
                raise NotImplementedError("training path: a layer without BatchNorm must be a plain linear layer")
            saved.append((x, None, y, None, relu, None))
            x = y
    if pending is not None:                          # the block's output leaves in activated (and pooled) form
        xin, pin, y, st, relu, _ = saved[-1]
        if pool_K:
            x, am = ops.bn_act_max(y, st, pool_K, relu)
            saved[-1] = (xin, pin, y, st, relu, am)
        else:
            x = ops.bn_act(y, st, relu)
    elif pool_K:
        raise NotImplementedError("training path: the pooled layer must have BatchNorm")
    return x, saved


def mlp_backward(saved, layers: Sequence[Tuple], dz: torch.Tensor, pool_K: Optional[int], need_dx: bool, arena=None):
    """-> (dx or None, [per layer: (dW [Co,Ci], db, dgamma, dbeta)]; None where the gradient went straight into p.grad).
    A layer whose input comes from a BatchNorm with running statistics (eval mode) and whose input-gradient GEMM is the
    fused one with fewer than BNEVAL_EPILOGUE_BELOW outputs runs that BatchNorm's backward in the GEMM's epilogue
    (ops.train_gemm_bneval): the layer below then gets its dy directly and has no BatchNorm pass of its own."""
    grads = [None] * len(layers)
    widest = max(c.weight.shape[0] for c, _, _ in layers)
    accs = torch.zeros((len(layers), 2, widest), dtype=torch.float64, device=dz.device)    # one fill for the block's reductions
    stats_done = False           # the reductions of this layer's BatchNorm backward were fused into the GEMM that produced dz
    bn_done = None               # this layer's whole BatchNorm backward was: dz is already dy; (dgamma, dbeta, direct flags)
    for li in range(len(layers) - 1, -1, -1):
        conv, bn, relu = layers[li]
        x, x_stats, y, st, _, am = saved[li]
        dgamma = dbeta = None
        g_direct = beta_direct = False
        if bn_done is not None:
            dy = dz
            dgamma, dbeta, g_direct, beta_direct = bn_done
        elif st is not None:
            dgamma, g_direct = _grad_sink(bn.weight, bn.weight.shape)
            dbeta, beta_direct = _grad_sink(bn.bias, bn.bias.shape)
            K = pool_K if am is not None else 1
            if st.running:           # fixed statistics: no batch coupling, one pass
                dy = ops.bn_eval_backward(y, st, dz, relu, argmax=am, K=K, dgamma=dgamma, dbeta=dbeta, acc=accs[li, :, :y.shape[1]])
            else:
                dy = ops.bn_act_backward(y, st, dz, relu, argmax=am, K=K, dgamma=dgamma, dbeta=dbeta,
                                         acc=accs[li, :, :y.shape[1]], acc_ready=stats_done)
        else:
            dy = dz
        stats_done, bn_done = False, None
        w = _w2d(conv)
        dw, w_direct = _grad_sink(conv.weight, w.shape)
        db, b_direct = _grad_sink(conv.bias, (w.shape[0],)) if conv.bias is not None else (None, False)
        ops.grad_weight(dy, x, dw, db, x_stats=x_stats)      # x_stats: x is the previous layer's y, activated on load
        grads[li] = (None if w_direct else dw, None if b_direct else db, None if g_direct else dgamma, None if beta_direct else dbeta)
        fused_t = (li > 0 and x_stats is not None and FUSED_BN and ops.mlp_mode() == "bf16x3"
                   and ops.train_gemm_supported(w.shape[0], w.shape[1]))
        if fused_t and x_stats.running and w.shape[1] < BNEVAL_EPILOGUE_BELOW:
            # x is the pre-normalisation output of the layer below, whose BatchNorm has fixed statistics: its backward
            # (dy = scale*g, dgamma, dbeta) happens in this GEMM's epilogue
            bn_below = layers[li - 1][1]
            gb, gb_direct = _grad_sink(bn_below.weight, bn_below.weight.shape)
            bb, bb_direct = _grad_sink(bn_below.bias, bn_below.bias.shape)
            dz = ops.train_gemm_bneval(dy, w, x, x_stats, accs[li - 1, :, :w.shape[1]], dgamma=gb, dbeta=bb,
                                       packed=arena.lookup(conv.weight, True) if arena is not None else None)
            bn_done = (gb, bb, gb_direct, bb_direct)
        elif fused_t and not x_stats.running and FUSED_BN_BWD:
            # the layer below kept only its pre-normalisation output (x here): the input-gradient GEMM also accumulates the
            # two reductions of THAT layer's BatchNorm backward in its epilogue, saving a pass over dz and x
            dz = ops.train_gemm_bnbwd(dy, w, x, x_stats, accs[li - 1, :, :w.shape[1]],
                                      packed=arena.lookup(conv.weight, True) if arena is not None else None)
            stats_done = True
        else:
            dz = _gemm(dy, w, None, transposed=True, arena=arena) if (li > 0 or need_dx) else None
    return dz, grads


def _layer_params(layers) -> List[torch.Tensor]:
    out = []
    for conv, bn, _ in layers:
        out.append(conv.weight)
        if conv.bias is not None:
            out.append(conv.bias)
        if bn is not None:
            out += [bn.weight, bn.bias]
    return out


def _layer_grads(layers, grads) -> List[torch.Tensor]:
    out = []
    for (conv, bn, _), (dw, db, dgamma, dbeta) in zip(layers, grads):
        out.append(dw.view_as(conv.weight) if dw is not None else None)
        if conv.bias is not None:
            out.append(db)
        if bn is not None:
            out += [dgamma, dbeta]
    return out


def _rows_of(grad: torch.Tensor, C: int) -> torch.Tensor:
    """An incoming gradient [B, n, C] (any strides) as a contiguous [B*n, C] row matrix."""
    return grad.contiguous().view(-1, C)


# ------------------------------------------------------------------------------------------------
class SetAbstractionFn(torch.autograd.Function):
    """Grouping + shared MLP (batch-stat BN) + max over nsample of PointNetSetAbstraction.forward
    (model/pointnet_util.py:187-199) or of one scale of PointNetSetAbstractionMsg.forward (:239-257; `branch` selects the
    scale, channel order [features, xyz_rel]).  Sampling / ball query carry no gradient and are done by the caller; the
    gather + recentring pass gradients to xyz_pm and new_xyz when they require one (pn_group_bwd_xyz_f32)."""

    @staticmethod
    def _layers(mod, branch):
        if branch is None:
            return [(c, b, True) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
        return [(c, b, True) for c, b in zip(mod.conv_blocks[branch], mod.bn_blocks[branch])]

    @staticmethod
    def forward(ctx, mod, branch, xyz_pm, pts_pm, new_xyz, idx, *params):
        B, S, K = idx.shape
        D = pts_pm.shape[2] if pts_pm is not None else 0
        layers = SetAbstractionFn._layers(mod, branch)
        msg = branch is not None
        grouped = ops.group(xyz_pm, pts_pm, new_xyz, idx, msg_order=msg, pad4=True)            # [B,S,K,ld]
        x0 = grouped.view(B * S * K, -1)[:, :3 + D]
        ctx.arena = getattr(mod, "_pn_arena", None)
        pooled, saved = mlp_forward(x0, layers, pool_K=K, arena=ctx.arena)
        ctx.mod, ctx.branch, ctx.saved, ctx.idx, ctx.geom = mod, branch, saved, idx, (B, xyz_pm.shape[1], S, K, D)
        return pooled.view(B, S, -1)

    @staticmethod
    def backward(ctx, dpooled):
        B, N, S, K, D = ctx.geom
        layers = SetAbstractionFn._layers(ctx.mod, ctx.branch)
        need_dpts = D > 0 and ctx.needs_input_grad[3]
        need_xyz = ctx.needs_input_grad[2] or ctx.needs_input_grad[4]
        dx0, grads = mlp_backward(ctx.saved, layers, _rows_of(dpooled, dpooled.shape[-1]), K, need_dpts or need_xyz,
                                  arena=ctx.arena)
        # the feature channels sit behind the three xyz columns (SSG order) or in front of them (MSG order)
        msg = ctx.branch is not None
        dpts = ops.group_backward(dx0, 0 if msg else 3, D, ctx.idx, N) if need_dpts else None
        dxyz = dnew = None
        if need_xyz:
            dxyz, dnew = ops.group_backward_xyz(dx0, D if msg else 0, ctx.idx, N, recentred=ctx.needs_input_grad[4])
        ctx.saved = None
        return (None, None, dxyz if ctx.needs_input_grad[2] else None, dpts, dnew, None, *_layer_grads(layers, grads))


class FeaturePropagationFn(torch.autograd.Function):
    """Interpolation + skip concat + shared MLP (batch-stat BN) of PointNetFeaturePropagation.forward
    (model/pointnet_util.py:301-312); the 3-NN search (the choice of neighbours) carries no gradient and is done by the
    caller.  xyz1 [B,N,3] / xyz2 [B,S,3] (point-major) receive the gradient through the interpolation weights when they
    require one (pn_three_interpolate_bwd_xyz_f32)."""

    @staticmethod
    def forward(ctx, mod, p1, p2, idx, w, xyz1, xyz2, *params):
        B, N, _ = idx.shape
        layers = [(c, b, True) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
        x0 = ops.three_interpolate(p1, p2, idx, w).view(B * N, -1)
        ctx.arena = getattr(mod, "_pn_arena", None)
        out, saved = mlp_forward(x0, layers, arena=ctx.arena)
        ctx.mod, ctx.saved, ctx.nn = mod, saved, (idx, w)
        ctx.geom = (B, N, p2.shape[1], p1.shape[2] if p1 is not None else 0, p2.shape[2])
        # the coordinate gradient goes through the 3-NN weights and needs the coarse features and both clouds
        ctx.xyz = (p2, xyz1, xyz2) if ctx.needs_input_grad[5] or ctx.needs_input_grad[6] else None
        return out.view(B, N, -1)

    @staticmethod
    def backward(ctx, dout):
        mod = ctx.mod
        B, N, S, D1, D2 = ctx.geom
        layers = [(c, b, True) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
        dx0, grads = mlp_backward(ctx.saved, layers, _rows_of(dout, dout.shape[-1]), None, True, arena=ctx.arena)
        dxyz1 = dxyz2 = None
        if ctx.xyz is not None and S > 1:
            dp1, dp2, dxyz1, dxyz2 = ops.three_interpolate_backward_xyz(dx0, D1, D2, ctx.nn[0], ctx.nn[1], *ctx.xyz)
        else:
            dp1, dp2 = ops.three_interpolate_backward(dx0, D1, D2, ctx.nn[0], ctx.nn[1], S)
            if ctx.xyz is not None:           # S == 1: the coarse point is broadcast (:292-293), no distance is involved
                dxyz1 = torch.zeros((B, N, 3), dtype=torch.float32, device=dx0.device)
                dxyz2 = torch.zeros((B, S, 3), dtype=torch.float32, device=dx0.device)
        ctx.saved = ctx.xyz = None
        return (None, dp1 if ctx.needs_input_grad[1] else None, dp2 if ctx.needs_input_grad[2] else None, None, None,
                dxyz1 if ctx.needs_input_grad[5] else None, dxyz2 if ctx.needs_input_grad[6] else None,
                *_layer_grads(layers, grads))


class SegHeadFn(torch.autograd.Function):
    """conv1 -> bn1 -> relu -> dropout -> conv2 -> log_softmax of pointnet2.py:172-175 in training mode."""

    @staticmethod
    def forward(ctx, net, feat, mask, seed_offset, *params):
        B, N, C = feat.shape
        layers = [(net.conv1, net.bn1, True)]
        ctx.set_materialize_grads(False)          # the second output is usually unused: no 33 MB of zeros for its gradient
        ctx.arena = arena = getattr(net, "_pn_arena", None)
        z1, saved = mlp_forward(feat.contiguous().view(B * N, C), layers, arena=arena)
        p = float(net.drop1.p)
        if _dropout_on(net.drop1, mask):
            zd, mask = ops.dropout(z1, p, seed_offset=seed_offset, mask=mask)
        else:
            zd, mask = z1, None
        logits = _gemm(zd, _w2d(net.conv2), net.conv2.bias.detach(), arena=arena)
        logp = ops.log_softmax(logits)
        ctx.net, ctx.saved, ctx.tail = net, saved, (zd, mask, logp, p)
        # second output: the activated conv1-bn1 features BEFORE dropout, which the part-segmentation nets return as well
        # (pointnet2.py:99-104); it carries a gradient of its own
        return logp.view(B, N, -1), z1.view(B, N, -1)

    @staticmethod
    def backward(ctx, dlogp, dfeat_out=None):
        net = ctx.net
        zd, mask, logp, p = ctx.tail
        k = logp.shape[1]
        if dlogp is None:
            raise NotImplementedError("segmentation head: the log-probabilities must take part in the loss")
        dlogits = ops.log_softmax_backward(_rows_of(dlogp, k), logp)
        w2 = _w2d(net.conv2)
        dw2, w_direct = _grad_sink(net.conv2.weight, w2.shape)
        db2, b_direct = _grad_sink(net.conv2.bias, (k,))
        ops.grad_weight(dlogits, zd, dw2, db2)
        dzd = _gemm(dlogits, w2, None, transposed=True, arena=ctx.arena)
        dz1 = ops.dropout(dzd, p, mask=mask)[0] if mask is not None else dzd
        if dfeat_out is not None:
            dz1 = dz1 + _rows_of(dfeat_out, dz1.shape[1])
        layers = [(net.conv1, net.bn1, True)]
        dfeat, grads = mlp_backward(ctx.saved, layers, dz1, None, True, arena=ctx.arena)
        B, N = dlogp.shape[0], dlogp.shape[1]
        ctx.saved = ctx.tail = None
        return (None, dfeat.view(B, N, -1), None, None, *_layer_grads(layers, grads),
                None if w_direct else dw2.view_as(net.conv2.weight), None if b_direct else db2)


class ClsHeadFn(torch.autograd.Function):
    """fc1-bn1-relu-drop1-fc2-bn2-relu-drop2-fc3-log_softmax of the classification nets (pointnet2.py:41-45, :68-72) in
    training mode, on rows = clouds.  masks: optional uint8 keep-masks of the two dropouts (parity tests)."""

    @staticmethod
    def forward(ctx, net, x, masks, seed_offset, *params):
        stages, cur = [], x.contiguous()
        for i, (fc, bn, drop) in enumerate(((net.fc1, net.bn1, net.drop1), (net.fc2, net.bn2, net.drop2))):
            z, saved = mlp_forward(cur, [(fc, bn, True)])
            p = float(drop.p)
            mask = masks[i] if masks is not None else None
            if _dropout_on(drop, mask):
                so = None if mask is not None else seed_offset + torch.tensor([0, 7919 * (i + 1)], dtype=torch.int64, device=x.device)
                cur, mask = ops.dropout(z, p, seed_offset=so, mask=mask)
            else:
                cur, mask = z, None
            stages.append((saved, mask, p))
        logits = _gemm(cur, _w2d(net.fc3), net.fc3.bias.detach())
        logp = ops.log_softmax(logits)
        ctx.net, ctx.stages, ctx.tail = net, stages, (cur, logp)
        return logp

    @staticmethod
    def backward(ctx, dlogp):
        net = ctx.net
        last_in, logp = ctx.tail
        dlogits = ops.log_softmax_backward(dlogp.contiguous(), logp)
        w3 = _w2d(net.fc3)
        dw3, w_direct = _grad_sink(net.fc3.weight, w3.shape)
        db3, b_direct = _grad_sink(net.fc3.bias, (w3.shape[0],))
        ops.grad_weight(dlogits, last_in, dw3, db3)
        dz = _gemm(dlogits, w3, None, transposed=True)
        out = []
        for (saved, mask, p), (fc, bn) in zip(reversed(ctx.stages), ((net.fc2, net.bn2), (net.fc1, net.bn1))):
            if mask is not None:
                dz = ops.dropout(dz, p, mask=mask)[0]
            dz, grads = mlp_backward(saved, [(fc, bn, True)], dz, None, True)
            out = _layer_grads([(fc, bn, True)], grads) + out
        ctx.stages = ctx.tail = None
        return (None, dz, None, None, *out, None if w_direct else dw3, None if b_direct else db3)


def cls_head_train(net, global_feat: torch.Tensor, dropout_masks=None, seed_offset=None) -> torch.Tensor:
    """global_feat [B, 1024] -> log-probabilities [B, classes] with grad_fn."""
    if dropout_masks is None and seed_offset is None and (_dropout_on(net.drop1) or _dropout_on(net.drop2)):
        seed_offset = dropout_seed(global_feat.device)
    params = [net.fc1.weight, net.fc1.bias, net.bn1.weight, net.bn1.bias, net.fc2.weight, net.fc2.bias, net.bn2.weight,
              net.bn2.bias, net.fc3.weight, net.fc3.bias]
    return ClsHeadFn.apply(net, global_feat, dropout_masks, seed_offset, *params)


class MlpRowsFn(torch.autograd.Function):
    """A conv1x1 / Linear + BatchNorm(batch statistics) + ReLU chain over rows [rows, cin], optionally max-pooled over runs of
    K rows (the per-point stacks, global max and fully connected layers of model/pointnet.py in train() mode)."""

    @staticmethod
    def forward(ctx, layers, pool_K, x, *params):
        out, saved = mlp_forward(x, layers, pool_K=pool_K)
        ctx.layers, ctx.pool_K, ctx.saved = layers, pool_K, saved
        return out

    @staticmethod
    def backward(ctx, dout):
        dx, grads = mlp_backward(ctx.saved, ctx.layers, dout.contiguous(), ctx.pool_K, ctx.needs_input_grad[2])
        ctx.saved = None
        return (None, None, dx, *_layer_grads(ctx.layers, grads))


def mlp_rows_train(layers, x: torch.Tensor, pool_K: Optional[int] = None) -> torch.Tensor:
    return MlpRowsFn.apply(layers, pool_K, x.contiguous(), *_layer_params(layers))


class BmmPointsFn(torch.autograd.Function):
    """torch.bmm(x [B,N,k], trans [B,k,k2]) of pointnet.py:105-107, :113-115 with both gradients."""

    @staticmethod
    def forward(ctx, x, trans):
        ctx.save_for_backward(x, trans)
        return ops.bmm_points(x, trans)

    @staticmethod
    def backward(ctx, dy):
        x, trans = ctx.saved_tensors
        dy = dy.contiguous()
        dx = ops.bmm_points(dy, trans.transpose(1, 2)) if ctx.needs_input_grad[0] else None
        dtrans = None
        if ctx.needs_input_grad[1]:
            B, N, k = x.shape
            dtrans = torch.zeros_like(trans)
            for b in range(B):                    # dtrans[b] = x[b]^T dy[b]: the weight-gradient kernel with the roles swapped
                ops.grad_weight(x[b].contiguous(), dy[b], dtrans[b], None)
        return dx, dtrans


class LogSoftmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        y = ops.log_softmax(x.contiguous())
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        return ops.log_softmax_backward(dy.contiguous(), ctx.saved_tensors[0])


class BatchNormActFn(torch.autograd.Function):
    """A BatchNorm + optional ReLU on rows that does not directly follow its linear layer (PointNetCls:
    relu(bn2(dropout(fc2(x)))), pointnet.py:148); batch or running statistics as the module's mode says."""

    @staticmethod
    def forward(ctx, bn, relu, x, gamma, beta):
        x = x.contiguous()
        st = ops.running_stats(bn) if ops.uses_running_stats(bn) else ops.bn_batch_stats(x, bn)
        ctx.bn, ctx.relu, ctx.st = bn, relu, st
        ctx.save_for_backward(x)
        return ops.bn_act(x, st, relu)

    @staticmethod
    def backward(ctx, dz):
        (x,) = ctx.saved_tensors
        bwd = ops.bn_eval_backward if ctx.st.running else ops.bn_act_backward
        dy, dgamma, dbeta = bwd(x, ctx.st, dz.contiguous(), ctx.relu)
        return None, None, dy, dgamma, dbeta


class DropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p, seed_offset, mask):
        y, mask = ops.dropout(x.contiguous(), p, seed_offset=seed_offset, mask=mask)
        ctx.p, ctx.mask = p, mask
        return y

    @staticmethod
    def backward(ctx, dy):
        return ops.dropout(dy.contiguous(), ctx.p, mask=ctx.mask)[0], None, None, None


def pointnet_cls_train(net, x: torch.Tensor, dropout_mask=None):
    """PointNetCls.forward (pointnet.py:146-151) in train() mode: x [B,3,N] -> (log_probs [B,k], trans_feat)."""
    ops._need_cuda(x, "x")
    g, _, _, trans_feat = pointnet_encoder_train(net.feat, x.permute(0, 2, 1))
    h = mlp_rows_train([(net.fc1, net.bn1, True), (net.fc2, None, False)], g)
    p = float(net.dropout.p)
    if _dropout_on(net.dropout, dropout_mask):
        h = DropoutFn.apply(h, p, None if dropout_mask is not None else dropout_seed(x.device), dropout_mask)
    h = BatchNormActFn.apply(net.bn2, True, h, net.bn2.weight, net.bn2.bias)
    logits = mlp_rows_train([(net.fc3, None, False)], h)
    return LogSoftmaxFn.apply(logits), trans_feat


def pointnet_densecls_train(net, point_cloud: torch.Tensor, label: torch.Tensor, dropout_mask=None):
    """PointNetDenseCls.forward (pointnet.py:186-228) in train() mode: (point_cloud [B,3,N], label [B,16]) ->
    (cls logits [B,cat_num], seg log_probs [B,N,part_num], trans_feat).  The per-point stacks, transforms and heads run on the
    autograd blocks above; the global max of out5 (which is also a per-point input of the segmentation head) and the concats are
    torch glue."""
    ops._need_cuda(point_cloud, "point_cloud")
    B, _, N = point_cloud.shape
    x_pm = point_cloud.permute(0, 2, 1).contiguous()
    trans = stn_train(net.stn, x_pm)
    pct = BmmPointsFn.apply(x_pm, trans)
    out1 = mlp_rows_train([(net.conv1, net.bn1, True)], pct.reshape(B * N, 3))
    out2 = mlp_rows_train([(net.conv2, net.bn2, True)], out1)
    out3 = mlp_rows_train([(net.conv3, net.bn3, True)], out2)
    trans_feat = stn_train(net.fstn, out3.view(B, N, 128))
    nt = BmmPointsFn.apply(out3.view(B, N, 128), trans_feat)
    out4 = mlp_rows_train([(net.conv4, net.bn4, True)], nt.reshape(B * N, 128))
    out5 = mlp_rows_train([(net.conv5, net.bn5, False)], out4)                              # BatchNorm without ReLU, :209
    out_max = out5.view(B, N, 2048).max(dim=1)[0]                                           # [B, 2048]
    # classification head: fc1-bnc1-relu, fc2-dropout-bnc2-relu, fc3 (raw logits, :213-215)
    h = mlp_rows_train([(net.fc1, net.bnc1, True), (net.fc2, None, False)], out_max)
    p = float(net.dropout.p)
    if _dropout_on(net.dropout, dropout_mask):
        h = DropoutFn.apply(h, p, None if dropout_mask is not None else dropout_seed(h.device), dropout_mask)
    h = BatchNormActFn.apply(net.bnc2, True, h, net.bnc2.weight, net.bnc2.bias)
    cls_logits = mlp_rows_train([(net.fc3, None, False)], h)
    # segmentation head on cat([expand(out_max | label), out1 .. out5]) = 4944 channels per point (:218-227)
    expand = torch.cat([out_max, label.float()], 1)[:, None, :].expand(B, N, 2048 + label.shape[1])
    concat = torch.cat([expand, out1.view(B, N, -1), out2.view(B, N, -1), out3.view(B, N, -1), out4.view(B, N, -1),
                        out5.view(B, N, -1)], dim=2).reshape(B * N, -1)
    seg = mlp_rows_train([(net.convs1, net.bns1, True), (net.convs2, net.bns2, True), (net.convs3, net.bns3, True),
                          (net.convs4, None, False)], concat)
    return cls_logits, LogSoftmaxFn.apply(seg).view(B, N, -1), trans_feat


def stn_train(stn, x_pm: torch.Tensor) -> torch.Tensor:
    """STN3d / STNkd.forward (pointnet.py:27-45, :66-84) in train() mode: x_pm [B,N,k] -> [B,k,k]."""
    B, N, k = x_pm.shape
    g = mlp_rows_train([(stn.conv1, stn.bn1, True), (stn.conv2, stn.bn2, True), (stn.conv3, stn.bn3, True)],
                       x_pm.reshape(B * N, k), pool_K=N)                                  # [B, 1024]
    h = mlp_rows_train([(stn.fc1, stn.bn4, True), (stn.fc2, stn.bn5, True), (stn.fc3, None, False)], g)
    return (h + torch.eye(stn.k, device=h.device, dtype=h.dtype).flatten()).view(B, stn.k, stn.k)


def pointnet_encoder_train(enc, x_pm: torch.Tensor):
    """PointNetEncoder.forward (pointnet.py:100-131) in train() mode on point-major rows:
    -> (global [B,1024], pointfeat [B,N,64], trans, trans_feat)."""
    B, N, _ = x_pm.shape
    trans = stn_train(enc.stn, x_pm)
    x = BmmPointsFn.apply(x_pm.contiguous(), trans)
    x = mlp_rows_train([(enc.conv1, enc.bn1, True)], x.reshape(B * N, -1)).view(B, N, 64)
    trans_feat = None
    if enc.feature_transform:
        trans_feat = stn_train(enc.fstn, x)
        x = BmmPointsFn.apply(x, trans_feat)
    g = mlp_rows_train([(enc.conv2, enc.bn2, True), (enc.conv3, enc.bn3, False)], x.reshape(B * N, 64), pool_K=N)
    return g, x, trans, trans_feat


def pointnet_seg_train(net, x: torch.Tensor):
    """PointNetSeg.forward (pointnet.py:243-254) in train() mode: x [B,D,N] -> (log_probs [B,N,k], trans_feat)."""
    ops._need_cuda(x, "x")
    B, _, N = x.shape
    g, pointfeat, _, trans_feat = pointnet_encoder_train(net.feat, x.permute(0, 2, 1))
    rows = torch.cat([g[:, None, :].expand(B, N, g.shape[1]), pointfeat], dim=2).reshape(B * N, -1)       # [global | pointfeat], :128-131
    logits = mlp_rows_train([(net.conv1, net.bn1, True), (net.conv2, net.bn2, True), (net.conv3, net.bn3, True),
                             (net.conv4, None, False)], rows)
    return LogSoftmaxFn.apply(logits).view(B, N, -1), trans_feat


# ------------------------------------------------------------------------------------------------
# train-mode forwards called by the modules (model/pointnet_util.py, model/pointnet2.py)
class GatherPointsFn(torch.autograd.Function):
    """index_points(points, idx) (pointnet_util.py:43-60) for idx [B, ...] with its gradient w.r.t. points: the scatter-add of
    pn_group_bwd_f32 through idx seen as groups of one point, so repeated indices accumulate.  new_xyz = index_points(xyz,
    fps_idx) of sample_and_group (:117) is one use."""

    @staticmethod
    def forward(ctx, points, idx):
        ctx.idx, ctx.N = idx, points.shape[1]
        return ops.index_points(points, idx)

    @staticmethod
    @once_differentiable
    def backward(ctx, dout):
        B, C = ctx.idx.shape[0], dout.shape[-1]
        flat = ctx.idx.reshape(B, -1, 1)
        if flat.shape[1] == 0:
            return torch.zeros((B, ctx.N, C), dtype=torch.float32, device=dout.device), None
        return ops.group_backward(_rows_of(dout, C), 0, C, flat, ctx.N), None


class GroupPointsFn(torch.autograd.Function):
    """new_points of sample_and_group (pointnet_util.py:127-131) = [xyz[idx] - new_xyz, points[idx]], or of
    sample_and_group_all (:151-156, recentred=False: xyz[idx] as it is), with the gradients w.r.t. xyz and new_xyz
    (pn_group_bwd_xyz_f32 on the xyz columns) and w.r.t. points (pn_group_bwd_f32 on the feature columns)."""

    @staticmethod
    def forward(ctx, xyz_pm, pts_pm, new_xyz, idx, recentred):
        ctx.idx, ctx.N, ctx.recentred = idx, xyz_pm.shape[1], recentred
        ctx.D = pts_pm.shape[2] if pts_pm is not None else 0
        return ops.group(xyz_pm, pts_pm, new_xyz, idx, msg_order=False)

    @staticmethod
    @once_differentiable
    def backward(ctx, dout):
        rows = _rows_of(dout, 3 + ctx.D)
        dxyz = dnew = dpts = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[2]:
            dxyz, dnew = ops.group_backward_xyz(rows, 0, ctx.idx, ctx.N, recentred=ctx.recentred and ctx.needs_input_grad[2])
        if ctx.D and ctx.needs_input_grad[1]:
            dpts = ops.group_backward(rows, 3, ctx.D, ctx.idx, ctx.N)
        return dxyz if ctx.needs_input_grad[0] else None, dpts, dnew, None, None


class SquareDistanceFn(torch.autograd.Function):
    """square_distance (pointnet_util.py:19-40) with the gradients w.r.t. src and dst (pn_square_distance_bwd_f32: one read
    of the incoming [B, N, M] gradient)."""

    @staticmethod
    def forward(ctx, src, dst):
        ctx.save_for_backward(src, dst)
        return ops.square_distance(src, dst)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        src, dst = ctx.saved_tensors
        return ops.square_distance_backward(g, src, dst, ctx.needs_input_grad[0], ctx.needs_input_grad[1])


class ChamferFn(torch.autograd.Function):
    """chamfer_batch (divisor = B) / chamfer_non_batch (divisor = 1) of model/chamfer.py:7-53 with the gradients w.r.t. both
    clouds: the forward keeps each p1 point's nearest p2 point (pn_chamfer_argmin_f32), the backward differentiates the norm
    of that pair (pn_chamfer_bwd_f32).  The value is the forward-only path's: the fp64 sum divided by the divisor, in fp32."""

    @staticmethod
    def forward(ctx, p1, p2, divisor):
        total, ctx.argmin = ops.chamfer_argmin(p1, p2)
        ctx.save_for_backward(p1, p2)
        ctx.scale = 1.0 / divisor
        return (total[0] / divisor).to(torch.float32)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        p1, p2 = ctx.saved_tensors
        dp1, dp2 = ops.chamfer_backward(p1, p2, ctx.argmin, g, ctx.scale, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return dp1, dp2, None


def sample_and_group_train(npoint, radius, nsample, xyz: torch.Tensor, points: Optional[torch.Tensor], returnfps=False,
                           start_idx=None):
    """sample_and_group (pointnet_util.py:110-137) with gradients w.r.t. xyz and points: sampling and ball query run on the
    detached coordinates (index outputs carry no gradient, as in the reference); the gathers and the recentring are
    differentiated.  Same draws and indices as the forward-only path."""
    from .model.pointnet_util import farthest_point_sample

    with torch.no_grad():
        xyz_d = xyz.detach()
        fps_idx = farthest_point_sample(xyz_d, npoint, start_idx)
        new_xyz = ops.index_points(xyz_d, fps_idx)
        idx = ops.ball_query(radius, nsample, xyz_d, new_xyz)
    grad_xyz = _wants_grad(xyz)
    if grad_xyz:
        new_xyz = GatherPointsFn.apply(xyz, fps_idx)
    new_points = GroupPointsFn.apply(xyz, points, new_xyz, idx, True)
    if returnfps:
        grouped_xyz = GatherPointsFn.apply(xyz, idx) if grad_xyz else ops.index_points(xyz, idx)
        return new_xyz, new_points, grouped_xyz, fps_idx
    return new_xyz, new_points


def _wants_grad(t: Optional[torch.Tensor]) -> bool:
    return t is not None and t.requires_grad and torch.is_grad_enabled()


def set_abstraction_train(mod, xyz: torch.Tensor, points: Optional[torch.Tensor], start_idx=None, geometry=None):
    """geometry: (new_xyz [B,S,3], group_idx [B,S,K]) when the caller has computed them already (side stream), with
    fps_idx [B,S] as a third element when xyz requires a gradient (new_xyz is then re-gathered differentiably)."""
    grad_xyz = _wants_grad(xyz)
    xyz_pm = (xyz if grad_xyz else xyz.detach()).permute(0, 2, 1)
    pts_pm = points.permute(0, 2, 1) if points is not None else None
    if mod.group_all:
        # sample_and_group_all (pointnet_util.py:140-157): one group holding every point, centroid = origin, no recentring
        # (x - 0 == x exactly, so the same gather kernel serves); the max then runs over all N rows of a cloud
        B, N, _ = xyz_pm.shape
        new_xyz = torch.zeros((B, 1, 3), dtype=torch.float32, device=xyz.device)
        idx = torch.arange(N, dtype=torch.int64, device=xyz.device).expand(B, 1, N).contiguous()
    else:
        if geometry is None:
            with torch.no_grad():
                geometry = mod.geometry(xyz_pm.detach(), start_idx, with_fps=grad_xyz)
        new_xyz, idx = geometry[0], geometry[1]
        if grad_xyz:
            if len(geometry) < 3:
                raise ValueError("set_abstraction_train: xyz requires a gradient, so the geometry must carry the FPS indices")
            new_xyz = GatherPointsFn.apply(xyz_pm, geometry[2])
    layers = SetAbstractionFn._layers(mod, None)
    pooled = SetAbstractionFn.apply(mod, None, xyz_pm, pts_pm, new_xyz, idx, *_layer_params(layers))
    return new_xyz.permute(0, 2, 1), pooled.permute(0, 2, 1)


def set_abstraction_msg_train(mod, xyz: torch.Tensor, points: Optional[torch.Tensor], start_idx=None):
    """PointNetSetAbstractionMsg.forward (pointnet_util.py:224-261) in train() mode: one FPS, then per radius ball query ->
    grouping ([features, xyz_rel]) -> shared MLP with batch statistics -> max; the scales are concatenated on the channels."""
    from .model.pointnet_util import farthest_point_sample

    grad_xyz = _wants_grad(xyz)
    xyz_pm = (xyz if grad_xyz else xyz.detach()).permute(0, 2, 1)
    pts_pm = points.permute(0, 2, 1) if points is not None else None
    with torch.no_grad():
        fps_idx = farthest_point_sample(xyz_pm.detach(), mod.npoint, start_idx)
    new_xyz = GatherPointsFn.apply(xyz_pm, fps_idx) if grad_xyz else ops.index_points(xyz_pm, fps_idx)
    outs = []
    for i, radius in enumerate(mod.radius_list):
        with torch.no_grad():
            idx = ops.ball_query(radius, mod.nsample_list[i], xyz_pm.detach(), new_xyz.detach())
        layers = SetAbstractionFn._layers(mod, i)
        outs.append(SetAbstractionFn.apply(mod, i, xyz_pm, pts_pm, new_xyz, idx, *_layer_params(layers)))
    return new_xyz.permute(0, 2, 1), torch.cat(outs, dim=2).permute(0, 2, 1)


def feature_propagation_train(mod, xyz1, xyz2, points1, points2, geometry=None):
    """geometry: (idx [B,N,3], weight [B,N,3]) of the 3-NN search when the caller has computed them already."""
    if geometry is None:
        with torch.no_grad():
            geometry = mod.geometry(xyz1.detach().permute(0, 2, 1), xyz2.detach().permute(0, 2, 1))
    idx, w = geometry
    p1 = points1.permute(0, 2, 1) if points1 is not None else None
    layers = [(c, b, True) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
    out = FeaturePropagationFn.apply(mod, p1, points2.permute(0, 2, 1), idx, w, xyz1.permute(0, 2, 1), xyz2.permute(0, 2, 1),
                                     *_layer_params(layers))
    return out.permute(0, 2, 1)


_GEO_STREAMS = {}


def _geometry_stream(device) -> torch.cuda.Stream:
    key = torch.device(device).index
    if key not in _GEO_STREAMS:
        _GEO_STREAMS[key] = torch.cuda.Stream(device)
    return _GEO_STREAMS[key]


_SEED = {"next": 0}


def dropout_seed(device) -> torch.Tensor:
    """{seed, offset} for the Philox stream of one dropout call: the seed comes from torch's CPU generator state
    (so torch.manual_seed makes runs repeatable), the offset counts the calls."""
    _SEED["next"] += 1
    return torch.tensor([torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, _SEED["next"]], dtype=torch.int64).to(device, non_blocking=True)


def semseg_geometry(net, points: torch.Tensor, fps_starts):
    """Everything of a PointNet2SemSeg forward that depends on the coordinates only (no gradient): sampling + ball query of
    the four set-abstraction levels and the four 3-NN searches, on the current stream.
    -> ([(new_xyz [B,S,3], group_idx [B,S,K])] * 4, [(nn_idx [B,N,3], weight [B,N,3])] * 4 indexed like fp1..fp4); the
    set-abstraction tuples also carry fps_idx [B,S] when `points` requires a gradient."""
    sa = [net.sa1, net.sa2, net.sa3, net.sa4]
    fp = [net.fp1, net.fp2, net.fp3, net.fp4]
    with_fps = points.requires_grad
    with torch.no_grad():
        xs_pm = [points[:, :3, :].detach().permute(0, 2, 1)]
        sa_geo, fp_geo = [], [None] * 4
        for i, m in enumerate(sa):
            geo = m.geometry(xs_pm[i], fps_starts[i], with_fps=with_fps)
            xs_pm.append(geo[0])
            sa_geo.append(geo)
        for i in (3, 2, 1, 0):
            fp_geo[i] = fp[i].geometry(xs_pm[i], xs_pm[i + 1])
    return sa_geo, fp_geo


def semseg_forward_train(net, points: torch.Tensor, fps_starts=None, dropout_mask: Optional[torch.Tensor] = None,
                         seed_offset: Optional[torch.Tensor] = None, geometry=None) -> torch.Tensor:
    """PointNet2SemSeg.forward in train() mode (see _semseg_forward_train).  With the fused tensor-core GEMMs every conv weight
    is converted to the kernels' layout ONCE here, for the forward and the backward of this iteration (PackedWeights)."""
    arena = None
    if FUSED_BN and PACK_ONCE and ops.mlp_mode() == "bf16x3" and points.is_cuda:
        arena = net.__dict__.get("_pn_packed")
        if arena is None or not arena.valid():
            arena = net.__dict__["_pn_packed"] = PackedWeights(_net_convs(net))
        if arena.n:
            arena.pack()
        else:
            arena = None
    holders = [net, net.sa1, net.sa2, net.sa3, net.sa4, net.fp4, net.fp3, net.fp2, net.fp1]
    for m in holders:
        m.__dict__["_pn_arena"] = arena          # read by the autograd blocks (kept in their ctx for the backward)
    try:
        return _semseg_forward_train(net, points, fps_starts, dropout_mask, seed_offset, geometry)
    finally:
        for m in holders:
            m.__dict__["_pn_arena"] = None


def _semseg_forward_train(net, points: torch.Tensor, fps_starts=None, dropout_mask: Optional[torch.Tensor] = None,
                          seed_offset: Optional[torch.Tensor] = None, geometry=None) -> torch.Tensor:
    """PointNet2SemSeg.forward (pointnet2.py:159-176) in train() mode -> log-probabilities [B, N, classes] with grad_fn.
    dropout_mask (extension): uint8 [B*N, 128] keep-mask to use instead of drawing one (parity tests)."""
    ops._need_cuda(points, "points")
    xyz = points[:, :3, :]
    feats = points[:, 3:, :] if points.shape[1] > 3 else None
    sa = [net.sa1, net.sa2, net.sa3, net.sa4]
    fp = [net.fp1, net.fp2, net.fp3, net.fp4]                     # fp[i] upsamples level i+1 -> level i
    B, _, N = points.shape
    if geometry is not None:
        # (extension) the caller computed semseg_geometry() for this batch already -- e.g. GraphedTrainStep prefetches it
        # during the previous iteration -- so the feature path starts at once
        sa_geo, fp_geo = geometry
        xs, fs = [xyz], [feats]
        for i, m in enumerate(sa):
            nx, nf = set_abstraction_train(m, xs[-1], fs[-1], geometry=sa_geo[i])
            xs.append(nx)
            fs.append(nf)
        up = fs[4]
        for i in (3, 2, 1, 0):
            up = feature_propagation_train(fp[i], xs[i], xs[i + 1], fs[i] if i > 0 else None, up, geometry=fp_geo[i])
        if dropout_mask is None and seed_offset is None and _dropout_on(net.drop1):
            seed_offset = dropout_seed(points.device)
        params = [net.conv1.weight, net.conv1.bias, net.bn1.weight, net.bn1.bias, net.conv2.weight, net.conv2.bias]
        return SegHeadFn.apply(net, up.permute(0, 2, 1), dropout_mask, seed_offset, *params)[0]
    if fps_starts is None:
        from .model.pointnet_util import draw_fps_starts

        fps_starts = draw_fps_starts(B, [N] + [m.npoint for m in sa[:-1]], points.device)
    # Everything that depends on the coordinates only -- sampling and ball query of the four levels, the four 3-NN
    # searches -- carries no gradient and runs back to back on a side stream; the feature path on the caller's stream
    # waits level by level, so after the level-1 sampling (the long serial kernel) the MLPs overlap the rest of it.
    user = torch.cuda.current_stream(points.device)
    geo = _geometry_stream(points.device)
    capturing = torch.cuda.is_current_stream_capturing()
    sa_geo, fp_geo, sa_ready, fp_ready = [], [None] * 4, [], [None] * 4
    geo.wait_stream(user)
    with_fps = _wants_grad(xyz)                                  # the coordinates' gradient needs the FPS indices
    with torch.no_grad(), torch.cuda.stream(geo):
        xs_pm = [xyz.detach().permute(0, 2, 1)]
        for i, m in enumerate(sa):
            level = m.geometry(xs_pm[i], fps_starts[i], with_fps=with_fps)
            xs_pm.append(level[0])
            sa_geo.append(level)
            ev = torch.cuda.Event()
            ev.record(geo)
            sa_ready.append(ev)
        for i in (3, 2, 1, 0):                                   # fp4 is needed first
            fp_geo[i] = fp[i].geometry(xs_pm[i], xs_pm[i + 1])
            fp_ready[i] = torch.cuda.Event()
            fp_ready[i].record(geo)
        if not capturing:
            for t in [t for pair in sa_geo + fp_geo for t in pair]:
                t.record_stream(user)
    xs, fs = [xyz], [feats]
    for i, m in enumerate(sa):
        user.wait_event(sa_ready[i])
        nx, nf = set_abstraction_train(m, xs[-1], fs[-1], geometry=sa_geo[i])
        xs.append(nx)
        fs.append(nf)
    up = fs[4]
    for i in (3, 2, 1, 0):
        user.wait_event(fp_ready[i])
        up = feature_propagation_train(fp[i], xs[i], xs[i + 1], fs[i] if i > 0 else None, up, geometry=fp_geo[i])
    if dropout_mask is None and seed_offset is None and _dropout_on(net.drop1):
        seed_offset = dropout_seed(points.device)
    params = [net.conv1.weight, net.conv1.bias, net.bn1.weight, net.bn1.bias, net.conv2.weight, net.conv2.bias]
    return SegHeadFn.apply(net, up.permute(0, 2, 1), dropout_mask, seed_offset, *params)[0]


def seg_head_train(net, l0_points: torch.Tensor, dropout_mask=None, seed_offset=None):
    """conv1-bn1-relu-drop1-conv2-log_softmax of the part-segmentation nets in train() mode (pointnet2.py:99-104):
    l0_points [B,128,N] -> (log_probs [B,N,k], feat [B,128,N]), both with grad_fn."""
    if dropout_mask is None and seed_offset is None and _dropout_on(net.drop1):
        seed_offset = dropout_seed(l0_points.device)
    params = [net.conv1.weight, net.conv1.bias, net.bn1.weight, net.bn1.bias, net.conv2.weight, net.conv2.bias]
    logp, feat = SegHeadFn.apply(net, l0_points.permute(0, 2, 1), dropout_mask, seed_offset, *params)
    return logp, feat.permute(0, 2, 1)


# ------------------------------------------------------------------------------------------------
class CrossEntropyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logp, target):
        B, N, k = logp.shape
        loss, dx = ops.cross_entropy(logp.contiguous().view(B * N, k), target)
        ctx.dx, ctx.shape = dx, (B, N, k)
        return loss

    @staticmethod
    def backward(ctx, g):
        return (ctx.dx * g).view(ctx.shape), None


def cross_entropy(logp: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """nn.CrossEntropyLoss()(logp.transpose(2, 1), target) of pcdseg.py:177-178 for logp [B, N, classes], target [B, N]
    (or [B, N, 1]): one kernel computes the loss and its gradient."""
    return CrossEntropyFn.apply(logp, target)


# ------------------------------------------------------------------------------------------------
class FlatAdam:
    """torch.optim.Adam semantics (pcdseg.py:136-141) over ONE flat parameter buffer.

    The module's parameters are re-pointed into `self.flat` and their .grad into `self.grad` (views), so a backward pass
    fills one contiguous gradient: the data-parallel exchange is one all-reduce and the update one kernel launch.
    `param_groups[0]['lr']` may be changed between steps like the reference's decay does (pcdseg.py:160-164)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("FlatAdam: no parameters")
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty((n,), dtype=torch.float32, device=dev)
        self.grad = torch.zeros((n,), dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        o = 0
        for p in self.params:
            k = p.numel()
            self.flat[o:o + k].copy_(p.detach().reshape(-1))
            p.data = self.flat[o:o + k].view(p.shape)
            p.grad = self.grad[o:o + k].view(p.shape)
            p._pn_direct_grad = True          # the backward kernels accumulate straight into the flat gradient
            o += k
        self.param_groups = [{"lr": lr, "betas": betas, "eps": eps, "weight_decay": weight_decay, "params": self.params}]
        # learning rate and step count live on the device (pn_adam_dev_f32): the update is capturable in a CUDA graph
        self._lr_host = float(lr)
        self.lr_dev = torch.full((1,), float(lr), dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros((1,), dtype=torch.int64, device=dev)

    @property
    def steps(self) -> int:
        return int(self.step_dev.item())

    def zero_grad(self, set_to_none: bool = False):
        self.grad.zero_()
        o = 0
        for p in self.params:              # keep .grad pointing into the flat buffer (autograd accumulates in place)
            k = p.numel()
            if p.grad is None or p.grad.data_ptr() != self.grad.data_ptr() + 4 * o:
                p.grad = self.grad[o:o + k].view(p.shape)
            o += k

    def _adopt_stray_grads(self):
        """`net.zero_grad()` (set_to_none) or an assignment to p.grad detaches a parameter from the flat gradient: autograd
        then accumulates into a fresh tensor the update would never see.  Fold such gradients back into the flat buffer and
        re-point .grad (a parameter without a gradient contributes zeros, like torch.optim.Adam skipping it would not --
        so that case raises instead of silently applying stale values)."""
        o = 0
        for p in self.params:
            k = p.numel()
            if p.grad is None:
                raise RuntimeError("FlatAdam: a parameter has no .grad (was net.zero_grad(set_to_none=True) called after the "
                                   "backward pass?); use FlatAdam.zero_grad()")
            if p.grad.data_ptr() != self.grad.data_ptr() + 4 * o:
                self.grad[o:o + k].copy_(p.grad.detach().reshape(-1))
                p.grad = self.grad[o:o + k].view(p.shape)
            o += k

    def all_reduce(self, group=None):
        """Sum the flat gradient over the data-parallel ranks (one NCCL all-reduce of numel*4 bytes); the division by
        the world size is folded into the update (grad_scale)."""
        import torch.distributed as dist

        self._adopt_stray_grads()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=group)
            return 1.0 / dist.get_world_size(group)
        return 1.0

    def step(self, grad_scale: float = 1.0):
        self._adopt_stray_grads()
        g = self.param_groups[0]
        if float(g["lr"]) != self._lr_host:          # the reference's per-epoch decay (pcdseg.py:160-164)
            self._lr_host = float(g["lr"])
            self.lr_dev.fill_(self._lr_host)
        ops.adam_step_dev(self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.lr_dev, self.step_dev, g["betas"], g["eps"],
                          g["weight_decay"], grad_scale)
        self.mark_updated()

    def mark_updated(self):
        """The kernel wrote the parameters through the flat buffer: bump their version counters so that caches keyed on
        them (the eval path's folded / packed weights) notice."""
        torch.autograd.graph.increment_version(self.params)


# ------------------------------------------------------------------------------------------------
class SegMetrics:
    """test_kitti_semseg (pcdseg.py:58-97) with the per-batch, per-class bookkeeping on the device.

        m = SegMetrics(num_classes, device)
        for points, target in loader:  m.update(model(points), target)
        acc, miou, per_class = m.result()          # the only host synchronisation

    Bit-compatible with the reference's arithmetic: iou = 1 if U == 0 else I/U per batch and class (double division,
    added into an fp32 array), count starts at 1 for class 0 (pcdseg.py:61), miou = mean(ious[1:] / count[1:])."""

    def __init__(self, num_classes: int, device):
        self.k = int(num_classes)
        self.ious = torch.zeros((self.k,), dtype=torch.float32, device=device)
        self.count = torch.zeros((self.k,), dtype=torch.int32, device=device)
        self.count[0] = 1
        self.acc_sum = torch.zeros((1,), dtype=torch.float64, device=device)
        self.batches = torch.zeros((1,), dtype=torch.int64, device=device)

    def update(self, logp: torch.Tensor, target: torch.Tensor) -> None:
        from . import _native as nv

        counts = ops.seg_metrics(logp, target)
        points = target.numel()
        with ops._on_device(counts):
            nv.call("pn_seg_metrics_accumulate", counts.data_ptr(), self.k, points, self.ious.data_ptr(), self.count.data_ptr(),
                    self.acc_sum.data_ptr(), self.batches.data_ptr(), ops._stream())

    def result(self):
        import numpy as np

        ious = self.ious.cpu().numpy()
        count = self.count.cpu().numpy().astype(np.uint32)
        categorical = ious / count
        acc = float(self.acc_sum.item() / max(1, int(self.batches.item())))
        return acc, float(np.mean(categorical[1:])), categorical


# ------------------------------------------------------------------------------------------------
def _mode_modules(net) -> List[torch.nn.Module]:
    return [m for m in net.modules() if isinstance(m, (torch.nn.modules.batchnorm._BatchNorm, torch.nn.Dropout))]


def _modes(modules) -> Tuple[bool, ...]:
    return tuple(m.training for m in modules)


class GraphedTrainStep:
    """One training iteration of PointNet2SemSeg as ONE CUDA-graph replay + the gradient exchange + the Adam launch.

    An eager iteration is ~240 kernel launches plus the autograd engine and is bound by the host (7.7 ms at config C5 for
    ~3.5 ms of GPU work); captured once per input shape, forward + loss + backward replay as a single graph launch.

        step = GraphedTrainStep(net, FlatAdam(net.parameters(), lr=1e-3, weight_decay=1e-4))
        loss = step(points, target)                            # points [B, 4, N], target [B, N] -> the (device) loss
        loss = step(points, target, next_points=upcoming)      # ... and prefetch the NEXT batch's geometry meanwhile

    Per call the FPS start indices are drawn on the CPU generator exactly like the reference draws them
    (pointnet_util.py:75) and reach the graph, together with the dropout stream's {seed, offset}, through one small
    pinned staging buffer; the gradient all-reduce (when torch.distributed is initialised) and Adam run right behind
    the replay on the same stream.  Warm-up iterations needed for the capture are rolled back.

    next_points: sampling / ball query / 3-NN depend on the coordinates only, and level-1 sampling is 0.4 ms of serial
    latency at the head of every iteration.  Given the upcoming batch, the replay computes ITS geometry on a side stream
    while the current batch's feature path runs (two static geometry sets, two graphs that alternate); the next call, if
    it gets exactly that batch, starts its feature path at once.  A call whose batch was not prefetched computes the
    geometry first (eagerly); results are the same either way."""

    RING = 8

    def __init__(self, net, optimizer: "FlatAdam", group=None, warmup: int = 2):
        self.net = net.module if hasattr(net, "module") else net
        self.opt, self.group, self.warmup = optimizer, group, warmup
        self._graphs = {}
        self._calls = 0
        self._bn_buffers = [b for m in self.net.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)
                            for b in (m.running_mean, m.running_var, m.num_batches_tracked) if b is not None]
        self._mode_modules = _mode_modules(self.net)

    @staticmethod
    def _starts(st, p):
        return list(st["ctl"][p][:-2].view(4, -1).unbind(0))

    def _forward_backward(self, st, p):
        logp = semseg_forward_train(self.net, st["x"][p], seed_offset=st["ctl"][p][-2:], geometry=st["geo"][p])
        loss = cross_entropy(logp, st["target"])
        self.opt.zero_grad()
        loss.backward()
        return loss

    def _geometry_into(self, st, p):
        """semseg_geometry of the batch in slot p -> the static geometry set p (on the current stream)."""
        sa_geo, fp_geo = semseg_geometry(self.net, st["x"][p], self._starts(st, p))
        if st["geo"][p] is None:
            st["geo"][p] = ([tuple(t.clone() for t in pair) for pair in sa_geo], [tuple(t.clone() for t in pair) for pair in fp_geo])
            return
        for dst, src in zip(st["geo"][p][0] + st["geo"][p][1], sa_geo + fp_geo):
            for d, t in zip(dst, src):
                d.copy_(t)

    def _build(self, points, target):
        from . import _native as nv

        dev = points.device
        B, C, N = points.shape
        net = self.net
        sizes = [N] + [m.npoint for m in (net.sa1, net.sa2, net.sa3)]
        st = {"x": [points.clone(), points.clone()], "target": target.clone().long().view(B, N), "sizes": sizes,
              "ctl": [torch.zeros((4 * B + 2,), dtype=torch.int64, device=dev) for _ in range(2)],
              "geo": [None, None], "pinned": [torch.zeros((4 * B + 2,), dtype=torch.int64).pin_memory() for _ in range(self.RING)],
              "events": [None] * self.RING, "slot": 0, "cur": 0, "prefetched": None, "graphs": [None, None], "loss": [None, None]}
        keep = [t.clone() for t in (self.opt.flat, *self._bn_buffers)]           # warm-up must not train
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self._geometry_into(st, 0)
            self._geometry_into(st, 1)
            for _ in range(self.warmup):
                self._forward_backward(st, 0)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        with torch.no_grad():
            for t, k in zip((self.opt.flat, *self._bn_buffers), keep):
                t.copy_(k)
        geo_stream = torch.cuda.Stream(dev)      # the runner's own side stream: never shared with eager (uncaptured) work
        st["geo_stream"] = geo_stream
        for p in (0, 1):
            graph = torch.cuda.CUDAGraph()
            n0 = nv.launch_count
            with torch.cuda.graph(graph):
                cap = torch.cuda.current_stream(dev)
                geo_stream.wait_stream(cap)
                with torch.cuda.stream(geo_stream):              # the other slot's geometry, beside this slot's feature path
                    self._geometry_into(st, 1 - p)
                st["loss"][p] = self._forward_backward(st, p)
                cap.wait_stream(geo_stream)
            st["launches"] = nv.launch_count - n0                 # entry-point calls captured in a graph (bench accounting)
            st["graphs"][p] = graph
        return st

    def _stage(self, st, p, B):
        """Draws the FPS starts of the batch in slot p like the reference draws them and sends them, with the dropout
        stream's {seed, offset}, to the slot's control buffer."""
        slot = st["slot"] = (st["slot"] + 1) % self.RING
        if st["events"][slot] is not None:
            st["events"][slot].synchronize()
        pinned = st["pinned"][slot]
        for i, n in enumerate(st["sizes"]):                   # the reference's draws, same generator, same order
            pinned[i * B:(i + 1) * B] = torch.randint(0, n, (B,), dtype=torch.long)
        self._calls += 1
        pinned[-2] = torch.initial_seed() & 0x7FFFFFFFFFFFFFFF
        pinned[-1] = self._calls
        st["ctl"][p].copy_(pinned, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        st["events"][slot] = ev

    def __call__(self, points: torch.Tensor, target: torch.Tensor, next_points: Optional[torch.Tensor] = None) -> torch.Tensor:
        from . import _native as nv

        if not self.net.training:
            raise RuntimeError("GraphedTrainStep: call net.train() first")
        # a graph bakes in which BatchNorm layers use batch statistics and which dropouts apply: one capture per mode set
        key = (tuple(points.shape), points.device, _modes(self._mode_modules))
        st = self._graphs.get(key)
        if st is None:
            st = self._graphs[key] = self._build(points, target)
        B = points.shape[0]
        # the prefetched batch is recognised by storage and version; the runner keeps a reference to it until then, so the
        # storage cannot have been freed and handed to another tensor in between
        ref = st["prefetched"]
        if ref is not None and points.data_ptr() == ref[0].data_ptr() and points._version == ref[1] and points.shape == ref[0].shape:
            p = st["cur"] = 1 - st["cur"]                       # this batch's geometry was computed during the last replay
        else:
            p = st["cur"]
            st["x"][p].copy_(points, non_blocking=True)
            self._stage(st, p, B)
            self._geometry_into(st, p)
        if next_points is not None:
            st["x"][1 - p].copy_(next_points, non_blocking=True)
            self._stage(st, 1 - p, B)
            st["prefetched"] = (next_points, next_points._version)
        else:
            st["prefetched"] = None       # (the replay then recomputes the other slot's old geometry: harmless, no draws consumed)
        if target.data_ptr() != st["target"].data_ptr():
            st["target"].copy_(target.view(st["target"].shape), non_blocking=True)
        st["graphs"][p].replay()
        nv.launch_count += st["launches"]
        torch.autograd.graph.increment_version(self._bn_buffers)
        self.opt.step(self.opt.all_reduce(self.group))
        return st["loss"][p]


class GraphedStep:
    """Generic CUDA-graph training iteration for nets whose train-mode forward draws nothing on the host (PointNetSeg: no
    sampling, no dropout): forward + loss + backward are captured once per input shape and replayed; the gradient exchange and
    Adam follow on the same stream.  loss_fn(net, points, target) -> scalar loss tensor with grad_fn.

        step = GraphedStep(net, FlatAdam(net.parameters(), ...),
                           lambda net, x, t: cross_entropy((out := net(x))[0], t) + feature_transform_reguliarzer(out[1]) * 0.001)
        loss = step(points, target)
    """

    def __init__(self, net, optimizer: "FlatAdam", loss_fn, group=None, warmup: int = 2):
        self.net = net.module if hasattr(net, "module") else net
        self.opt, self.loss_fn, self.group, self.warmup = optimizer, loss_fn, group, warmup
        self._graphs = {}
        self._bn_buffers = [b for m in self.net.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)
                            for b in (m.running_mean, m.running_var, m.num_batches_tracked) if b is not None]
        self._mode_modules = _mode_modules(self.net)

    def _fb(self, st):
        loss = self.loss_fn(self.net, st["x"], st["target"])
        self.opt.zero_grad()
        loss.backward()
        return loss

    def _build(self, points, target):
        from . import _native as nv

        dev = points.device
        st = {"x": points.clone(), "target": target.clone()}
        keep = [t.clone() for t in (self.opt.flat, *self._bn_buffers)]           # warm-up must not train
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self._fb(st)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        with torch.no_grad():
            for t, k in zip((self.opt.flat, *self._bn_buffers), keep):
                t.copy_(k)
        graph = torch.cuda.CUDAGraph()
        n0 = nv.launch_count
        with torch.cuda.graph(graph):
            st["loss"] = self._fb(st)
        st["launches"], st["graph"] = nv.launch_count - n0, graph
        return st

    def __call__(self, points: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        from . import _native as nv

        if not self.net.training:
            raise RuntimeError("GraphedStep: call net.train() first")
        key = (tuple(points.shape), tuple(target.shape), points.device, _modes(self._mode_modules))
        st = self._graphs.get(key)
        if st is None:
            st = self._graphs[key] = self._build(points, target)
        if points.data_ptr() != st["x"].data_ptr():
            st["x"].copy_(points, non_blocking=True)
        if target.data_ptr() != st["target"].data_ptr():
            st["target"].copy_(target, non_blocking=True)
        st["graph"].replay()
        nv.launch_count += st["launches"]
        torch.autograd.graph.increment_version(self._bn_buffers)
        self.opt.step(self.opt.all_reduce(self.group))
        return st["loss"]
