"""B200-native drop-in for the reference's model/pointnet_util.py.

Same names, argument order, layouts and state_dict as the reference (so its checkpoints load
unchanged), but every step is a hand-written sm_100a kernel reached through the C ABI of
libpn12_b200.so:

    reference (model/pointnet_util.py)              here
    ------------------------------------------      ---------------------------------------------
    square_distance            :19-40               pn_square_distance_f32 (never used on the hot path)
    index_points               :43-60               pn_index_points_f32
    farthest_point_sample      :63-84               pn_fps_f32 (cluster per cloud, register resident)
    query_ball_point           :87-107              pn_ball_query_grid_f32 (uniform-grid buckets, N >= 4096) /
                                                    pn_ball_query_f32 (ordered scan): no distance cube, no sort
    sample_and_group(_all)     :110-157             the three above + pn_group_f32
    PointNetSetAbstraction     :160-201             pn_sa_mlp_bf16x3: gather + recentre + MLP chain + max in ONE
                                                    tensor-core kernel (pn_linear_f32 + pn_group_max_f32 in fp32 mode)
    PointNetSetAbstractionMsg  :204-261             same, one ball query per radius, MSG channel order
    PointNetFeaturePropagation :264-313             pn_three_nn_f32 / pn_three_nn_blocks_f32 + pn_fp_mlp_bf16x3:
                                                    interpolation + concat + MLP chain in ONE tensor-core kernel
                                                    (pn_three_interpolate_f32 + pn_linear_f32 in fp32 mode)

Functions take point-major [B, N, C] float32 CUDA tensors (strided views welcome) and return int64
indices; modules take and return channel-major [B, C, N] like the reference.  Internally features stay
point-major (a row per point, channels contiguous); the channel-major tensors the modules return are
views of that storage, so chaining modules costs no transposes.

eval(): BatchNorm is folded into the conv weights from the running statistics and the fused tensor-core chains run.
train(): PointNetSetAbstraction and PointNetFeaturePropagation normalise with batch statistics and return tensors with a
grad_fn (pointnet12_b200/train.py: forward and backward on our kernels), and so does PointNetSetAbstractionMsg.
The functions (square_distance, index_points, sample_and_group(_all)) return results with a grad_fn when grad mode is on
and a floating-point input requires a gradient, like the reference's torch expressions; index outputs carry none.
CPU tensors raise: there is no CPU fallback.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from .. import ops


# ------------------------------------------------------------------------------------------------
# L1 primitives
def grad_path(*inputs) -> bool:
    """Whether grad mode is on and one of the floating-point tensor inputs requires a gradient: then the function-level API
    returns results with a grad_fn (pointnet12_b200/train.py), otherwise it makes the forward-only launches."""
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.is_floating_point() and t.requires_grad
                                           for t in inputs)


def square_distance(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """[B,N,3] x [B,M,3] -> [B,N,M] with the reference's |a|^2 + |b|^2 - 2ab rounding sequence."""
    if grad_path(src, dst):
        from ..train import SquareDistanceFn
        return SquareDistanceFn.apply(src, dst)
    return ops.square_distance(src, dst)


def index_points(points: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """points [B,N,C], idx [B,S] or [B,S,K] -> [B,S,C] / [B,S,K,C]."""
    if grad_path(points):
        from ..train import GatherPointsFn
        return GatherPointsFn.apply(points, idx)
    return ops.index_points(points, idx)


def farthest_point_sample(xyz: torch.Tensor, npoint: int, start_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
    """xyz [B,N,3] -> centroids [B,npoint] int64.

    The first centroid is drawn exactly like the reference draws it -- torch.randint on the CPU default
    generator (pointnet_util.py:75) -- so torch.manual_seed(s) reproduces the reference's indices.
    `start_idx` ([B], any device) overrides the draw.
    """
    B, N, _ = xyz.shape
    if start_idx is None:
        start_idx = torch.randint(0, N, (B,), dtype=torch.long)
    elif not start_idx.is_cuda and (int(start_idx.min()) < 0 or int(start_idx.max()) >= N):
        raise IndexError(f"start_idx out of range for N={N}")
    if not start_idx.is_cuda:
        start_idx = start_idx.to(xyz.device, non_blocking=True)
    return ops.fps(xyz, npoint, start_idx)


def query_ball_point(radius: float, nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor) -> torch.Tensor:
    """xyz [B,N,3], new_xyz [B,S,3] -> group_idx [B,S,nsample] int64: first nsample in-ball points in index order."""
    return ops.ball_query(radius, nsample, xyz, new_xyz)


# The HostDraws log (pointnet12_b200/train.py) of a CUDA-graph training runner while it warms up and captures, else None.
draw_log = None


def draw_fps_starts(batch: int, level_sizes: Sequence[int], device) -> List[torch.Tensor]:
    """All FPS start-index draws of one forward, made up front in call order on the CPU generator (the very
    torch.randint calls of pointnet_util.py:75, so torch.manual_seed reproduces the reference), staged in one
    pinned buffer and sent with a single asynchronous copy: the host never waits for the device mid-forward.
    While a graph runner records (`draw_log`), nothing is drawn: the starts are views of its control buffer, which the
    runner fills with these same draws before every replay."""
    if draw_log is not None:
        n = len(level_sizes)
        return list(draw_log.take(("fps", int(batch), tuple(int(s) for s in level_sizes)), n * batch).view(n, batch).unbind(0))
    draws = torch.stack([torch.randint(0, n, (batch,), dtype=torch.long) for n in level_sizes]).pin_memory()
    return list(draws.to(device, non_blocking=True).unbind(0))


def sample_and_group(npoint: int, radius: float, nsample: int, xyz: torch.Tensor, points: Optional[torch.Tensor],
                     returnfps: bool = False, start_idx: Optional[torch.Tensor] = None):
    """-> new_xyz [B,npoint,3], new_points [B,npoint,nsample,3+D] (xyz relative to the centroid first)."""
    if grad_path(xyz, points):
        from ..train import sample_and_group_train
        return sample_and_group_train(npoint, radius, nsample, xyz, points, returnfps, start_idx)
    fps_idx = farthest_point_sample(xyz, npoint, start_idx)
    new_xyz = ops.index_points(xyz, fps_idx)
    idx = ops.ball_query(radius, nsample, xyz, new_xyz)
    new_points = ops.group(xyz, points, new_xyz, idx, msg_order=False)
    if returnfps:
        return new_xyz, new_points, ops.index_points(xyz, idx), fps_idx
    return new_xyz, new_points


def sample_and_group_all(xyz: torch.Tensor, points: Optional[torch.Tensor]):
    """-> new_xyz zeros [B,1,3], new_points [B,1,N,3+D]: one group holding every point, not recentred."""
    B, N, _ = xyz.shape
    new_xyz = torch.zeros((B, 1, 3), dtype=torch.float32, device=xyz.device)
    everyone = torch.arange(N, dtype=torch.int64, device=xyz.device).expand(B, 1, N).contiguous()
    if grad_path(xyz, points):
        from ..train import GroupPointsFn
        return new_xyz, GroupPointsFn.apply(xyz, points, new_xyz, everyone, False)
    return new_xyz, ops.group(xyz, points, new_xyz, everyone, msg_order=False)   # x - 0 == x exactly


# ------------------------------------------------------------------------------------------------
# BatchNorm folding shared by the blocks and the networks
def fold_conv_bn(conv: nn.Module, bn: Optional[nn.Module]) -> Tuple[torch.Tensor, torch.Tensor]:
    """(W', b') with eval-mode BatchNorm folded in: W' = W*g/sqrt(var+eps), b' = (b-mean)*g/sqrt(var+eps)+beta."""
    w = conv.weight.detach().reshape(conv.weight.shape[0], -1).float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(w.shape[0], device=w.device)
    if bn is not None:
        scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        w = w * scale[:, None]
        b = (b - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()
    return w.contiguous(), b.contiguous()


class FoldedLayers:
    """Lazily folded (W', b') list for a conv/bn chain; refolded when any parameter or buffer changes."""

    def __init__(self):
        self._key = None
        self._layers: List[Tuple[torch.Tensor, torch.Tensor]] = []

    @staticmethod
    def _tensors(convs, bns):
        for conv, bn in zip(convs, bns):
            yield conv.weight
            if conv.bias is not None:
                yield conv.bias
            if bn is not None:
                yield from (bn.weight, bn.bias, bn.running_mean, bn.running_var)

    def get(self, convs: Sequence[nn.Module], bns: Sequence[Optional[nn.Module]]):
        key = tuple((t.data_ptr(), t._version) for t in self._tensors(convs, bns))
        if key != self._key:
            self._layers = [fold_conv_bn(c, b) for c, b in zip(convs, bns)]
            self._key = key
            self._chain = None
        return self._layers

    def chain(self, convs: Sequence[nn.Module], bns: Sequence[Optional[nn.Module]],
              relus: Optional[Sequence[bool]] = None, xyz_last: bool = False) -> Optional[ops.PackedChain]:
        """The same layers packed for the tensor-core kernels, or None when the mode is 'fp32' or the chain
        does not fit them (then the caller uses the layer-by-layer CUDA-core path).
        xyz_last: the first layer's input columns are rotated from [xyz_rel(3), features] (sample_and_group order,
        pointnet_util.py:131) to [features, xyz_rel]: the same dot products, but the gathered feature rows then start
        at channel 0 and can be read with aligned 16-byte loads (the kernel is called with msg_order=1)."""
        if ops.mlp_mode() != "bf16x3":
            return None
        layers = self.get(convs, bns)
        if getattr(self, "_chain", None) is None:
            dims = [(w.shape[1], w.shape[0]) for w, _ in layers]
            if not ops.PackedChain.supported(dims):
                self._chain = False
            else:
                relus = [True] * len(layers) if relus is None else list(relus)
                packed = [(w, b, r) for (w, b), r in zip(layers, relus)]
                if xyz_last:
                    w0, b0, r0 = packed[0]
                    packed[0] = (torch.cat([w0[:, 3:], w0[:, :3]], 1).contiguous(), b0, r0)
                self._chain = ops.PackedChain(packed)
        return self._chain or None

    def layer_chains(self, convs, bns, relus=None, xyz_last: bool = False):
        """Every layer as its own packed single-layer chain (for levels with so few row tiles that a fused chain
        would leave most SMs idle: a single-layer launch is N-sliced over the grid instead), or None."""
        if ops.mlp_mode() != "bf16x3":
            return None
        layers = self.get(convs, bns)
        if getattr(self, "_per_layer", None) is None or self._per_layer_key is not self._layers:
            dims = [(w.shape[1], w.shape[0]) for w, _ in layers]
            if not all(ops.PackedChain.supported([d]) for d in dims):
                self._per_layer = False
            else:
                relus = [True] * len(layers) if relus is None else list(relus)
                packed = [(w, b, r) for (w, b), r in zip(layers, relus)]
                if xyz_last:
                    w0, b0, r0 = packed[0]
                    packed[0] = (torch.cat([w0[:, 3:], w0[:, :3]], 1).contiguous(), b0, r0)
                self._per_layer = [ops.PackedChain([t]) for t in packed]
            self._per_layer_key = self._layers
        return self._per_layer or None

    def chain_resident_split(self, convs, bns, relus=None, xyz_last: bool = False):
        """(first, rest): the chain cut after its first layer, when the whole chain is too large to keep its weights in shared
        memory but both parts are not.  A level with many row tiles then runs as two resident-weight launches with the first
        layer's output rows in between (HBM traffic of rows * C1 * 8 bytes) instead of re-streaming every layer's weights for
        every 128-row tile.  None when the chain fits as a whole, a part does not fit, or the mode is 'fp32'."""
        if ops.mlp_mode() != "bf16x3" or len(convs) < 2:
            return None
        layers = self.get(convs, bns)
        if getattr(self, "_res_split", None) is None or self._res_split_key is not self._layers:
            whole = self.chain(convs, bns, relus, xyz_last=xyz_last)
            self._res_split = False
            if whole is not None and not whole.resident:
                relus_l = [True] * len(layers) if relus is None else list(relus)
                packed = [(w, b, r) for (w, b), r in zip(layers, relus_l)]
                if xyz_last:
                    w0, b0, r0 = packed[0]
                    packed[0] = (torch.cat([w0[:, 3:], w0[:, :3]], 1).contiguous(), b0, r0)
                dims = [(w.shape[1], w.shape[0]) for w, _, _ in packed]
                if ops.PackedChain.supported(dims[:1]) and ops.PackedChain.supported(dims[1:]):
                    first, rest = ops.PackedChain(packed[:1]), ops.PackedChain(packed[1:])
                    if first.resident and rest.resident:
                        self._res_split = (first, rest)
            self._res_split_key = self._layers
        return self._res_split or None

    def chain_skip_split(self, convs, bns, relus, d1: int):
        """(skip, rest) for a feature-propagation level with skip input: the first layer's weight is cut at column d1 --
        `skip` = W[:, :d1] alone (no bias, no activation: applied to the skip features ahead of time), `rest` = the chain
        with W[:, d1:] as its first layer (the interpolated half; the kernel adds the skip term before the activation).
        None when the mode is 'fp32', the chain is a single layer or a part does not fit."""
        if ops.mlp_mode() != "bf16x3" or len(convs) < 2:
            return None
        layers = self.get(convs, bns)
        if getattr(self, "_skip_split", None) is None or self._skip_split_key is not self._layers:
            (w0, b0), rest = layers[0], layers[1:]
            dims_b = [(w0.shape[1] - d1, w0.shape[0])] + [(w.shape[1], w.shape[0]) for w, _ in rest]
            if not (0 < d1 < w0.shape[1] and ops.PackedChain.supported([(d1, w0.shape[0])]) and ops.PackedChain.supported(dims_b)):
                self._skip_split = False
            else:
                self._skip_split = (ops.PackedChain([(w0[:, :d1].contiguous(), None, False)]),
                                    ops.PackedChain([(w0[:, d1:].contiguous(), b0, relus[0])] +
                                                    [(w, b, r) for (w, b), r in zip(rest, relus[1:])]))
            self._skip_split_key = self._layers
        return self._skip_split or None

    def chain_folded_first(self, convs, bns, relus):
        """(first, rest): the first layer as a one-layer chain WITHOUT activation and the remaining layers, for a
        feature-propagation level without skip input: conv(interp(p2)) + b == interp(conv(p2) + b) because the
        interpolation is linear and its weights sum to one, so the first layer runs once over the coarse points and
        the fine level starts from relu(interp(.)).  None when the mode is 'fp32' or a part does not fit."""
        if ops.mlp_mode() != "bf16x3" or len(convs) < 2:
            return None
        layers = self.get(convs, bns)
        if getattr(self, "_split", None) is None or self._split_key is not self._layers:
            dims = [(w.shape[1], w.shape[0]) for w, _ in layers]
            if not (relus[0] and ops.PackedChain.supported(dims[:1]) and ops.PackedChain.supported(dims[1:])):
                self._split = False
            else:
                (w0, b0), rest = layers[0], layers[1:]
                self._split = (ops.PackedChain([(w0, b0, False)]),
                               ops.PackedChain([(w, b, r) for (w, b), r in zip(rest, relus[1:])]))
            self._split_key = self._layers
        return self._split or None


RESIDENT_SPLIT_MIN_TILES = 1024     # row tiles from which re-streaming a chain's weights per tile costs more than the split


def _eval_only(module: nn.Module) -> None:
    if module.training:
        raise NotImplementedError(
            f"{type(module).__name__}: only the inference forward is implemented in this round "
            "(BatchNorm is folded from running statistics); call .eval() first")


def autograd_path(module: nn.Module, *inputs) -> bool:
    """Whether a module runs on the autograd blocks of pointnet12_b200/train.py: in training mode, and in eval mode when grad
    mode is on and one of its floating-point inputs requires a gradient -- there BatchNorm normalises with its running
    statistics and dropout is the identity, as in the torch modules.  Otherwise the fused eval forward runs (no grad_fn)."""
    return module.training or grad_path(*inputs)


def _mlp_rows(rows: torch.Tensor, layers) -> torch.Tensor:
    for w, b in layers:
        rows = ops.linear(rows, w, b, relu=True)
    return rows


# ------------------------------------------------------------------------------------------------
# L2 blocks
class PointNetSetAbstraction(nn.Module):
    """Sample (FPS) -> group (ball query) -> shared MLP -> max over the group.  Reference :160-201."""

    def __init__(self, npoint, radius, nsample, in_channel, mlp, group_all):
        super().__init__()
        self.npoint, self.radius, self.nsample, self.group_all = npoint, radius, nsample, group_all
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        c = in_channel
        for width in mlp:
            self.mlp_convs.append(nn.Conv2d(c, width, 1))
            self.mlp_bns.append(nn.BatchNorm2d(width))
            c = width
        self._folded = FoldedLayers()

    # The level splits into a geometry half (depends on xyz only: FPS + ball query) and a feature half
    # (grouping + MLP + max).  The networks run the geometry of all levels on side streams.
    def geometry(self, xyz_pm: torch.Tensor, start_idx: Optional[torch.Tensor] = None, with_fps: bool = False):
        """xyz_pm [B,N,3] -> (new_xyz [B,S,3], group_idx [B,S,K]), and fps_idx [B,S] as a third element when `with_fps`
        (the training path differentiates new_xyz = xyz[fps_idx] when the coordinates require a gradient)."""
        fps_idx = farthest_point_sample(xyz_pm, self.npoint, start_idx)
        new_xyz = ops.index_points(xyz_pm, fps_idx)
        idx = ops.ball_query(self.radius, self.nsample, xyz_pm, new_xyz)
        return (new_xyz, idx, fps_idx) if with_fps else (new_xyz, idx)

    def features(self, xyz_pm, pts_pm, new_xyz, idx) -> torch.Tensor:
        """-> pooled [B,S,C'] point-major."""
        B, S, K = idx.shape
        tc_ok = K == 16 or K % 32 == 0          # group sizes the fused kernel pools
        if K == 32 and len(self.mlp_convs) > 1 and B * S * K // 128 < ops.LAYERWISE_MAX_TILES:
            per_layer = self._folded.layer_chains(self.mlp_convs, self.mlp_bns, xyz_last=True)
            if per_layer is not None:
                # few row tiles: layer by layer, every launch N-sliced over the whole GPU
                rows = ops.sa_mlp_max_tc(per_layer[0], xyz_pm, pts_pm, new_xyz, idx, msg_order=True, out_mode=ops.OUT_ROWS)
                for c in per_layer[1:-1]:
                    rows = ops.mlp_rows_tc(c, rows)
                return ops.mlp_rows_tc(per_layer[-1], rows, ops.OUT_MAX32).view(B, S, -1)
        chain = self._folded.chain(self.mlp_convs, self.mlp_bns, xyz_last=True) if tc_ok else None
        if chain is not None:
            # one kernel: gather + recentre + concat -> tensor-core MLP chain -> max over the group
            # (weights packed with the xyz columns last, hence msg_order=True: aligned feature gathers)
            return ops.sa_mlp_max_tc(chain, xyz_pm, pts_pm, new_xyz, idx, msg_order=True)
        grouped = ops.group(xyz_pm, pts_pm, new_xyz, idx, msg_order=False)
        rows = _mlp_rows(grouped.view(B * S * K, -1), self._folded.get(self.mlp_convs, self.mlp_bns))
        return ops.group_max(rows, K).view(B, S, -1)

    def forward(self, xyz: torch.Tensor, points: Optional[torch.Tensor], start_idx: Optional[torch.Tensor] = None):
        """xyz [B,3,N], points [B,D,N] or None -> new_xyz [B,3,S], new_points [B,C',S].
        `start_idx` (extension): the FPS start indices, when the caller has already drawn them."""
        if autograd_path(self, xyz, points):
            from ..train import set_abstraction_train      # autograd blocks (SURVEY 8 f-1)
            return set_abstraction_train(self, xyz, points, start_idx)
        xyz_pm = xyz.permute(0, 2, 1)
        pts_pm = points.permute(0, 2, 1) if points is not None else None
        if self.group_all:
            new_xyz, grouped = sample_and_group_all(xyz_pm, pts_pm)
            B, S, K, C = grouped.shape
            per_layer = self._folded.layer_chains(self.mlp_convs, self.mlp_bns)
            if per_layer is not None:
                # the group-all MLP (e.g. 643 -> 256 -> 512 -> 1024) is wider than a fused chain takes (hidden layers <= 256),
                # but every layer alone fits: one tensor-core launch per layer instead of the CUDA-core SGEMM
                rows = grouped.view(B * S * K, C)
                for c in per_layer:
                    rows = ops.mlp_rows_tc(c, rows)
            else:
                rows = _mlp_rows(grouped.view(B * S * K, C), self._folded.get(self.mlp_convs, self.mlp_bns))
            pooled = ops.group_max(rows, K).view(B, S, -1)
        else:
            new_xyz, idx = self.geometry(xyz_pm, start_idx)
            pooled = self.features(xyz_pm, pts_pm, new_xyz, idx)
        return new_xyz.permute(0, 2, 1), pooled.permute(0, 2, 1)


class PointNetSetAbstractionMsg(nn.Module):
    """Multi-scale grouping: one FPS, then per radius ball query -> MLP -> max, scales concatenated.
    Reference :204-261 (channel order inside a group is [features, xyz_rel], :247)."""

    def __init__(self, npoint, radius_list, nsample_list, in_channel, mlp_list):
        super().__init__()
        self.npoint, self.radius_list, self.nsample_list = npoint, radius_list, nsample_list
        self.conv_blocks = nn.ModuleList()
        self.bn_blocks = nn.ModuleList()
        for widths in mlp_list:
            convs, bns = nn.ModuleList(), nn.ModuleList()
            c = in_channel + 3
            for width in widths:
                convs.append(nn.Conv2d(c, width, 1))
                bns.append(nn.BatchNorm2d(width))
                c = width
            self.conv_blocks.append(convs)
            self.bn_blocks.append(bns)
        self._folded = [FoldedLayers() for _ in mlp_list]

    def forward(self, xyz: torch.Tensor, points: Optional[torch.Tensor], start_idx: Optional[torch.Tensor] = None):
        if autograd_path(self, xyz, points):
            from ..train import set_abstraction_msg_train

            return set_abstraction_msg_train(self, xyz, points, start_idx)
        xyz_pm = xyz.permute(0, 2, 1)
        pts_pm = points.permute(0, 2, 1) if points is not None else None
        B = xyz_pm.shape[0]
        S = self.npoint
        new_xyz = ops.index_points(xyz_pm, farthest_point_sample(xyz_pm, S, start_idx))
        widths = [blk[-1].out_channels for blk in self.conv_blocks]
        out = torch.empty((B, S, sum(widths)), dtype=torch.float32, device=xyz.device)
        # (the scales are independent, but running them on three streams was measured SLOWER -- 2.25 vs 1.90 ms at C4: their
        # persistent chain kernels fight for the same SMs -- so they run back to back)
        col = 0
        for i, radius in enumerate(self.radius_list):
            self._scale(i, radius, xyz_pm, pts_pm, new_xyz, out.view(B * S, -1)[:, col:col + widths[i]], B, S)
            col += widths[i]
        return new_xyz.permute(0, 2, 1), out.permute(0, 2, 1)


def _msg_scale(self, i, radius, xyz_pm, pts_pm, new_xyz, out_cols, B, S):
    """One scale of PointNetSetAbstractionMsg on the current stream: ball query -> chain -> max, written into its output
    columns.  Returns the temporaries (kept alive / recorded on the caller's stream by forward)."""
    K = self.nsample_list[i]
    idx = ops.ball_query(radius, K, xyz_pm, new_xyz)
    chain = self._folded[i].chain(self.conv_blocks[i], self.bn_blocks[i]) if (K == 16 or K % 32 == 0) else None
    split = None
    if chain is not None and K % 32 == 0 and B * S * K // 128 >= RESIDENT_SPLIT_MIN_TILES:
        split = self._folded[i].chain_resident_split(self.conv_blocks[i], self.bn_blocks[i])
    if split is not None:
        # many row tiles and a chain too large for shared memory but whose halves fit: two resident-weight launches instead of
        # streaming all weights once per tile
        rows = ops.sa_mlp_max_tc(split[0], xyz_pm, pts_pm, new_xyz, idx, msg_order=True, out_mode=ops.OUT_ROWS)
        part = ops.mlp_rows_tc(split[1], rows, ops.OUT_MAX32)
        ops.group_max(part, K // 32, out=out_cols)
        return (idx, rows, part)
    if chain is not None:
        ops.sa_mlp_max_tc(chain, xyz_pm, pts_pm, new_xyz, idx, msg_order=True, out=out_cols)
        return (idx,)
    grouped = ops.group(xyz_pm, pts_pm, new_xyz, idx, msg_order=True)
    rows = _mlp_rows(grouped.view(B * S * K, -1), self._folded[i].get(self.conv_blocks[i], self.bn_blocks[i]))
    ops.group_max(rows, K, out=out_cols)   # written in place: no concat
    return (idx, grouped, rows)


PointNetSetAbstractionMsg._scale = _msg_scale


class PointNetFeaturePropagation(nn.Module):
    """3-NN inverse-distance interpolation of coarse features onto the fine points, skip concat, MLP.
    Reference :264-313."""

    def __init__(self, in_channel, mlp):
        super().__init__()
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        c = in_channel
        for width in mlp:
            self.mlp_convs.append(nn.Conv1d(c, width, 1))
            self.mlp_bns.append(nn.BatchNorm1d(width))
            c = width
        self._folded = FoldedLayers()

    def geometry(self, x1: torch.Tensor, x2: torch.Tensor, order=None, background: bool = False):
        """x1 [B,N,3] fine points, x2 [B,S,3] coarse points -> (idx [B,N,3], weight [B,N,3]).
        `order`: an ops.BallGrid of the fine cloud (bucket order) -> the pruned block search for large N x S."""
        B, N, _ = x1.shape
        if x2.shape[1] == 1:   # a single coarse point: broadcast it (reference :292-293)
            idx = torch.zeros((B, N, 3), dtype=torch.int64, device=x1.device)
            w = torch.zeros((B, N, 3), dtype=torch.float32, device=x1.device)
            w[:, :, 0] = 1.0             # weights (1, 0, 0) made on the device: no host copy, so a CUDA graph can capture it
            return idx, w
        return ops.three_nn(x1, x2, order=order, background=background)

    def fold_first_layer(self, p2, head=None):
        """(remaining chain, z): the level's first layer applied to the coarse features p2 [B,S,D2] (no activation).
        Needs no neighbour search, so a network can issue it before it waits for the 3-NN result; the value is cached
        until `features` has consumed it.  None when the tensor-core path is off or a part does not fit."""
        cached = getattr(self, "_z_cache", None)
        if cached is not None and cached[0] is p2:
            return cached[1], cached[2]
        convs, bns, relus = list(self.mlp_convs), list(self.mlp_bns), [True] * len(self.mlp_convs)
        folded = self._folded
        if head is not None:
            folded, hconvs, hbns, hrelus, _ = head
            convs, bns, relus = convs + hconvs, bns + hbns, relus + hrelus
        split = folded.chain_folded_first(convs, bns, relus)
        if split is None:
            return None
        first, rest = split
        B, S, D2 = p2.shape
        z = ops.mlp_rows_tc(first, p2.reshape(B * S, D2)).view(B, S, -1)
        self._z_cache = (p2, rest, z)
        return rest, z

    def first_layer_spec(self, head=None):
        """(conv, bn) of this level's first layer if `features` would fold it into the coarse level (no skip input,
        tensor-core engine, chains supported), else None.  A network can then append that layer to the chain of the
        level that PRODUCES the coarse features and hand the result over with `adopt_folded` -- one launch less."""
        if not ops.FOLD_FIRST_FP_LAYER:
            return None
        convs, bns, relus = list(self.mlp_convs), list(self.mlp_bns), [True] * len(self.mlp_convs)
        folded = self._folded
        if head is not None:
            folded, hconvs, hbns, hrelus, _ = head
            convs, bns, relus = convs + hconvs, bns + hbns, relus + hrelus
        if folded.chain_folded_first(convs, bns, relus) is None:
            return None
        return self.mlp_convs[0], self.mlp_bns[0]

    def adopt_folded(self, z: torch.Tensor, head=None) -> None:
        """z [B,S,C1] = this level's first layer (BatchNorm folded, no activation) already applied to the coarse
        features by the caller.  `features(None, z, ...)` then starts from relu(interp(z))."""
        convs, bns, relus = list(self.mlp_convs), list(self.mlp_bns), [True] * len(self.mlp_convs)
        folded = self._folded
        if head is not None:
            folded, hconvs, hbns, hrelus, _ = head
            convs, bns, relus = convs + hconvs, bns + hbns, relus + hrelus
        _, rest = folded.chain_folded_first(convs, bns, relus)
        self._z_cache = (z, rest, z)

    def skip_ahead(self, p1: torch.Tensor, head=None) -> bool:
        """Computes the skip half of the first layer, W[:, :D1] p1, for the skip features p1 [B,N,D1] NOW (on the current
        stream) and keeps it for the next `features(p1, ...)` call with the same tensor, which then only interpolates,
        multiplies the other half and adds this term.  A network calls it on a side stream as soon as p1 exists, long
        before the coarse features arrive.  Returns False when the level cannot be split (then features() is unchanged)."""
        if not ops.FP_SKIP_AHEAD:
            return False
        convs, bns, relus = list(self.mlp_convs), list(self.mlp_bns), [True] * len(self.mlp_convs)
        folded = self._folded
        if head is not None:
            folded, hconvs, hbns, hrelus, _ = head
            convs, bns, relus = convs + hconvs, bns + hbns, relus + hrelus
        B, N, D1 = p1.shape
        split = folded.chain_skip_split(convs, bns, relus, D1)
        if split is None:
            return False
        skip, rest = split
        width = (skip.cout + 31) // 32 * 32
        term = torch.zeros((B, N, width), dtype=torch.float32, device=p1.device)
        ops.mlp_rows_tc(skip, p1.reshape(B * N, D1), out=term.view(B * N, width)[:, :skip.cout])
        self._skip_cache = (p1, rest, term)
        return True

    def features(self, p1, p2, idx, w, head=None, order=None, out=None, clouds=None) -> torch.Tensor:
        """p1 [B,N,D1] or None, p2 [B,S,D2] point-major -> [B,N,D'] point-major.
        `head`: (FoldedLayers, convs, bns, relus, out_mode) appended by a network: the segmentation head runs
        in the same kernel and the result is the [B,N,classes] log-probabilities.
        `order`: an ops.BallGrid of the fine cloud; the fused kernel then walks the points in bucket order.
        `out`, `clouds`: write into a caller-provided [B,N,D'] buffer / compute only the batch slice (b0, b1)
        (tensor-core path only)."""
        B, N, _ = idx.shape
        convs, bns, relus = list(self.mlp_convs), list(self.mlp_bns), [True] * len(self.mlp_convs)
        folded, out_mode = self._folded, ops.OUT_ROWS
        if head is not None:
            folded, hconvs, hbns, hrelus, out_mode = head
            convs, bns, relus = convs + hconvs, bns + hbns, relus + hrelus
        ahead = getattr(self, "_skip_cache", None)
        if ahead is not None:
            self._skip_cache = None
            if ahead[0] is p1 and out is None and clouds is None:
                # the skip half of the first layer was computed ahead of time: interpolate, multiply the other half, add it
                return ops.fp_mlp_tc(ahead[1], None, p2, idx, w, out_mode, order=order, residual=ahead[2])
        if p1 is None and ops.FOLD_FIRST_FP_LAYER and N > p2.shape[1]:
            folded_first = self.fold_first_layer(p2, head)
            if folded_first is not None:
                # first layer at the coarse level (S rows instead of N), then one kernel: relu(weighted 3-row gather)
                # -> the remaining layers (-> head -> log_softmax)
                rest, z = folded_first
                if clouds is None or clouds[1] == B:
                    self._z_cache = None                               # last use in this forward
                return ops.fp_mlp_tc(rest, None, z, idx, w, out_mode, relu_in=True, order=order, out=out, clouds=clouds)
        if (head is None and out is None and clouds is None and len(convs) > 1
                and B * ((N + 127) // 128) < ops.LAYERWISE_MAX_TILES):
            per_layer = folded.layer_chains(convs, bns, relus)
            if per_layer is not None:
                # few row tiles: layer by layer, every launch N-sliced over the whole GPU
                rows = ops.fp_mlp_tc(per_layer[0], p1, p2, idx, w, ops.OUT_ROWS, order=order).view(B * N, -1)
                for c in per_layer[1:]:
                    rows = ops.mlp_rows_tc(c, rows)
                return rows.view(B, N, -1)
        chain = folded.chain(convs, bns, relus)
        if chain is not None:
            # one kernel: weighted 3-row gather + skip concat -> tensor-core MLP chain (-> head -> log_softmax)
            return ops.fp_mlp_tc(chain, p1, p2, idx, w, out_mode, order=order, out=out, clouds=clouds)
        rows = ops.three_interpolate(p1, p2, idx, w).view(B * N, -1)
        for (wt, b), r in zip(folded.get(convs, bns), relus):
            rows = ops.linear(rows, wt, b, relu=r)
        if out_mode == ops.OUT_LOG_SOFTMAX:
            rows = ops.log_softmax(rows)
        return rows.view(B, N, -1)

    def forward(self, xyz1, xyz2, points1, points2):
        """xyz1 [B,3,N], xyz2 [B,3,S], points1 [B,D1,N] or None, points2 [B,D2,S] -> [B,D',N]."""
        if autograd_path(self, xyz1, xyz2, points1, points2):
            from ..train import feature_propagation_train
            return feature_propagation_train(self, xyz1, xyz2, points1, points2)
        idx, w = self.geometry(xyz1.permute(0, 2, 1), xyz2.permute(0, 2, 1))
        p1 = points1.permute(0, 2, 1) if points1 is not None else None
        return self.features(p1, points2.permute(0, 2, 1), idx, w).permute(0, 2, 1)
