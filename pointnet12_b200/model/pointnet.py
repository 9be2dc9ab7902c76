"""B200-native drop-in for the reference's model/pointnet.py (PointNet networks).

Same class names, constructor arguments, submodule names (state_dict keys) and return values as the
reference.  Everything is computed on point-major rows [B*N, C] by the C-ABI kernels:

  * per-point conv chains + max    -> one tensor-core chain each (pn_mlp_rows_bf16x3, pooled in the kernel) +
                                      pn_group_max_f32 over the partial rows; pn_linear_f32 (BatchNorm folded) in
                                      fp32 mode, for layers wider than the chains take, and when N % 32 != 0
  * STN fully connected tail       -> pn_linear_f32 on [B, 1024] rows; the "+ identity" of
                                      pointnet.py:40-43 / 77-83 is folded into fc3's bias
  * torch.bmm(x, trans)            -> pn_linear_f32 with one weight matrix per cloud (w_bstride)
  * seg head on cat([global, pointfeat]) (pointnet.py:128-131, 247): the 1024 global channels are the
    same for every point of a cloud, so that half of conv1 becomes a per-cloud bias
    (bias_bstride) and the per-point work drops from 1088 to 64 input channels.

In train() mode, and in eval() mode on an input that requires a gradient, the nets and their spatial transformers /
encoder run on the autograd blocks of pointnet12_b200/train.py instead; no CPU fallback.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from .. import ops
from .pointnet_util import FoldedLayers, autograd_path


def _chain_global_max(folded: FoldedLayers, convs, bns, relus, rows: torch.Tensor, B: int, N: int) -> Optional[torch.Tensor]:
    """relu(bn(conv)) chain over the [B*N, C] rows followed by the max over the N points of each cloud, as ONE
    tensor-core chain (pn_mlp_rows_bf16x3 pooling runs of 32 rows) + pn_group_max_f32 over the N/32 partial rows.
    None when the tensor-core engine is off, the chain does not fit it, or N is not a multiple of 32."""
    if N % 32:
        return None
    chain = folded.chain(convs, bns, relus)
    if chain is None:
        return None
    part = ops.mlp_rows_tc(chain, rows, ops.OUT_MAX32)            # [B*N/32, C]
    return ops.group_max(part, N // 32)                           # [B, C]


def _point_rows(x_cm: torch.Tensor) -> torch.Tensor:
    """User input [B, C, N] channel-major -> point-major [B, N, C] (layout change of the raw input)."""
    ops._need_cuda(x_cm, "input")
    return x_cm.permute(0, 2, 1).contiguous()


class _STN(nn.Module):
    """Shared implementation of the spatial transformers (pointnet.py:10-84)."""

    def __init__(self, k: int):
        super().__init__()
        self.conv1 = nn.Conv1d(k, 64, 1)
        self.conv2 = nn.Conv1d(64, 128, 1)
        self.conv3 = nn.Conv1d(128, 1024, 1)
        self.fc1 = nn.Linear(1024, 512)
        self.fc2 = nn.Linear(512, 256)
        self.fc3 = nn.Linear(256, k * k)
        self.relu = nn.ReLU()
        self.bn1 = nn.BatchNorm1d(64)
        self.bn2 = nn.BatchNorm1d(128)
        self.bn3 = nn.BatchNorm1d(1024)
        self.bn4 = nn.BatchNorm1d(512)
        self.bn5 = nn.BatchNorm1d(256)
        self.k = k
        self._folded = FoldedLayers()
        self._folded_convs = FoldedLayers()

    def transform_rows(self, x_pm: torch.Tensor) -> torch.Tensor:
        """x_pm [B,N,k] point-major -> [B,k,k]."""
        B, N, k = x_pm.shape
        layers = self._folded.get([self.conv1, self.conv2, self.conv3, self.fc1, self.fc2, self.fc3],
                                  [self.bn1, self.bn2, self.bn3, self.bn4, self.bn5, None])
        h = x_pm.reshape(B * N, k)
        # conv1-3 + max over the points: one tensor-core chain (k -> 64 -> 128 -> 1024, pooled in the kernel)
        g = _chain_global_max(self._folded_convs, [self.conv1, self.conv2, self.conv3], [self.bn1, self.bn2, self.bn3],
                              [True, True, True], h, B, N)
        if g is None:
            for w, b in layers[:3]:
                h = ops.linear(h, w, b, relu=True)
            g = ops.group_max(h, N)                                               # [B,1024]
        # fc1-bn4-relu, fc2-bn5-relu, fc3 on the [B, 1024] rows: one row tile, so each layer is a single-layer tensor-core chain
        # sliced over its output channels (16 CTAs read the 1024 x 512 weights instead of one SIMT tile marching through them:
        # 100 -> ~12 us per layer at B = 1); "+ iden" is added afterwards, in the reference's own order (pointnet.py:40-43)
        slabs = self._fc_chains(layers[3:])
        if slabs is not None:
            for parts in slabs:
                if len(parts) == 1:
                    g = ops.mlp_rows_tc(parts[0][0], g)
                else:        # fc3 of the 64 x 64 transform has 4096 outputs: column slabs of <= 1024, written side by side
                    out = torch.empty((B, sum(c.cout for c, _ in parts)), dtype=torch.float32, device=g.device)
                    for c, col in parts:
                        ops.mlp_rows_tc(c, g, out=out[:, col:col + c.cout])
                    g = out
            return g.view(B, self.k, self.k) + torch.eye(self.k, device=g.device, dtype=g.dtype)
        g = ops.linear(g, *layers[3], relu=True)
        g = ops.linear(g, *layers[4], relu=True)
        w3, b3 = layers[5]
        b3 = b3 + torch.eye(self.k, device=b3.device, dtype=b3.dtype).flatten()   # "+ iden" as a bias
        return ops.linear(g, w3, b3, relu=False).view(B, self.k, self.k)

    def _fc_chains(self, fc_layers):
        """fc1 / fc2 / fc3 (BatchNorm folded) as single-layer tensor-core chains: per layer a list of (chain, first output
        column); layers with more than 1024 outputs are cut into column slabs.  None in fp32 mode / when a layer does not fit.
        Cached until the folded weights change."""
        if ops.mlp_mode() != "bf16x3":
            return None
        cached = self.__dict__.get("_fc_chain_cache")
        if cached is not None and cached[0] is fc_layers[0][0]:
            return cached[1]
        relus = [True, True, False]
        out = []
        for (w, b), relu in zip(fc_layers, relus):
            cout, cin = w.shape
            parts = []
            for col in range(0, cout, 1024):
                n = min(1024, cout - col)
                if not ops.PackedChain.supported([(cin, n)]):
                    out = None
                    break
                parts.append((ops.PackedChain([(w[col:col + n].contiguous(), b[col:col + n].contiguous(), relu)]), col))
            if out is None:
                break
            out.append(parts)
        self.__dict__["_fc_chain_cache"] = (fc_layers[0][0], out)
        return out

    def forward(self, x):
        if autograd_path(self, x):        # autograd blocks (pointnet12_b200/train.py)
            from ..train import stn_train

            ops._need_cuda(x, "input")
            return stn_train(self, x.permute(0, 2, 1))
        return self.transform_rows(_point_rows(x))


class STN3d(_STN):
    """Reference pointnet.py:10-45: [B,3,N] -> [B,3,3]."""

    def __init__(self):
        super().__init__(3)


class STNkd(_STN):
    """Reference pointnet.py:47-84: [B,k,N] -> [B,k,k]."""

    def __init__(self, k=64):
        super().__init__(k)


class PointNetEncoder(nn.Module):
    """Reference pointnet.py:86-131."""

    def __init__(self, global_feat=True, input_dims=4, feature_transform=False):
        super().__init__()
        self.stn = STNkd(k=input_dims)
        self.conv1 = nn.Conv1d(input_dims, 64, 1)
        self.conv2 = nn.Conv1d(64, 128, 1)
        self.conv3 = nn.Conv1d(128, 1024, 1)
        self.bn1 = nn.BatchNorm1d(64)
        self.bn2 = nn.BatchNorm1d(128)
        self.bn3 = nn.BatchNorm1d(1024)
        self.global_feat = global_feat
        self.feature_transform = feature_transform
        if self.feature_transform:
            self.fstn = STNkd(k=64)
        self._folded = FoldedLayers()
        self._folded_tail = FoldedLayers()

    def encode_rows(self, x_pm: torch.Tensor):
        """x_pm [B,N,k] -> (global [B,1024], pointfeat [B,N,64], trans, trans_feat)."""
        B, N, _ = x_pm.shape
        (w1, b1), (w2, b2), (w3, b3) = self._folded.get([self.conv1, self.conv2, self.conv3],
                                                        [self.bn1, self.bn2, self.bn3])
        trans = self.stn.transform_rows(x_pm)
        x = ops.bmm_points(x_pm, trans)                                           # pointnet.py:105-107
        x = ops.linear(x.view(B * N, -1), w1, b1, relu=True).view(B, N, 64)
        trans_feat = None
        if self.feature_transform:
            trans_feat = self.fstn.transform_rows(x)
            x = ops.bmm_points(x, trans_feat)                                     # pointnet.py:111-114
        pointfeat = x
        # relu(bn2(conv2)) -> bn3(conv3) (no ReLU, :120) -> max over the points: one tensor-core chain
        g = _chain_global_max(self._folded_tail, [self.conv2, self.conv3], [self.bn2, self.bn3], [True, False],
                              x.reshape(B * N, 64), B, N)
        if g is None:
            h = ops.linear(x.view(B * N, 64), w2, b2, relu=True)
            h = ops.linear(h, w3, b3, relu=False)
            g = ops.group_max(h, N)
        return g, pointfeat, trans, trans_feat

    def forward(self, x):
        B, _, N = x.shape
        if autograd_path(self, x):        # autograd blocks (pointnet12_b200/train.py)
            from ..train import pointnet_encoder_train

            ops._need_cuda(x, "input")
            g, pointfeat, trans, trans_feat = pointnet_encoder_train(self, x.permute(0, 2, 1))
        else:
            g, pointfeat, trans, trans_feat = self.encode_rows(_point_rows(x))
        if self.global_feat:
            return g, trans, trans_feat
        cat = torch.cat([g.view(B, 1024, 1).expand(B, 1024, N), pointfeat.permute(0, 2, 1)], 1)   # API parity only
        return cat, trans, trans_feat


class PointNetCls(nn.Module):
    """Reference pointnet.py:133-151: [B,3,N] -> (log_probs [B,k], trans_feat)."""

    def __init__(self, k=2, feature_transform=False):
        super().__init__()
        self.feature_transform = feature_transform
        self.feat = PointNetEncoder(global_feat=True, feature_transform=feature_transform, input_dims=3)
        self.fc1 = nn.Linear(1024, 512)
        self.fc2 = nn.Linear(512, 256)
        self.fc3 = nn.Linear(256, k)
        self.dropout = nn.Dropout(p=0.3)
        self.bn1 = nn.BatchNorm1d(512)
        self.bn2 = nn.BatchNorm1d(256)
        self.relu = nn.ReLU()
        self._folded = FoldedLayers()

    def forward(self, x, dropout_mask=None):
        if autograd_path(self, x):
            from ..train import pointnet_cls_train

            return pointnet_cls_train(self, x, dropout_mask)
        g, _, _, trans_feat = self.feat.encode_rows(_point_rows(x))
        (w1, b1), (w2, b2), (w3, b3) = self._folded.get([self.fc1, self.fc2, self.fc3], [self.bn1, self.bn2, None])
        h = ops.linear(g, w1, b1, relu=True)
        h = ops.linear(h, w2, b2, relu=True)                                      # dropout = identity in eval
        return ops.log_softmax(ops.linear(h, w3, b3, relu=False)), trans_feat


class PointNetSeg(nn.Module):
    """Reference pointnet.py:230-254: [B,input_dims,N] -> (log_probs [B,N,num_class], trans_feat [B,64,64])."""

    def __init__(self, num_class, input_dims=4, feature_transform=False):
        super().__init__()
        self.k = num_class
        self.feat = PointNetEncoder(global_feat=False, input_dims=input_dims, feature_transform=feature_transform)
        self.conv1 = nn.Conv1d(1088, 512, 1)
        self.conv2 = nn.Conv1d(512, 256, 1)
        self.conv3 = nn.Conv1d(256, 128, 1)
        self.conv4 = nn.Conv1d(128, self.k, 1)
        self.bn1 = nn.BatchNorm1d(512)
        self.bn2 = nn.BatchNorm1d(256)
        self.bn3 = nn.BatchNorm1d(128)
        self._folded = FoldedLayers()
        self._folded_c2 = FoldedLayers()
        self._folded_tail = FoldedLayers()

    def forward(self, x):
        if autograd_path(self, x):          # autograd blocks (pointnet12_b200/train.py), pcdseg.py:166-186
            from ..train import pointnet_seg_train

            return pointnet_seg_train(self, x)
        B, _, N = x.shape
        g, pointfeat, _, trans_feat = self.feat.encode_rows(_point_rows(x))
        (w1, b1), (w2, b2), (w3, b3), (w4, b4) = self._folded.get(
            [self.conv1, self.conv2, self.conv3, self.conv4], [self.bn1, self.bn2, self.bn3, None])
        # conv1 on cat([global(1024) repeated, pointfeat(64)]): the global half is a per-cloud bias
        cb = self.__dict__.get("_cloud_bias_chain")
        if cb is None or cb[0] is not w1:      # (re)packed when the folded weights change
            chain = None
            if ops.mlp_mode() == "bf16x3" and ops.PackedChain.supported([(1024, w1.shape[0])]):
                chain = ops.PackedChain([(w1[:, :1024].contiguous(), b1, False)])
            cb = self.__dict__["_cloud_bias_chain"] = (w1, chain, w1[:, 1024:].contiguous())
        if cb[1] is not None and ops.mlp_mode() == "bf16x3":
            cloud_bias = ops.mlp_rows_tc(cb[1], g)                                # [B,512]: one N-sliced tensor-core launch
        else:
            cloud_bias = ops.linear(g, w1[:, :1024].contiguous(), b1, relu=False)     # [B,512]
        if cb[1] is not None and ops.mlp_mode() == "bf16x3" and B <= 4:
            # per-point half of conv1 (64 -> 512) on the tensor cores; the per-cloud bias is written into the packed chain's bias
            # table right before each cloud's launch (stream-ordered, so a graph replays it) instead of re-packing the weights
            pc = self.__dict__.get("_point_chain")
            if pc is None or pc[0] is not w1:
                chain = ops.PackedChain([(cb[2], torch.zeros_like(b1), True)])
                pc = self.__dict__["_point_chain"] = (w1, chain, chain.bias_view(0))
            h = torch.empty((B, N, w1.shape[0]), dtype=torch.float32, device=pointfeat.device)
            for b in range(B):
                pc[2].copy_(cloud_bias[b])
                ops.mlp_rows_tc(pc[1], pointfeat[b], out=h[b])
            h = h.view(B * N, w1.shape[0])
        else:
            h = ops.linear_cloud_bias(pointfeat, cb[2], cloud_bias, relu=True).view(B * N, 512)
        # conv2 (512 -> 256) as a single-layer tensor-core chain, conv3 -> conv4 -> log_softmax as one more
        c2 = self._folded_c2.chain([self.conv2], [self.bn2], [True])
        tail = self._folded_tail.chain([self.conv3, self.conv4], [self.bn3, None], [True, False])
        if c2 is not None and tail is not None:
            logp = ops.mlp_rows_tc(tail, ops.mlp_rows_tc(c2, h), ops.OUT_LOG_SOFTMAX)
        else:
            h = ops.linear(h, w2, b2, relu=True)
            h = ops.linear(h, w3, b3, relu=True)
            logp = ops.log_softmax(ops.linear(h, w4, b4, relu=False))
        return logp.view(B, N, self.k), trans_feat


class PointNetDenseCls(nn.Module):
    """Reference pointnet.py:153-228 (ShapeNet part segmentation net):
    forward(point_cloud [B,3,N], label [B,16]) -> (cls logits [B,cat_num], seg log_probs [B,N,part_num], trans_feat)."""

    def __init__(self, cat_num=16, part_num=50):
        super().__init__()
        self.cat_num = cat_num
        self.part_num = part_num
        self.stn = STN3d()
        self.conv1 = nn.Conv1d(3, 64, 1)
        self.conv2 = nn.Conv1d(64, 128, 1)
        self.conv3 = nn.Conv1d(128, 128, 1)
        self.conv4 = nn.Conv1d(128, 512, 1)
        self.conv5 = nn.Conv1d(512, 2048, 1)
        self.bn1 = nn.BatchNorm1d(64)
        self.bn2 = nn.BatchNorm1d(128)
        self.bn3 = nn.BatchNorm1d(128)
        self.bn4 = nn.BatchNorm1d(512)
        self.bn5 = nn.BatchNorm1d(2048)
        self.fstn = STNkd(k=128)
        self.fc1 = nn.Linear(2048, 256)
        self.fc2 = nn.Linear(256, 256)
        self.fc3 = nn.Linear(256, cat_num)
        self.dropout = nn.Dropout(p=0.3)
        self.bnc1 = nn.BatchNorm1d(256)
        self.bnc2 = nn.BatchNorm1d(256)
        self.convs1 = nn.Conv1d(4944, 256, 1)
        self.convs2 = nn.Conv1d(256, 256, 1)
        self.convs3 = nn.Conv1d(256, 128, 1)
        self.convs4 = nn.Conv1d(128, part_num, 1)
        self.bns1 = nn.BatchNorm1d(256)
        self.bns2 = nn.BatchNorm1d(256)
        self.bns3 = nn.BatchNorm1d(128)
        self._folded = FoldedLayers()

    def forward(self, point_cloud, label, dropout_mask=None):
        if autograd_path(self, point_cloud, label):
            from ..train import pointnet_densecls_train

            return pointnet_densecls_train(self, point_cloud, label, dropout_mask)
        B, _, N = point_cloud.shape
        L = self._folded.get(
            [self.conv1, self.conv2, self.conv3, self.conv4, self.conv5, self.fc1, self.fc2, self.fc3,
             self.convs1, self.convs2, self.convs3, self.convs4],
            [self.bn1, self.bn2, self.bn3, self.bn4, self.bn5, self.bnc1, self.bnc2, None,
             self.bns1, self.bns2, self.bns3, None])
        x = _point_rows(point_cloud)
        x = ops.bmm_points(x, self.stn.transform_rows(x))
        # per-point features out1..out5 are written side by side: they are the per-point half of `concat`
        widths = [64, 128, 128, 512, 2048]
        cat = torch.empty((B * N, sum(widths)), dtype=torch.float32, device=x.device)
        cols = [0, 64, 192, 320, 832, 2880]
        out1 = ops.linear(x.view(B * N, 3), *L[0], relu=True, out=cat[:, cols[0]:cols[1]])
        out2 = ops.linear(out1, *L[1], relu=True, out=cat[:, cols[1]:cols[2]])
        out3 = ops.linear(out2, *L[2], relu=True, out=cat[:, cols[2]:cols[3]])
        trans_feat = self.fstn.transform_rows(out3.view(B, N, 128))
        net_t = ops.bmm_points(out3.view(B, N, 128), trans_feat).view(B * N, 128)
        out4 = ops.linear(net_t, *L[3], relu=True, out=cat[:, cols[3]:cols[4]])
        out5 = ops.linear(out4, *L[4], relu=False, out=cat[:, cols[4]:cols[5]])
        out_max = ops.group_max(out5, N)                                          # [B,2048]
        net = ops.linear(out_max, *L[5], relu=True)
        net = ops.linear(net, *L[6], relu=True)
        net = ops.linear(net, *L[7], relu=False)                                  # [B,cat_num] (no log_softmax in the reference)
        # segmentation: convs1 over cat([out_max, label] expanded, out1..out5): global half -> per-cloud bias
        ws1, bs1 = L[8]
        glob = torch.cat([out_max, label.to(out_max.dtype)], 1)                   # [B,2064]
        cloud_bias = ops.linear(glob, ws1[:, :2064].contiguous(), bs1, relu=False)
        h = ops.linear_cloud_bias(cat.view(B, N, -1), ws1[:, 2064:].contiguous(), cloud_bias, relu=True).view(B * N, 256)
        h = ops.linear(h, *L[9], relu=True)
        h = ops.linear(h, *L[10], relu=True)
        seg = ops.log_softmax(ops.linear(h, *L[11], relu=False)).view(B, N, self.part_num)
        return net, seg, trans_feat


def feature_transform_reguliarzer(trans: torch.Tensor) -> torch.Tensor:
    """Reference pointnet.py:257-263 (training-side regulariser; tiny, plain torch):
    mean Frobenius norm of trans @ (trans^T - I)."""
    d = trans.shape[1]
    eye = torch.eye(d, device=trans.device, dtype=trans.dtype)[None]
    return torch.mean(torch.norm(torch.bmm(trans, trans.transpose(2, 1) - eye), dim=(1, 2)))


class PointNetLoss(nn.Module):
    """Reference pointnet.py:266-278."""

    def __init__(self, weight=1, mat_diff_loss_scale=0.001):
        super().__init__()
        self.mat_diff_loss_scale = mat_diff_loss_scale
        self.weight = weight

    def forward(self, labels_pred, label, seg_pred, seg, trans_feat):
        seg_loss = nn.functional.nll_loss(seg_pred, seg)
        label_loss = nn.functional.nll_loss(labels_pred, label)
        reg = feature_transform_reguliarzer(trans_feat)
        total = self.weight * seg_loss + (1 - self.weight) * label_loss + reg * self.mat_diff_loss_scale
        return total, seg_loss, label_loss
