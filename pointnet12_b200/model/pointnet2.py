"""B200-native drop-in for the reference's model/pointnet2.py (PointNet++ networks).

Class names, constructor arguments, submodule names (hence state_dict keys) and return values follow
the reference; `checkpoints/pointnet2-inview-0.55884-0001.pth` loads with strict=True.  The five
networks differ only in their level tables, so they are built from specs; the heads
(conv/linear + BatchNorm + ReLU, log_softmax) run through the same C-ABI kernels as the blocks, on
point-major rows, so a segmentation output [B, N, k] is produced directly in its final layout
(the reference permutes at the end, pointnet2.py:175).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from .pointnet_util import (FoldedLayers, PointNetFeaturePropagation, PointNetSetAbstraction,
                            PointNetSetAbstractionMsg, _eval_only, autograd_path, draw_fps_starts, farthest_point_sample)


def _ssg(npoint, radius, nsample, in_channel, mlp):
    return PointNetSetAbstraction(npoint, radius, nsample, in_channel, mlp, False)


def _msg(npoint, radii, nsamples, in_channel, mlps):
    return PointNetSetAbstractionMsg(npoint, radii, nsamples, in_channel, mlps)


def _all(in_channel, mlp):
    return PointNetSetAbstraction(None, None, None, in_channel, mlp, True)


def _fp(in_channel, mlp):
    return PointNetFeaturePropagation(in_channel, mlp)


class _Net(nn.Module):
    """Registers named levels in order and owns the folded head weights."""

    def _levels(self, **named):
        for name, module in named.items():
            setattr(self, name, module)
        self._head = FoldedLayers()

    def _cls_fc(self, dropout: float, classes: int):
        """fc1-bn1-drop1-fc2-bn2-drop2-fc3 of the classification nets (pointnet2.py:28-35)."""
        self.fc1, self.bn1, self.drop1 = nn.Linear(1024, 512), nn.BatchNorm1d(512), nn.Dropout(dropout)
        self.fc2, self.bn2, self.drop2 = nn.Linear(512, 256), nn.BatchNorm1d(256), nn.Dropout(dropout)
        self.fc3 = nn.Linear(256, classes)

    def _seg_convs(self, classes: int):
        """conv1-bn1-drop1-conv2 of the segmentation nets (pointnet2.py:154-157)."""
        self.conv1, self.bn1, self.drop1 = nn.Conv1d(128, 128, 1), nn.BatchNorm1d(128), nn.Dropout(0.5)
        self.conv2 = nn.Conv1d(128, classes, 1)

    # -- heads (eval: dropout is the identity) ---------------------------------------------------
    def _cls_head(self, global_feat: torch.Tensor) -> torch.Tensor:
        # three single-layer tensor-core chains (a [B, 1024] matrix is one row tile: each launch is sliced over the output
        # channels, so the 1024 x 512 weights are read by 16 CTAs instead of one SIMT tile marching through them: 200 -> 45 us at B=32)
        per_layer = self._head.layer_chains([self.fc1, self.fc2, self.fc3], [self.bn1, self.bn2, None], [True, True, False])
        if per_layer is not None:
            x = ops.mlp_rows_tc(per_layer[0], global_feat)
            x = ops.mlp_rows_tc(per_layer[1], x)
            return ops.mlp_rows_tc(per_layer[2], x, ops.OUT_LOG_SOFTMAX)
        (w1, b1), (w2, b2), (w3, b3) = self._head.get([self.fc1, self.fc2, self.fc3], [self.bn1, self.bn2, None])
        x = ops.linear(global_feat, w1, b1, relu=True)
        x = ops.linear(x, w2, b2, relu=True)
        return ops.log_softmax(ops.linear(x, w3, b3, relu=False))

    def _seg_head(self, l0_points: torch.Tensor):
        """[B,128,N] -> (log_probs [B,N,k], feat [B,128,N])."""
        B, C, N = l0_points.shape
        (w1, b1), (w2, b2) = self._head.get([self.conv1, self.conv2], [self.bn1, None])
        rows = l0_points.permute(0, 2, 1).reshape(B * N, C)        # a view when it comes from our own blocks
        feat = ops.linear(rows, w1, b1, relu=True)
        logp = ops.log_softmax(ops.linear(feat, w2, b2, relu=False))
        return logp.view(B, N, -1), feat.view(B, N, -1).permute(0, 2, 1)

    ENCODER = ("sa1", "sa2", "sa3")     # the set-abstraction levels `_encode` runs (PointNet2SemSeg has its own forward)

    def fps_level_sizes(self, n_points: int):
        """Cloud sizes the sampling levels of this net draw their FPS start index from, in call order (pointnet_util.py:75):
        what a CUDA-graph runner must draw on the host for every batch (runtime.GraphedModule)."""
        sizes, n = [], int(n_points)
        for name in self.ENCODER:
            lvl = getattr(self, name)
            if not getattr(lvl, "group_all", False):
                sizes.append(n)
                n = lvl.npoint
        return sizes

    def _encode(self, names, xyz, points, fps_starts=None):
        """Run set-abstraction levels in order; returns the per-level (xyz, features) lists.
        The FPS start indices of all sampling levels are drawn up front (same generator, same order as the
        reference's per-level draws) so that they reach the device in one asynchronous copy; `fps_starts` (extension):
        the caller has drawn them already ([B] int64 device tensors, one per sampling level)."""
        ops._need_cuda(xyz, "xyz")
        levels = [getattr(self, name) for name in names]
        sizes, n = [], xyz.shape[2]
        for lvl in levels:
            if not getattr(lvl, "group_all", False):
                sizes.append(n)
                n = lvl.npoint
        starts = iter(fps_starts if fps_starts is not None else draw_fps_starts(xyz.shape[0], sizes, xyz.device))
        xs, fs = [xyz], [points]
        for lvl in levels:
            if getattr(lvl, "group_all", False):
                x, f = lvl(xs[-1], fs[-1])
            else:
                x, f = lvl(xs[-1], fs[-1], start_idx=next(starts))
            xs.append(x)
            fs.append(f)
        return xs, fs


class PointNet2ClsMsg(_Net):
    """Reference pointnet2.py:7-47.  forward(xyz [B,3,N]) -> (log_probs [B,40], l3_points [B,1024,1])."""

    def __init__(self):
        super().__init__()
        self._levels(
            sa1=_msg(512, [0.1, 0.2, 0.4], [16, 32, 128], 0, [[32, 32, 64], [64, 64, 128], [64, 96, 128]]),
            sa2=_msg(128, [0.2, 0.4, 0.8], [32, 64, 128], 320, [[64, 64, 128], [128, 128, 256], [128, 128, 256]]),
            sa3=_all(640 + 3, [256, 512, 1024]))
        self._cls_fc(0.4, 40)

    def forward(self, xyz, dropout_masks=None, fps_starts=None):
        _, fs = self._encode(("sa1", "sa2", "sa3"), xyz, None, fps_starts)
        if autograd_path(self, xyz):          # autograd blocks (pointnet12_b200/train.py)
            from ..train import cls_head_train

            return cls_head_train(self, fs[3].reshape(xyz.shape[0], 1024), dropout_masks), fs[3]
        return self._cls_head(fs[3].reshape(xyz.shape[0], 1024)), fs[3]


class PointNet2ClsSsg(_Net):
    """Reference pointnet2.py:49-73.  forward(xyz [B,3,N]) -> log_probs [B,40]."""

    def __init__(self):
        super().__init__()
        self._levels(sa1=_ssg(512, 0.2, 32, 3, [64, 64, 128]),
                     sa2=_ssg(128, 0.4, 64, 128 + 3, [128, 128, 256]),
                     sa3=_all(256 + 3, [256, 512, 1024]))
        self._cls_fc(0.4, 40)

    def forward(self, xyz, dropout_masks=None, fps_starts=None):
        _, fs = self._encode(("sa1", "sa2", "sa3"), xyz, None, fps_starts)
        if autograd_path(self, xyz):
            from ..train import cls_head_train

            return cls_head_train(self, fs[3].reshape(xyz.shape[0], 1024), dropout_masks)
        return self._cls_head(fs[3].reshape(xyz.shape[0], 1024))


class PointNet2PartSegSsg(_Net):
    """Reference pointnet2.py:75-104.  forward(xyz [B,3,N]) -> (log_probs [B,N,k], feat [B,128,N])."""

    def __init__(self, num_classes):
        super().__init__()
        self._levels(sa1=_ssg(512, 0.2, 64, 3, [64, 64, 128]),
                     sa2=_ssg(128, 0.4, 64, 128 + 3, [128, 128, 256]),
                     sa3=_all(256 + 3, [256, 512, 1024]),
                     fp3=_fp(1280, [256, 256]), fp2=_fp(384, [256, 128]), fp1=_fp(128, [128, 128, 128]))
        self._seg_convs(num_classes)

    def forward(self, xyz, dropout_mask=None, fps_starts=None):
        xs, fs = self._encode(("sa1", "sa2", "sa3"), xyz, None, fps_starts)
        f2 = self.fp3(xs[2], xs[3], fs[2], fs[3])
        f1 = self.fp2(xs[1], xs[2], fs[1], f2)
        if autograd_path(self, xyz):
            from ..train import seg_head_train

            return seg_head_train(self, self.fp1(xyz, xs[1], None, f1), dropout_mask)
        return self._seg_head(self.fp1(xyz, xs[1], None, f1))


class PointNet2PartSegMsg_one_hot(_Net):
    """Reference pointnet2.py:106-139.  forward(xyz, norm_plt, cls_label [B,16]) -> log_probs [B,N,k]."""

    def __init__(self, num_classes):
        super().__init__()
        self._levels(
            sa1=_msg(512, [0.1, 0.2, 0.4], [32, 64, 128], 0 + 3, [[32, 32, 64], [64, 64, 128], [64, 96, 128]]),
            sa2=_msg(128, [0.4, 0.8], [64, 128], 128 + 128 + 64, [[128, 128, 256], [128, 196, 256]]),
            sa3=_all(512 + 3, [256, 512, 1024]),
            fp3=_fp(1536, [256, 256]), fp2=_fp(576, [256, 128]), fp1=_fp(150, [128, 128]))
        self._seg_convs(num_classes)

    def forward(self, xyz, norm_plt, cls_label, dropout_mask=None, fps_starts=None):
        B, _, N = xyz.shape
        xs, fs = self._encode(("sa1", "sa2", "sa3"), xyz, norm_plt, fps_starts)
        f2 = self.fp3(xs[2], xs[3], fs[2], fs[3])
        f1 = self.fp2(xs[1], xs[2], fs[1], f2)
        skip = torch.cat([cls_label.view(B, 16, 1).expand(B, 16, N), xyz, norm_plt], 1)   # host-side glue [B,22,N]
        if autograd_path(self, xyz, norm_plt, cls_label):
            from ..train import seg_head_train

            return seg_head_train(self, self.fp1(xyz, xs[1], skip, f1), dropout_mask)[0]
        return self._seg_head(self.fp1(xyz, xs[1], skip, f1))[0]


class PointNet2SemSeg(_Net):
    """Reference pointnet2.py:141-176.  forward(points [B, 3+feature_dims, N]) -> log_probs [B, N, num_classes]."""

    def __init__(self, num_classes, feature_dims=3):
        super().__init__()
        self.feature_dims = feature_dims
        self._levels(sa1=_ssg(1024, 0.1, 32, feature_dims + 3, [32, 32, 64]),
                     sa2=_ssg(256, 0.2, 32, 64 + 3, [64, 64, 128]),
                     sa3=_ssg(64, 0.4, 32, 128 + 3, [128, 128, 256]),
                     sa4=_ssg(16, 0.8, 32, 256 + 3, [256, 256, 512]),
                     fp4=_fp(768, [256, 256]), fp3=_fp(384, [256, 256]),
                     fp2=_fp(320, [256, 128]), fp1=_fp(128, [128, 128, 128]))
        self._seg_convs(num_classes)

    def forward(self, points, fps_starts=None, host_out=None):
        """points [B, 3+feature_dims, N] -> log-probabilities [B, N, num_classes].
        `host_out` (extension): a pinned host tensor [B, N, num_classes]; the last level then runs in batch slices
        and each slice starts its device-to-host copy on a copy stream as soon as it is computed, so the
        transfer of the first clouds overlaps the computation of the last ones.  The copies are ordered before
        anything issued later on the current stream.
        `fps_starts` (extension): the four FPS start-index tensors ([B] int64 on the device) when the caller has
        drawn them already (CUDA-graph replay); by default they are drawn like the reference draws them.

        Schedule (DESIGN.md section 6): everything that depends on xyz only -- bucket build, the level-1 ball query
        (answered on the idle SMs WHILE level-1 sampling runs), sampling / grouping of levels 2-4, the 3-NN searches --
        runs on internal side streams beside the critical path FPS1 -> sa1..sa4 -> fp4..fp1; fp1 and the
        segmentation head run as one tensor-core chain whose first layer is folded into fp2's chain."""
        if autograd_path(self, points):
            from ..train import semseg_forward_train        # SURVEY 8 f-1: the autograd blocks
            if host_out is not None and torch.is_grad_enabled() and points.requires_grad:
                raise ValueError("PointNet2SemSeg: host_out cannot be combined with an input that requires a gradient")
            return semseg_forward_train(self, points, fps_starts)
        ops._need_cuda(points, "points")
        B, _, N = points.shape
        pm = points.permute(0, 2, 1)
        x0, f0 = pm[:, :, :3], (pm[:, :, 3:] if points.shape[1] > 3 else None)
        sa = [self.sa1, self.sa2, self.sa3, self.sa4]
        fp = [self.fp1, self.fp2, self.fp3, self.fp4]              # fp[i] upsamples level i+1 -> level i
        if fps_starts is None:
            fps_starts = draw_fps_starts(B, [N] + [m.npoint for m in sa[:-1]], points.device)
        # Streams: the caller's stream only brackets the forward.  `main` (high priority) carries the critical path
        # FPS1 -> ball query 1 -> SA chains -> FP chains; `geo` (high priority) the sampling / grouping of levels 2-4, which
        # the SA chains wait for; the 3-NN searches are only needed by the FP chains at the end, so they run at default
        # (= lower) priority on two more streams and fill whatever the critical path leaves idle instead of competing
        # with it: the big one (24000 x 1024 per cloud, for fp1) on its own stream, released after sa2.
        user = torch.cuda.current_stream(points.device)
        main, geo, nn_small, nn_big, feed, ahead = self._side_streams(points.device)
        begin = torch.cuda.Event()
        begin.record(user)
        main.wait_event(begin)

        # the level-1 ball-query buckets depend on xyz only: built beside the level-1 sampling.  If sampling leaves
        # enough SMs idle, the level-1 ball query itself runs there WHILE sampling runs, fed centroid by centroid
        # (ops.ball_query_stream); the regular query afterwards only fills in what the streamed one did not finish.
        grid1, streamed = None, None
        S1, K1 = sa[0].npoint, sa[0].nsample
        fps1_cfg = ops.fps1_config()
        if N >= ops.GRID_MIN_POINTS:
            if ops.stream_ball_query() and N <= 32768:
                fps_ctas, fps_smem = ops.fps_launch_info(B, N, S1, fps1_cfg)
                sms = torch.cuda.get_device_properties(points.device).multi_processor_count
                ctas = ops.stream_ball_ctas(sms - fps_ctas, B)
                if ctas >= max(B, ops.STREAM_BALL_MIN_FREE_SMS if not ops.stream_ball_share() else B):
                    streamed = {"progress": torch.zeros((B, S1), dtype=torch.int64, device=points.device),
                                "done": torch.zeros((B, S1), dtype=torch.int32, device=points.device),
                                "out": torch.empty((B, S1, K1), dtype=torch.int64, device=points.device)}
                    begin.record(user)                       # (again: the zero fills come first)
                    main.wait_event(begin)
        sorted_cfg = None
        if ops.GRID_MIN_POINTS <= N <= ops.FPS_SORTED_MAX_POINTS and streamed is None:
            sorted_cfg = ops.fps1_sorted()
        if sorted_cfg is None:
            with torch.cuda.stream(main):
                # level-1 sampling (the long serial kernel), issued FIRST: its clusters need whole groups of free SMs, so the
                # kernels that run beside it must find it already in place
                fps1 = self._whatif("fps1", lambda: ops.fps(x0, S1, ops._i64(fps_starts[0], "start_idx"),
                                                            progress=streamed["progress"] if streamed else None, config=fps1_cfg))
        if N >= ops.GRID_MIN_POINTS:
            with torch.cuda.stream(geo):
                geo.wait_event(begin)
                grid1 = ops.ball_grid(x0, sa[0].radius)
                grid_ready = torch.cuda.Event()
                grid_ready.record(geo)
            if streamed is not None:
                with torch.cuda.stream(feed):                # its own stream: `geo` must be free for level 2 when sampling ends
                    feed.wait_event(grid_ready)
                    ops.ball_query_stream(sa[0].radius, K1, x0, grid1, streamed["progress"], streamed["done"], streamed["out"],
                                          ctas, 0 if ops.stream_ball_share() else 227 * 1024 - fps_smem + 1024)
                    streamed["finished"] = torch.cuda.Event()
                    streamed["finished"].record(feed)
        if sorted_cfg is not None:
            with torch.cuda.stream(main):
                # throughput mode (several batches in flight): the bucket-pruned sampling kernel reads the cloud in the cell
                # order of the ball-query buckets, so it starts after the bucket build (~35 us) and occupies fewer SMs
                main.wait_event(grid_ready)
                fps1 = self._whatif("fps1", lambda: ops.fps_sorted(x0, grid1, S1, ops._i64(fps_starts[0], "start_idx"),
                                                                   config=sorted_cfg))

        with torch.cuda.stream(main):
            x1 = ops.index_points(x0, fps1)
            fork = torch.cuda.Event()
            fork.record(main)
        xs, balls, nns, ready = [x0, x1], [None] * 4, [None] * 4, [None] * 4
        with torch.cuda.stream(geo):                               # sampling / grouping of levels 2..4, back to back
            geo.wait_event(fork)
            for i in (1, 2, 3):
                nx, balls[i] = sa[i].geometry(xs[i], fps_starts[i])
                xs.append(nx)
                ready[i] = torch.cuda.Event()
                ready[i].record(geo)
        with torch.cuda.stream(nn_small):                          # 3-NN of levels 2..4 (inputs: the level centroids)
            for i in (3, 2, 1):                                    # fp4 is the first to need its neighbours
                nn_small.wait_event(ready[i])
                nns[i] = fp[i].geometry(xs[i], xs[i + 1])
            done_small = torch.cuda.Event()
            done_small.record(nn_small)

        with torch.cuda.stream(main):
            # feature path
            if grid1 is not None:
                main.wait_event(grid_ready)
            if streamed is not None:
                main.wait_event(streamed["finished"])
                balls[0] = ops.ball_query(sa[0].radius, K1, x0, x1, grid=grid1, done=streamed["done"], out=streamed["out"])
            else:
                balls[0] = self._whatif("bq1", lambda: ops.ball_query(sa[0].radius, K1, x0, x1, grid=grid1))
            # fp1 and the segmentation head (conv1-bn1-relu, conv2, log_softmax) run as ONE chain: 70 % of the FLOPs.  Its
            # first layer acts on the 1024 coarse points (interpolation commutes with it): it is appended to fp2's chain,
            # whose output rows are exactly those points, so fp2 hands over z = W1 * l1_features + b1 directly.
            head = (self._head, [self.conv1, self.conv2], [self.bn1, None], [True, False], ops.OUT_LOG_SOFTMAX)
            # (only when fp1 really upsamples: `features` folds its first layer under the same N > S condition; with
            # N <= sa1.npoint the fine level runs the complete chain and must be handed the plain fp2 features)
            first = fp[0].first_layer_spec(head) if (ops.mlp_mode() == "bf16x3" and N > S1) else None
            fp2z = None
            if first is not None:
                fp2z = (self.__dict__.setdefault("_fp2z", FoldedLayers()), [first[0]], [first[1]], [False], ops.OUT_ROWS)
            skipped = [None] * 4

            def skip_ahead(i):
                # the skip half of fp[i]'s first layer depends on the encoder feature fs[i] only: computed on a side
                # stream as soon as that level exists, while the encoder goes on
                made = torch.cuda.Event()
                made.record(main)
                with torch.cuda.stream(ahead):
                    ahead.wait_event(made)
                    if fp[i].skip_ahead(fs[i], fp2z if i == 1 else None):
                        skipped[i] = torch.cuda.Event()
                        skipped[i].record(ahead)

            # sa1 / sa2 run one persistent CTA per SM while level 2-4 sampling holds a few SMs: leave those out
            ops.set_reserved_sms(ops.fps_launch_info(B, S1, sa[1].npoint)[0] if ops.reserve_level2_sms() else 0)
            try:
                fs = [f0, self._whatif("sa1", lambda: sa[0].features(x0, f0, x1, balls[0]))]
                main.wait_event(ready[1])
                fs.append(self._whatif("sa2", lambda: sa[1].features(xs[1], fs[1], xs[2], balls[1])))
            finally:
                ops.set_reserved_sms(0)
            skip_ahead(1)
            skip_ahead(2)
            for i in (1, 2, 3):
                if i > 1:
                    main.wait_event(ready[i])
                    fs.append(sa[i].features(xs[i], fs[i], xs[i + 1], balls[i]))
                    if i == 2:
                        skip_ahead(3)
                if i == 1:
                    # fp1's 3-NN search (24000 x 1024 per cloud) fills the GPU with long-lived CTAs, which stream
                    # priorities cannot displace: it is released only now, when the wide kernels of the critical path
                    # (ball query 1, sa1, sa2) are through and the small levels leave most SMs idle
                    wide_done = torch.cuda.Event()
                    wide_done.record(main)
                    with torch.cuda.stream(nn_big):
                        nn_big.wait_event(wide_done)
                        if grid1 is not None:
                            nn_big.wait_event(grid_ready)
                        nns[0] = self._whatif("nn1", lambda: fp[0].geometry(x0, x1, order=grid1, background=ops.nn1_background()))
                        done_big = torch.cuda.Event()
                        done_big.record(nn_big)
            main.wait_event(done_small)
            up = fs[4]
            for i in (3, 2):
                if skipped[i] is not None:
                    main.wait_event(skipped[i])
                up = fp[i].features(fs[i], up, *nns[i])
            if skipped[1] is not None:
                main.wait_event(skipped[1])
            if fp2z is not None:
                up = fp[1].features(fs[1], up, *nns[1], head=fp2z)       # = z
                fp[0].adopt_folded(up, head)
            else:
                up = fp[1].features(fs[1], up, *nns[1])
            main.wait_event(done_big)
            if host_out is None or ops.mlp_mode() != "bf16x3":
                logp = self._whatif("fp1", lambda: fp[0].features(None, up, *nns[0], head=head,
                                                                  order=grid1 if ops.FP1_BUCKET_ORDER else None))
                if host_out is not None:
                    host_out.copy_(logp, non_blocking=True)
            else:
                logp = torch.empty((B, N, self.conv2.out_channels), dtype=torch.float32, device=points.device)
                copier = self._copy_stream(points.device)
                # batch slices: the device-to-host copy (the slower side: 14.6 MB at ~55 GB/s vs 134 us of compute at C2)
                # should start as early as possible, so the slices are small -- one or two clouds
                nslice = min(B, ops.host_out_slices())
                cuts = [round(i * B / nslice) for i in range(nslice + 1)]
                for b0, b1 in zip(cuts[:-1], cuts[1:]):
                    if b0 == b1:
                        continue
                    fp[0].features(None, up, *nns[0], head=head, order=grid1 if ops.FP1_BUCKET_ORDER else None, out=logp, clouds=(b0, b1))
                    part = torch.cuda.Event()
                    part.record(main)
                    with torch.cuda.stream(copier):
                        copier.wait_event(part)
                        host_out[b0:b1].copy_(logp[b0:b1], non_blocking=True)
                main.wait_stream(copier)
        user.wait_stream(main)
        if not torch.cuda.is_current_stream_capturing():
            logp.record_stream(user)       # allocated on `main`, handed to the caller's stream
        return logp

    def _whatif(self, name, fn):
        """Analysis hook (tools/pipeline_sweep.py --whatif): with PN12_WHATIF=name[,name] the named kernel group is launched
        once and its (stale) result reused afterwards -- the step time without that group bounds what optimising it can buy.
        Results are wrong in that mode; unset (the default) this is just fn()."""
        import os

        skip = os.environ.get("PN12_WHATIF", "")
        if not skip or name not in skip.split(","):
            return fn()
        cache = self.__dict__.setdefault("_whatif_cache", {})
        if name not in cache:
            cache[name] = fn()
        return cache[name]

    def _copy_stream(self, device):
        key = ("copy", torch.device(device).index)
        streams = self.__dict__.setdefault("_streams", {})
        if key not in streams:
            streams[key] = torch.cuda.Stream(device)
        return streams[key]

    def _side_streams(self, device):
        key = torch.device(device).index
        streams = self.__dict__.setdefault("_streams", {})
        if key not in streams:
            rng = torch.cuda.Stream.priority_range()             # lower number = higher priority; 0 = default = lowest
            lo, hi = max(rng), min(rng)
            streams[key] = (torch.cuda.Stream(device, priority=hi), torch.cuda.Stream(device, priority=hi),
                            torch.cuda.Stream(device, priority=lo), torch.cuda.Stream(device, priority=lo),
                            torch.cuda.Stream(device, priority=hi), torch.cuda.Stream(device, priority=lo))
        return streams[key]
