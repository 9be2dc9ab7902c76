"""Every schedule switch of PointNet2SemSeg.forward (eval) and of the training step, against the default schedule and the
oracles.

The eval forward spreads its work over seven streams, and about a dozen switches choose which kernels run and in what
order: `ops.options(...)` keys, `PN12_*` environment variables read per forward, and module constants of `ops` / `train`
read at import.  The kernels behind each branch are tested on their own elsewhere; here each branch runs INSIDE the network,
where stream order, event waits and buffer reuse matter.

- Each case switches one schedule, wraps the ops its branch calls in counting spies and asserts that the branch ran: a
  switch that is silently ignored must not pass.
- Switches that only change which kernel or grid computes an exact quantity (the level-1 sampling kernel and launch shape,
  the streamed / plain / tail / shared / CTA-count variants of the level-1 ball query, the grid of fp1's 3-NN search, the
  SMs sa1 / sa2 leave free, the order fp1 walks the fine points in, the batch slices of the host output) give log-
  probabilities torch.equal to the default schedule's.  The skip half of an FP level's first layer computed ahead changes
  the order of that layer's sum: within 1e-5 of the default.
- At B = 2, N = 8192 every schedule is also held against the C oracle (oracle.pointnet2_semseg), which anchors the
  bit-identity chain; at the C2 size (B = 8, N = 24000, whose default is pinned to golden vectors) and at the B / N edges of
  the branches, bit-identity with the default only.
- The training switches (unfused BatchNorm, per-GEMM weight packing, BatchNorm-backward reductions in the GEMM epilogue,
  tensor-core weight gradients for every layer) each run one step on the shipped checkpoint against the float64 training
  oracle and the reference's own step.

`test_every_switch_is_covered` (no GPU) fails when a `PN12_*` switch appears in the package that this file neither covers
nor exempts with a reason.
"""
import contextlib
import glob
import os
import re

import numpy as np
import pytest
import torch

from pointnet12_b200 import synthetic as syn
from test_gpu_parity import LOGP_TOL, rel_err, starts
from test_train_oracle import check_step_against_golden, rl2, step_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# module constants the switches of this file set, with their defaults (the value they take with no PN12_* variable set)
DEFAULT_CONSTANTS = {
    ("ops", "FP_SKIP_AHEAD"): False,
    ("ops", "FP1_BUCKET_ORDER"): False,
    ("ops", "HOST_OUT_SLICES"): 8,
    ("ops", "STREAM_BALL_TAIL"): 0,
    ("ops", "GRAD_TC_MIN_TILE"): 1024,
    ("train", "FUSED_BN"): True,
    ("train", "PACK_ONCE"): True,
    ("train", "FUSED_BN_BWD"): False,
}


@pytest.fixture(autouse=True)
def isolated(monkeypatch):
    """No PN12_* variable (PN12_WHATIF above all: it reuses stale results by design) and every module constant at its
    default; a case then switches one schedule through this monkeypatch, which undoes it afterwards."""
    from pointnet12_b200 import ops, train

    for k in list(os.environ):
        if k.startswith("PN12_"):
            monkeypatch.delenv(k)
    mods = {"ops": ops, "train": train}
    for (mod, name), value in DEFAULT_CONSTANTS.items():
        monkeypatch.setattr(mods[mod], name, value)
    return monkeypatch


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (run with -m 'not gpu' on CPU boxes)")
    return torch.device("cuda", 0)


def _net(dev, ckpt_path):
    from pointnet12_b200.model.utils import load_pointnet

    return load_pointnet("pointnet2", 19, ckpt_path, device=dev)


class Spy:
    """Wraps owner.name (a module function or a class's method); the wrapped function still runs.  calls: (args, kwargs, result)."""

    def __init__(self, mp, owner, name):
        self.calls = []
        real = getattr(owner, name)

        def spy(*args, **kwargs):
            out = real(*args, **kwargs)
            self.calls.append((args, kwargs, out))
            return out

        mp.setattr(owner, name, spy)


class Trace:
    """What the level-1 stage, fp1 and the head of one forward did, read from spies on the ops they call."""

    def __init__(self, mp):
        from pointnet12_b200 import ops
        from pointnet12_b200.model.pointnet_util import PointNetFeaturePropagation

        self.spies = {n: Spy(mp, ops, n) for n in ("fps", "fps_sorted", "ball_query_stream", "ball_query", "three_nn",
                                                   "set_reserved_sms", "fp_mlp_tc")}
        self.spies["skip_ahead"] = Spy(mp, PointNetFeaturePropagation, "skip_ahead")

    def calls(self, name):
        return self.spies[name].calls

    def level1_fps(self, N):
        return [kw.get("config") for a, kw, _ in self.calls("fps") if a[0].shape[1] == N]

    def level1_sorted(self, N):
        return [kw.get("config") for a, kw, _ in self.calls("fps_sorted") if a[0].shape[1] == N]

    def streamed(self):
        """[(done [B, S] int32, ctas, min_smem)] of the streamed level-1 queries."""
        return [(a[5], a[7], a[8]) for a, _, _ in self.calls("ball_query_stream")]

    def level1_query(self, N):
        return [kw for a, kw, _ in self.calls("ball_query") if a[2].shape[1] == N]

    def nn1_background(self, N):
        return [kw.get("background") for a, kw, _ in self.calls("three_nn") if a[0].shape[1] == N]

    def head(self):
        """(kwargs) of the fp1 + head chain launches (log-softmax output)."""
        from pointnet12_b200 import ops

        return [kw for a, kw, _ in self.calls("fp_mlp_tc") if (a[5] if len(a) > 5 else kw.get("out_mode")) == ops.OUT_LOG_SOFTMAX]


def _forward(net, pts, fps_starts, host_out=None):
    with torch.no_grad():
        out = net(pts, fps_starts=fps_starts, host_out=host_out)
    torch.cuda.synchronize()
    return out


_INPUTS, _DEFAULTS, _ORACLE = {}, {}, {}


def _inputs(dev, B, N, config):
    key = (B, N, config)
    if key not in _INPUTS:
        pts = syn.kitti_batch(B, N, config=config)
        st = starts([N, 1024, 256, 64], B, seed=B * 100000 + N)
        _INPUTS[key] = (pts, st, torch.from_numpy(pts).to(dev), [s.to(dev) for s in st])
    return _INPUTS[key]


def _default(dev, ckpt_path, B, N, config):
    """Log-probabilities of the default schedule (computed with no switch set: call it before switching)."""
    key = (B, N, config)
    if key not in _DEFAULTS:
        _, _, x, st = _inputs(dev, B, N, config)
        _DEFAULTS[key] = _forward(_net(dev, ckpt_path), x, st)
    return _DEFAULTS[key]


# ------------------------------------------------------------------------------------------------ schedules
# name -> (switch it on through the monkeypatch, what the trace of a forward at (B, N) must show).  Each check
# holds for shapes where the streamed level-1 query is possible (N <= 32768 and enough free SMs), as at the two sizes
# every schedule runs at; the B / N edges state their own expectations.
def _set(**env):
    def setup(mp, stack):
        for k, v in env.items():
            mp.setenv(k, v)
    return setup


def _const(mod, name, value):
    def setup(mp, stack):
        from pointnet12_b200 import ops, train

        mp.setattr({"ops": ops, "train": train}[mod], name, value)
    return setup


def _options(**kw):
    def setup(mp, stack):
        from pointnet12_b200 import ops

        stack.enter_context(ops.options(**kw))
    return setup


def _check_default(t, B, N):
    assert t.level1_fps(N) == [None] and t.level1_sorted(N) == []
    assert len(t.streamed()) == 1
    assert t.nn1_background(N) == [True]
    assert any(r > 0 for (r,), _, _ in t.calls("set_reserved_sms"))
    assert t.head() and all(kw.get("order") is None for kw in t.head())
    assert not any(out for _, _, out in t.calls("skip_ahead"))


def _check_fps1(t, B, N):
    assert t.level1_fps(N) == [(2, 256, 2)] and len(t.streamed()) == 1


def _check_plain_query(t, B, N):
    assert t.streamed() == [] and t.level1_fps(N) == [None] and t.level1_sorted(N) == []
    (kw,) = t.level1_query(N)
    assert kw.get("done") is None and kw.get("grid") is not None


def _check_sorted(t, B, N):
    assert t.streamed() == [] and t.level1_fps(N) == [] and t.level1_sorted(N) == [(0, 0, 0)]


def _check_sorted_ignored(t, B, N):
    # the bucket-pruned sampling is consulted only when the streamed query does not run
    assert len(t.streamed()) == 1 and t.level1_fps(N) == [None] and t.level1_sorted(N) == []


def _check_share(t, B, N):
    ((_, ctas, min_smem),) = t.streamed()
    assert min_smem == 0 and ctas >= B


def _check_ctas(t, B, N):
    ((_, ctas, _),) = t.streamed()
    assert ctas == 40 // B * B


def _check_tail(t, B, N):
    ((done, _, _),) = t.streamed()
    assert done.shape == (B, 1024)
    assert int(done[:, 1024 - 64:].abs().sum()) == 0, "the streamed query answered rows it was told to leave to the follow-up"
    (kw,) = t.level1_query(N)
    assert kw.get("done") is done             # the follow-up query fills in the rest


def _check_nn1_full(t, B, N):
    assert t.nn1_background(N) == [False]


def _check_no_reserve(t, B, N):
    assert t.calls("set_reserved_sms") and all(r == 0 for (r,), _, _ in t.calls("set_reserved_sms"))


def _check_bucket_order(t, B, N):
    assert t.head() and all(kw.get("order") is not None for kw in t.head())


def _check_skip_ahead(t, B, N):
    made = [(a[0], a[2] if len(a) > 2 else kw.get("head")) for a, kw, out in t.calls("skip_ahead") if out]
    assert len(made) == 3, "fp4 / fp3 / fp2 skip halves computed ahead"
    assert sum(head is not None for _, head in made) == 1, "fp2's skip half folded into fp2z"
    assert sum(kw.get("residual") is not None for _, kw, _ in t.calls("fp_mlp_tc")) == 3, "every term ahead consumed"


SCHEDULES = {
    "default": (lambda mp, stack: None, _check_default),
    "fps1_shape_env": (_set(PN12_FPS1="2,256,2"), _check_fps1),
    "fps1_shape_option": (_options(fps1_config=(2, 256, 2)), _check_fps1),
    "plain_query_env": (_set(PN12_STREAM_BALL="0"), _check_plain_query),
    "plain_query_option": (_options(stream_ball=False), _check_plain_query),
    "sorted_env": (_set(PN12_STREAM_BALL="0", PN12_FPS1_SORTED="0,0,0"), _check_sorted),
    "sorted_option": (_options(stream_ball=False, fps1_sorted=(0, 0, 0)), _check_sorted),
    "sorted_while_streaming": (_options(fps1_sorted=(0, 0, 0)), _check_sorted_ignored),
    "stream_share": (_set(PN12_STREAM_BALL_SHARE="1"), _check_share),
    "stream_ctas": (_set(PN12_STREAM_BALL_CTAS="40"), _check_ctas),
    "stream_tail": (_const("ops", "STREAM_BALL_TAIL", 64), _check_tail),
    "nn1_full_grid_env": (_set(PN12_NN1_BACKGROUND="0"), _check_nn1_full),
    "nn1_full_grid_option": (_options(nn1_background=False), _check_nn1_full),
    "no_reserve_env": (_set(PN12_RESERVE_L2="0"), _check_no_reserve),
    "no_reserve_option": (_options(reserve_level2=False), _check_no_reserve),
    "fp1_bucket_order": (_const("ops", "FP1_BUCKET_ORDER", True), _check_bucket_order),
    "skip_ahead": (_const("ops", "FP_SKIP_AHEAD", True), _check_skip_ahead),
}
INEXACT = {"skip_ahead"}          # changes the order of the first layer's sum: compared within 1e-5, not bit for bit


@pytest.fixture
def switch(isolated):
    """switch(name) turns a schedule of SCHEDULES on until the end of the test and installs the spies -> Trace."""
    with contextlib.ExitStack() as stack:
        def on(name):
            SCHEDULES[name][0](isolated, stack)
            return Trace(isolated)

        yield on


def _compare(name, got, want):
    if name in INEXACT:
        assert rel_err(got, want.cpu().numpy()) < 1e-5
    else:
        assert torch.equal(got, want), "not bit-identical to the default schedule"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCHEDULES))
def test_schedule_vs_oracle(dev, ckpt_path, ckpt_state, switch, name):
    """B = 2, N = 8192: every schedule against the C oracle (LOGP_TOL; labels equal where the oracle's top-2 margin exceeds
    2e-3) and against the default schedule (torch.equal; the skip half ahead within 1e-5)."""
    from oracle import oracle as orc

    B, N, config = 2, 8192, 24
    pts, st, x, st_dev = _inputs(dev, B, N, config)
    if "want" not in _ORACLE:
        _ORACLE["want"] = orc.pointnet2_semseg(ckpt_state, pts, [s.numpy() for s in st])
    want = _ORACLE["want"]
    default = _default(dev, ckpt_path, B, N, config)
    net = _net(dev, ckpt_path)
    t = switch(name)
    got = _forward(net, x, st_dev)
    SCHEDULES[name][1](t, B, N)
    assert rel_err(got, want) < LOGP_TOL
    top2 = np.sort(want, -1)[..., -2:]
    sure = (top2[..., 1] - top2[..., 0]) > 2e-3
    assert np.array_equal(got.argmax(-1).cpu().numpy()[sure], want.argmax(-1)[sure])
    _compare(name, got, default)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCHEDULES))
def test_schedule_at_c2(dev, ckpt_path, switch, name):
    """Config C2 (B = 8, N = 24000): every schedule against the default.  Sampling runs long enough there for the streamed
    query to answer rows beside it (timing-dependent, as test_ball_query_streamed_beside_fps asserts it), unless a tail
    leaves them to the follow-up query."""
    B, N, config = 8, 24000, 2
    _, _, x, st_dev = _inputs(dev, B, N, config)
    default = _default(dev, ckpt_path, B, N, config)
    net = _net(dev, ckpt_path)
    t = switch(name)
    got = _forward(net, x, st_dev)
    SCHEDULES[name][1](t, B, N)
    for done, _, _ in t.streamed():
        if name != "stream_tail":
            assert int(done.sum()) > 0, "the streamed query never ran beside the sampling"
    _compare(name, got, default)


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,name,streamed,sorted_", [
    (16, 24000, "default", False, False),               # 128 sampling CTAs leave 20 SMs: fewer than STREAM_BALL_MIN_FREE_SMS
    (16, 24000, "stream_share", True, False),           # sharing SMs, one CTA per cloud is enough
    (16, 24000, "sorted_while_streaming", False, True),  # the streamed query refused: the bucket-pruned sampling runs
    (2, 32768, "default", True, False),                 # the largest cloud the streamed query takes
    (2, 32768, "plain_query_env", False, False),
    (2, 32769, "default", False, False),
    (2, 32769, "sorted_while_streaming", False, True),
    (2, 49152, "sorted_option", False, True),           # FPS_SORTED_MAX_POINTS
    (2, 49153, "sorted_option", False, False),
])
def test_schedule_at_edge_shapes(dev, ckpt_path, switch, B, N, name, streamed, sorted_):
    """The batch sizes and cloud sizes where the level-1 branches change: the streamed query refused for want of free SMs
    (B = 16 at N = 24000), its largest cloud (32768), the largest cloud of the bucket-pruned sampling (49152).  Which
    sampling kernel and which query ran is asserted; the log-probabilities are torch.equal to the default schedule's."""
    from pointnet12_b200 import ops

    assert ops.FPS_SORTED_MAX_POINTS == 49152
    _, _, x, st_dev = _inputs(dev, B, N, 5)
    default = _default(dev, ckpt_path, B, N, 5)
    net = _net(dev, ckpt_path)
    t = switch(name)
    got = _forward(net, x, st_dev)
    assert len(t.streamed()) == int(streamed)
    assert len(t.level1_sorted(N)) == int(sorted_) and len(t.level1_fps(N)) == 1 - int(sorted_)
    if not streamed:
        (kw,) = t.level1_query(N)
        assert kw.get("done") is None
    if B == 16 and name == "default":
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        print(f"B = 16, N = 24000: {ops.fps_launch_info(B, N, 1024)[0]} sampling CTAs on {sms} SMs")
    _compare(name, got, default)


# ------------------------------------------------------------------------------------------------ output to the host
@pytest.mark.gpu
@pytest.mark.parametrize("B,N,slices,cuts,bucket_order", [
    (8, 24000, None, [(b, b + 1) for b in range(8)], False),          # HOST_OUT_SLICES = 8
    (8, 24000, 2, [(0, 4), (4, 8)], False),
    (8, 24000, 3, [(0, 3), (3, 5), (5, 8)], False),                  # uneven cuts
    (8, 24000, 8, [(b, b + 1) for b in range(8)], False),
    (8, 24000, 11, [(b, b + 1) for b in range(8)], False),           # more slices than clouds
    (8, 24000, "const3", [(0, 3), (3, 5), (5, 8)], False),           # the module constant (PN12_HOST_OUT_SLICES)
    (8, 24000, 3, [(0, 3), (3, 5), (5, 8)], True),                   # with fp1 in bucket order
    (3, 8192, 2, [(0, 2), (2, 3)], False),
])
def test_host_out_slices(dev, ckpt_path, isolated, B, N, slices, cuts, bucket_order):
    """forward(host_out=pinned): the last level runs in batch slices, each copied to the host on the copier stream as soon as
    it is computed.  Every slice is launched once, and the pinned buffer (filled with NaN beforehand) and the returned device
    tensor are torch.equal to the default forward's log-probabilities."""
    from pointnet12_b200 import ops

    _, _, x, st_dev = _inputs(dev, B, N, 3)
    want = _default(dev, ckpt_path, B, N, 3)
    net = _net(dev, ckpt_path)
    opts = {}
    if slices == "const3":
        isolated.setattr(ops, "HOST_OUT_SLICES", 3)
    elif slices is not None:
        opts["host_out_slices"] = slices
    if bucket_order:
        isolated.setattr(ops, "FP1_BUCKET_ORDER", True)
    t = Trace(isolated)
    host = torch.full((B, N, 19), float("nan")).pin_memory()
    with ops.options(**opts):
        got = _forward(net, x, st_dev, host_out=host)
    assert [kw.get("clouds") for kw in t.head()] == cuts
    assert all((kw.get("order") is not None) == bucket_order for kw in t.head())
    assert torch.equal(got, want)
    assert torch.equal(host, want.cpu()), "a slice of the host output was not written"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_host_out_other_precisions(dev, ckpt_path, isolated, precision):
    """host_out with the exact-fp32 engine: the whole last level, then one copy.  With the single-pass bf16 precision the
    tensor-core chains run, so the last level is sliced as in the default precision.  Either way the host buffer is
    torch.equal to the device output of the same precision."""
    from pointnet12_b200 import ops

    B, N = 2, 8192
    _, _, x, st_dev = _inputs(dev, B, N, 3)
    with ops.options(precision=precision):
        want = _forward(_net(dev, ckpt_path), x, st_dev)
        net = _net(dev, ckpt_path)
        t = Trace(isolated)
        host = torch.full((B, N, 19), float("nan")).pin_memory()
        got = _forward(net, x, st_dev, host_out=host)
    if precision == "fp32":
        assert t.head() == []                          # no tensor-core chain, no slices
    else:
        assert [kw.get("clouds") for kw in t.head()] == [(0, 1), (1, 2)]
    assert torch.equal(got, want) and torch.equal(host, want.cpu())


@pytest.mark.gpu
def test_pipelined_host_slices(dev, ckpt_path, isolated):
    """GraphedSemSeg with batches in flight cuts the last level into PN12_PIPE_HOST_SLICES batch slices for a host output
    (1 by default): with 3, every captured forward launches the three slices, and the pinned results of 4 batches are
    torch.equal to the eager forward's."""
    from pointnet12_b200.runtime import GraphedSemSeg

    B, N = 4, 8192
    isolated.setenv("PN12_PIPE_HOST_SLICES", "3")
    net = _net(dev, ckpt_path)
    xs = [syn.kitti_batch(B, N, config=12, first=B * i) for i in range(4)]
    torch.manual_seed(11)
    with torch.no_grad():
        want = [net(torch.from_numpy(p).to(dev)).cpu() for p in xs]
    t = Trace(isolated)
    runner = GraphedSemSeg(net, depth=2)
    torch.manual_seed(11)
    got = runner.run_pipelined([torch.from_numpy(p).pin_memory() for p in xs], to_host=True)
    torch.cuda.synchronize()
    clouds = [kw.get("clouds") for kw in t.head()]
    assert clouds and set(clouds) == {(0, 1), (1, 3), (3, 4)} and len(clouds) % 3 == 0
    assert len(got) == 4 and all((not a.is_cuda) and torch.equal(a, b) for a, b in zip(got, want))


# ------------------------------------------------------------------------------------------------ the training step
def _train_net(dev, ckpt_path):
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg

    net = PointNet2SemSeg(19, feature_dims=1)
    sd = torch.load(ckpt_path, map_location="cpu")
    net.load_state_dict({k[len("module."):]: v for k, v in sd.items()}, strict=True)
    return net.to(dev).train()


def _check_unfused(spies):
    assert spies["train_gemm"].calls == [] and spies["bn_batch_stats"].calls


def _check_per_gemm_packing(spies):
    assert spies["train_gemm"].calls and all(kw.get("packed") is None for _, kw, _ in spies["train_gemm"].calls)


def _check_fused_bn_bwd(spies):
    assert spies["train_gemm_bnbwd"].calls


def _check_tc_weight_grads(spies):
    names = [a[0] for a, _, _ in spies["call"].calls]
    assert "pn_grad_weight_bf16x3" in names and "pn_grad_weight_f32" not in names


TRAIN_SWITCHES = {
    "unfused_bn": (("train", "FUSED_BN", False), _check_unfused),                     # PN12_TRAIN_FUSED=0
    "per_gemm_packing": (("train", "PACK_ONCE", False), _check_per_gemm_packing),     # PN12_TRAIN_PACK_ONCE=0
    "fused_bn_backward": (("train", "FUSED_BN_BWD", True), _check_fused_bn_bwd),      # PN12_TRAIN_FUSED_BWD=1
    "tc_weight_grads": (("ops", "GRAD_TC_MIN_TILE", 0), _check_tc_weight_grads),      # PN12_GRAD_TC_MIN=0
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAIN_SWITCHES))
def test_train_step_switch(dev, golden, ckpt_path, ckpt_state, isolated, name):
    """One training iteration (semseg_forward_train + the fused cross-entropy, backward) on the shipped checkpoint with one
    switch of the step set: against the float64 oracle with the bounds of test_train_step_vs_reference_and_oracle, and
    against the reference's own step inside the same band as the default step."""
    from oracle import train_oracle as tor
    from pointnet12_b200 import _native as nv
    from pointnet12_b200 import ops, train

    (mod, attr, value), check = TRAIN_SWITCHES[name]
    g, pts, target, st, keep = step_inputs(golden)
    if "train" not in _ORACLE:
        _ORACLE["train"] = tor.semseg_train_step(ckpt_state, pts, target, st, keep)
    ref = _ORACLE["train"]
    isolated.setattr({"ops": ops, "train": train}[mod], attr, value)
    spies = {n: Spy(isolated, ops, n) for n in ("train_gemm", "train_gemm_bnbwd", "bn_batch_stats")}
    spies["call"] = Spy(isolated, nv, "call")
    net = _train_net(dev, ckpt_path)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)       # noqa: E731
    logp = train.semseg_forward_train(net, T(pts), fps_starts=[T(s) for s in st], dropout_mask=T(keep.astype(np.uint8)))
    loss = train.cross_entropy(logp, T(target))
    net.zero_grad()
    loss.backward()
    torch.cuda.synchronize()
    check(spies)
    grads = {n: p.grad.detach().cpu().numpy() for n, p in net.named_parameters()}
    buffers = {n: b.cpu().numpy() for n, b in net.named_buffers()}
    lp = logp.detach().cpu().numpy()
    check_step_against_golden(g, loss.item(), lp, grads, buffers, band=3.0)
    assert rl2(lp, ref["logp"]) < 5e-4
    assert rl2(grads["conv2.weight"], ref["grads"]["conv2.weight"]) < 2e-4
    assert rl2(grads["sa1.mlp_convs.0.weight"], ref["grads"]["sa1.mlp_convs.0.weight"]) < 2e-2


# ------------------------------------------------------------------------------------------------ coverage (no GPU)
# every PN12_* name in the package -> the cases of this file that switch it
COVERED = {
    "PN12_FPS1": ["fps1_shape_env"],
    "PN12_STREAM_BALL": ["plain_query_env", "test_schedule_at_edge_shapes"],
    "PN12_FPS1_SORTED": ["sorted_env"],
    "PN12_STREAM_BALL_SHARE": ["stream_share", "test_schedule_at_edge_shapes"],
    "PN12_STREAM_BALL_CTAS": ["stream_ctas"],
    "PN12_STREAM_BALL_TAIL": ["stream_tail"],
    "PN12_NN1_BACKGROUND": ["nn1_full_grid_env"],
    "PN12_RESERVE_L2": ["no_reserve_env"],
    "PN12_FP1_ORDER": ["fp1_bucket_order", "test_host_out_slices"],
    "PN12_FP_SKIP_AHEAD": ["skip_ahead"],
    "PN12_HOST_OUT_SLICES": ["test_host_out_slices"],
    "PN12_PIPE_HOST_SLICES": ["test_pipelined_host_slices"],
    "PN12_TRAIN_FUSED": ["unfused_bn"],
    "PN12_TRAIN_PACK_ONCE": ["per_gemm_packing"],
    "PN12_TRAIN_FUSED_BWD": ["fused_bn_backward"],
    "PN12_GRAD_TC_MIN": ["tc_weight_grads"],
}
EXEMPT = {
    "PN12_WHATIF": "analysis only: reuses stale results of the named kernel groups, wrong by design",
    "PN12_GEMM_DEBUG": "compile-time profiling switch of gemm_tc.cu that disables the MMAs",
    "PN12_NN_BLOCK": "read once per process by three_nn.cu; covered by test_three_nn_block_size_hook in a subprocess",
    "PN12_PIPE_PACE": "host-side pacing of submits, no effect on results; covered by the CPU pacer tests",
    "PN12_FP_FOLD": "import-time constant; the folded and unfolded first FP layer are compared in test_gpu_parity.py",
    "PN12_LAYERWISE_TILES": "import-time constant; layer-wise vs fused chains are compared in test_gpu_parity.py",
    "PN12_MLP": "import-time default of the precision, which every precision test sets through ops.options / set_mlp_mode",
    "PN12_BQ_THRESHOLD": "its extremes are the grid-cells / grid-scan methods of test_ball_query_every_method",
}


def test_every_switch_is_covered():
    """Every PN12_* name in the package's Python and CUDA sources is either switched by a case of this file (COVERED names
    a schedule, a training switch or a test function here) or exempt with a reason; a switch added later without a test
    fails here.  Names that no longer exist in the package must leave the tables too."""
    found = set()
    for ext in ("py", "cu", "cuh"):
        for path in glob.glob(os.path.join(ROOT, "pointnet12_b200", "**", f"*.{ext}"), recursive=True):
            with open(path, encoding="utf-8") as f:
                found |= set(re.findall(r"PN12_[A-Z0-9_]+", f.read()))
    assert found, "no PN12_* switch found: the scan looks in the wrong place"
    assert not set(COVERED) & set(EXEMPT)
    assert sorted(found - set(COVERED) - set(EXEMPT)) == [], "switches with neither a test here nor a reason for exemption"
    assert sorted((set(COVERED) | set(EXEMPT)) - found) == [], "switches listed here that the package no longer has"
    cases = set(SCHEDULES) | set(TRAIN_SWITCHES) | {k for k, v in globals().items() if k.startswith("test_") and callable(v)}
    for name, where in COVERED.items():
        assert where and set(where) <= cases, (name, sorted(set(where) - cases))
    assert all(reason.strip() for reason in EXEMPT.values())
