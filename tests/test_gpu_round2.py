"""GPU parity tests added in round 2 (through the C ABI, against the CPU oracle and reference-generated golden vectors of
oracle/gen_golden_r2.py): the shapes the first review found untested, the batches-in-flight runner, the dynamic tile
scheduler of the resident-weight chains and the per-call launch options that replaced the process-wide setters."""
import threading

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pointnet12_b200 import synthetic as syn
from test_gpu_parity import LOGP_TOL, TC_TOL, _chain_ref, _rand_layers, _seeded, cuda, dev, rel_err, starts, views  # noqa: F401

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ sampling at the C3 sizes
@pytest.mark.parametrize("N", [32768, 65536, 120000])
def test_fps_large_n_golden_and_oracle(dev, golden, N):
    """farthest_point_sample (pointnet_util.py:63-84) at N = 32768 (cluster of 8 x 256 threads), 65536 (the same without the
    z table: fps_async_kernel<8,32,false>) and 120000 (cluster of 16, barrier exchange: fps_kernel<512,16,true>):
    B = 2 against the reference's own indices, B = 8 and B = 1 against the oracle."""
    from pointnet12_b200.model import pointnet_util as U

    g = golden("fps_large_n")
    pts = syn.kitti_batch(2, N, config=3)
    got = U.farthest_point_sample(views(cuda(pts, dev))[0], 1024, start_idx=torch.from_numpy(g[f"n{N}_start"]))
    assert np.array_equal(got.cpu().numpy(), g[f"n{N}_fps"].astype(np.int64))
    for B, npoint in ((8, 256), (1, 512)):
        pts = syn.kitti_batch(B, N, config=4)
        st = starts([N], B, seed=N + B)[0]
        want = orc.farthest_point_sample(pts.transpose(0, 2, 1)[:, :, :3], npoint, st.numpy())
        got = U.farthest_point_sample(views(cuda(pts, dev))[0], npoint, start_idx=st)
        assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("B,N,npoint,config", [(8, 24000, 1024, None), (3, 5000, 300, None), (2, 33000, 256, None), (1, 49152, 128, None),
                                                (5, 777, 100, None), (2, 24000, 256, (0, 512, 0)), (2, 24000, 256, (0, 256, 0)),
                                                (2, 12289, 200, (0, 0, 1))])
def test_fps_bucket_pruned_equals_reference_order(dev, B, N, npoint, config):
    """pn_fps_sorted_f32: farthest-point sampling with exact bucket pruning over the cell-sorted copy of the cloud (32 x 12,
    16 x 24 and 8 x 24 warps x points per lane; 1-4 CTAs per cloud; pruning off): the same indices as the oracle, bit for
    bit -- ties between duplicated points are resolved by ORIGINAL index although storage order is bucket order."""
    from pointnet12_b200 import ops

    pts = syn.kitti_batch(B, N, config=8)
    st = starts([N], B, seed=N)[0]
    want = orc.farthest_point_sample(pts.transpose(0, 2, 1)[:, :, :3], npoint, st.numpy())
    x0 = views(cuda(pts, dev))[0]
    grid = ops.ball_grid(x0, 0.1)
    got = ops.fps_sorted(x0, grid, npoint, st.to(dev), config=config)
    assert np.array_equal(got.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------ N <= sa1.npoint
@pytest.mark.parametrize("N", [1024, 512])
@pytest.mark.parametrize("mode", ["bf16x3", "fp32"])
def test_pointnet2_semseg_small_n_golden(dev, golden, ckpt_path, N, mode):
    """PointNet2SemSeg with no more points than level 1 samples (pointnet2.py:159-176): fp1 does not upsample, so its first
    layer must NOT be folded into fp2's chain (round-1 advisor finding: it was applied twice)."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    g = golden("semseg_small_n")
    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    x = cuda(syn.kitti_batch(2, N, config=21), dev)
    with ops.options(precision=mode), torch.no_grad():
        torch.manual_seed(N)
        got = net(x)
        assert rel_err(got, g[f"n{N}_logp"]) < LOGP_TOL
        assert (got.argmax(-1).cpu().numpy() == g[f"n{N}_logp"].argmax(-1)).mean() > 0.999
        torch.manual_seed(N)
        assert torch.equal(GraphedSemSeg(net)(x), got)


# ------------------------------------------------------------------------------------------------ C4 in the mode the config names
def test_pointnet2_cls_msg_b32_bf16_and_bf16x3(dev, golden):
    """Config C4: PointNet2ClsMsg (pointnet2.py:7-47), 32 ModelNet40-shaped clouds of 1024 points.
    bf16x3 (fp32 parity): within 1e-3 relative of the reference's log-probabilities, labels equal.
    bf16 (the mode the config names: single-pass bf16 products, fp32 accumulation), STATED TOLERANCE against the reference:
    max |delta log-prob| <= 0.25, mean <= 0.03, the pooled 1024-channel descriptor within 3 % of its range, and the label
    equal wherever the reference's own top-2 margin exceeds 0.25 (seeded random weights give near-uniform log-probs, so the
    margin condition matters here; with trained weights margins are far larger)."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model.pointnet2 import PointNet2ClsMsg

    g = golden("cls_msg_b32")
    net = _seeded(PointNet2ClsMsg(), 1234, dev)
    x = cuda(syn.modelnet_batch(32, 1024), dev)
    with torch.no_grad():
        torch.manual_seed(0)
        logp, l3 = net(x)
        assert logp.shape == (32, 40) and l3.shape == (32, 1024, 1)
        assert rel_err(l3, g["l3_points"]) < LOGP_TOL and rel_err(logp, g["logp"]) < LOGP_TOL
        assert np.array_equal(logp.argmax(-1).cpu().numpy(), g["logp"].argmax(-1))
        with ops.options(precision="bf16"):
            assert ops.mlp_precision() == "bf16"
            torch.manual_seed(0)
            logp16, l316 = net(x)
    err = np.abs(logp16.cpu().numpy() - g["logp"])
    print(f"C4 bf16: max |dlogp| {err.max():.4f} mean {err.mean():.5f}; l3 rel {rel_err(l316, g['l3_points']):.4f}")
    assert err.max() <= 0.25 and err.mean() <= 0.03
    assert rel_err(l316, g["l3_points"]) <= 0.03
    top2 = np.sort(g["logp"], -1)[:, -2:]
    sure = (top2[:, 1] - top2[:, 0]) > 0.25
    assert np.array_equal(logp16.argmax(-1).cpu().numpy()[sure], g["logp"].argmax(-1)[sure])


# ------------------------------------------------------------------------------------------------ remaining golden gaps
def test_partseg_msg_one_hot_golden(dev, golden):
    """PointNet2PartSegMsg_one_hot (pointnet2.py:106-139) on the reference's own smoke input (pointnet2.py:179-187)."""
    from pointnet12_b200.model.pointnet2 import PointNet2PartSegMsg_one_hot

    g = golden("partseg_msg_one_hot")
    net = _seeded(PointNet2PartSegMsg_one_hot(50), 5, dev)
    gen = torch.Generator().manual_seed(0)
    x = torch.randn((8, 3, 2048), generator=gen).to(dev)
    label = torch.randn((8, 16), generator=gen).to(dev)
    with torch.no_grad():
        torch.manual_seed(0)
        out = net(x, x, label)
    assert out.shape == (8, 2048, 50)
    assert rel_err(out[:, ::8], g["logp_sub"]) < LOGP_TOL
    sure = g["margin"].astype(np.float32) > 2e-3
    assert np.array_equal(out.argmax(-1).cpu().numpy()[sure], g["label"].astype(np.int64)[sure])


def test_pointnet_seg_c1_golden(dev, golden):
    """Config C1: PointNetSeg (pointnet.py:230-254), B = 1, N = 24000, eager and through the CUDA-graph runner."""
    from pointnet12_b200.model.pointnet import PointNetSeg
    from pointnet12_b200.runtime import GraphedModule

    g = golden("pointnet_seg_c1")
    net = _seeded(PointNetSeg(19, input_dims=4, feature_transform=True), 1234, dev)
    x = cuda(syn.kitti_batch(1, 24000, config=1), dev)
    with torch.no_grad():
        logp, tf = net(x)
    assert logp.shape == (1, 24000, 19) and tf.shape == (1, 64, 64)
    assert rel_err(tf, g["trans_feat"]) < LOGP_TOL and rel_err(logp[:, ::8], g["logp_sub"]) < LOGP_TOL
    sure = g["margin"].astype(np.float32) > 2e-3
    assert np.array_equal(logp.argmax(-1).cpu().numpy()[sure], g["label"].astype(np.int64)[sure])
    runner = GraphedModule(net)
    for _ in range(2):
        glogp, gtf = runner(x)
        assert torch.equal(glogp, logp) and torch.equal(gtf, tf)


# ------------------------------------------------------------------------------------------------ batches in flight
@pytest.mark.parametrize("config", [(2, 256, 2), (2, 256, 3), (3, 256, 2), (3, 256, 3)])
def test_fps_few_wide_ctas(dev, config):
    """The level-1 shapes of the deep pipelines: a 24000-point cloud on 2 CTAs x 8 warps (48 points per thread, the whole
    register file) or 3 CTAs (cluster of three) -- bit-exact against the oracle like every other shape."""
    from pointnet12_b200 import ops

    B, N, npoint = 2, 24000, 256
    pts = syn.kitti_batch(B, N, config=17)
    st = starts([N], B, seed=23)[0]
    want = orc.farthest_point_sample(pts.transpose(0, 2, 1)[:, :, :3], npoint, st.numpy())
    got = ops.fps(views(cuda(pts, dev))[0], npoint, st.to(dev), config=config)
    assert np.array_equal(got.cpu().numpy(), want)
    ctas, _ = ops.fps_launch_info(B, N, npoint, config)
    assert ctas == B * config[0]


@pytest.mark.parametrize("depth", [2, 3, 8])
def test_pipelined_runner_equals_sequential(dev, ckpt_path, depth):
    """GraphedSemSeg(depth = 2, 3, 8; from 8 on level-1 sampling runs on 2 CTAs per cloud): the forwards of consecutive batches overlap on the GPU (sampling of batch k+1 beside
    the chains of batch k, chain tiles handed out dynamically); over 6 different batches the log-probabilities are
    torch.equal to the sequential (depth 1) runner's and to the eager forward's, on the device and through the pinned
    host output."""
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    B, N = 8, 24000
    xs = [cuda(syn.kitti_batch(B, N, config=2, first=8 * i), dev) for i in range(6)]
    torch.manual_seed(3)
    want = GraphedSemSeg(net, depth=1).run_pipelined(xs)
    torch.manual_seed(3)
    with torch.no_grad():
        assert torch.equal(net(xs[0]), want[0])
    runner = GraphedSemSeg(net, depth=depth)
    for rep in range(2):
        torch.manual_seed(3)
        got = runner.run_pipelined(xs)
        assert len(got) == 6 and all(torch.equal(a, b) for a, b in zip(got, want)), f"device output, pass {rep}"
    hosts = [x.cpu().pin_memory() for x in xs]
    torch.manual_seed(3)
    got = runner.run_pipelined(hosts, to_host=True)
    assert all((not a.is_cuda) and torch.equal(a, b.cpu()) for a, b in zip(got, want)), "pinned host output"
    # a ticket whose buffer set has been reused is refused instead of returning another batch's result
    tickets = [runner.submit(xs[i % len(xs)]) for i in range(depth + 1)]
    with pytest.raises(RuntimeError, match="overwritten"):
        runner.result(tickets[0])
    torch.cuda.synchronize()


def test_graph_runner_follows_weight_updates(dev, ckpt_path):
    """The captured graphs bake in the packed-weight blobs: after a parameter / BatchNorm buffer changes (optimizer step,
    load_state_dict) the runner must rebuild instead of replaying the old weights (round-1 advisor finding)."""
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    x = cuda(syn.kitti_batch(2, 4096, config=7), dev)
    runner = GraphedSemSeg(net)
    torch.manual_seed(1)
    before = runner(x).clone()
    with torch.no_grad():
        net.module.conv2.bias.add_(0.5 * torch.arange(19, device=dev, dtype=torch.float32))    # in place: version bump
        net.module.sa1.mlp_bns[0].running_mean.mul_(0.9)
        torch.manual_seed(1)
        want = net(x).clone()
    torch.manual_seed(1)
    got = runner(x)
    assert torch.equal(got, want) and not torch.equal(got, before)
    sd = {k: v.clone() for k, v in torch.load(ckpt_path, map_location="cpu").items()}
    net.load_state_dict(sd)
    torch.manual_seed(1)
    assert torch.equal(runner(x), before)


# ------------------------------------------------------------------------------------------------ dynamic tile scheduler
@pytest.mark.parametrize("dims,rows,mode", [([(4, 32), (32, 32), (32, 64)], 128 * 700 + 32, "max"),
                                            ([(128, 128), (128, 128), (128, 128), (128, 19)], 128 * 400 + 5, "logsoftmax"),
                                            ([(67, 64), (64, 64), (64, 128)], 128 * 3 + 64, "rows")])
def test_mlp_resident_dynamic_tiles(dev, dims, rows, mode):
    """pn_launch_opts.tile_counter: the resident-weight kernel hands out its tiles through a counter (more tiles than CTAs,
    fewer tiles than CTAs, ragged tail); results are bit-identical to the static round-robin and the counter is back at
    zero after every launch, so a captured graph can replay it."""
    from pointnet12_b200 import ops

    layers = _rand_layers(dims, seed=rows % 1000, last_relu=(mode == "max"))
    x = cuda(np.random.default_rng(rows).normal(size=(rows, dims[0][0])).astype(np.float32), dev)
    chain = ops.PackedChain([(cuda(w, dev), cuda(b, dev), r) for w, b, r in layers])
    out_mode = {"max": ops.OUT_MAX32, "logsoftmax": ops.OUT_LOG_SOFTMAX, "rows": ops.OUT_ROWS}[mode]
    ops.set_mlp_engine("resident")
    try:
        want = ops.mlp_rows_tc(chain, x, out_mode)
        pool = ops.TileCounters(dev, 8)
        with ops.options(tile_counters=pool):
            for _ in range(3):
                got = ops.mlp_rows_tc(chain, x, out_mode)
                assert torch.equal(got, want)
        with ops.options(tile_counters=pool, reserved_sms=100):      # a grid of 48 CTAs
            assert torch.equal(ops.mlp_rows_tc(chain, x, out_mode), want)
        assert pool.used == 4 and int(pool.buf.abs().sum()) == 0
        # the same word used by consecutive launches (what a graph replay does)
        one = ops.TileCounters(dev, 1)
        for _ in range(3):
            one.used = 0
            with ops.options(tile_counters=one):
                assert torch.equal(ops.mlp_rows_tc(chain, x, out_mode), want)
    finally:
        ops.set_mlp_engine("auto")


# ------------------------------------------------------------------------------------------------ per-call launch options
def test_two_threads_two_precisions(dev, ckpt_path):
    """The ABI keeps no process-wide settings (pn_launch_opts travels with every call): one thread runs the fp32-parity
    mode while another runs single-pass bf16, concurrently on two streams, and each gets its own mode's result."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model.utils import load_pointnet

    nets = [load_pointnet("pointnet2", 19, ckpt_path, device=dev) for _ in range(2)]
    x = cuda(syn.kitti_batch(2, 4096, config=9), dev)
    st = [s.to(dev) for s in starts([4096, 1024, 256, 64], 2, seed=2)]
    want = {}
    with torch.no_grad():
        for i, mode in enumerate(("bf16x3", "bf16")):
            with ops.options(precision=mode):
                want[mode] = nets[i](x, fps_starts=st).clone()
    assert not torch.equal(want["bf16x3"], want["bf16"])
    torch.cuda.synchronize()
    got, errors = {}, []
    barrier = threading.Barrier(2)

    def work(i, mode):
        try:
            torch.cuda.set_device(dev)
            stream = torch.cuda.Stream(dev)
            with torch.cuda.stream(stream), torch.no_grad(), ops.options(precision=mode):
                barrier.wait()
                for _ in range(5):
                    assert ops.mlp_precision() == mode
                    out = nets[i](x, fps_starts=st)
                got[mode] = out.clone()
            stream.synchronize()
        except Exception as e:   # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=work, args=(i, m)) for i, m in enumerate(("bf16x3", "bf16"))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert ops.mlp_precision() == "bf16x3"
    for mode in ("bf16x3", "bf16"):
        assert torch.equal(got[mode], want[mode]), mode


def test_cross_entropy_poisons_out_of_range_labels(dev):
    """nn.CrossEntropyLoss raises on a label outside [0, C) other than its ignore_index -100; the asynchronous kernel
    returns NaN instead of silently training on a clamped label (round-1 advisor finding): labels C (19 here) and -1.
    Label -100 is ignored, as torch does (tests/test_gpu_train_edges.py compares that case with torch)."""
    from pointnet12_b200 import ops

    x = torch.randn(64, 19, device=dev)
    t = torch.randint(0, 19, (64,), device=dev)
    loss, dx = ops.cross_entropy(x, t)
    ref = torch.nn.functional.cross_entropy(x, t)
    assert abs(float(loss) - float(ref)) < 1e-5 and bool(torch.isfinite(dx).all())
    t[7] = 19
    loss, dx = ops.cross_entropy(x, t)
    assert bool(torch.isnan(loss)) and bool(torch.isnan(dx[7]).all()) and bool(torch.isfinite(dx[8]).all())
    t[7] = -1
    loss, dx = ops.cross_entropy(x, t)
    assert bool(torch.isnan(loss)) and bool(torch.isnan(dx[7]).all()) and bool(torch.isfinite(dx[8]).all())
    t[7] = -100
    loss, dx = ops.cross_entropy(x, t)
    assert bool(torch.isfinite(loss)) and not bool(dx[7].any()) and bool(torch.isfinite(dx).all())


def test_labels_output_mode(dev, ckpt_path):
    """to_host="labels": only pred.argmax(-1) (pcdseg.py:75) travels to the host, as uint8; equal to the arg-max of the
    log-probabilities (first maximum wins, like torch.argmax), sequential and with batches in flight."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    x = torch.randn(1000, 19, device=dev)
    x[5, 3] = x[5, 7] = 9.0                                   # a tie: the first maximum wins
    assert torch.equal(ops.argmax_labels(x).long(), x.argmax(-1)) and int(ops.argmax_labels(x)[5]) == 3
    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    xs = [cuda(syn.kitti_batch(4, 8000, config=2, first=4 * i), dev) for i in range(4)]
    for depth in (1, 3):
        runner = GraphedSemSeg(net, depth=depth)
        torch.manual_seed(9)
        want = [r.argmax(-1).to(torch.uint8).cpu() for r in runner.run_pipelined(xs)]
        torch.manual_seed(9)
        got = runner.run_pipelined([x.cpu().pin_memory() for x in xs], to_host="labels")
        assert all(g.dtype == torch.uint8 and not g.is_cuda and torch.equal(g, w) for g, w in zip(got, want))


def test_graphed_module_cls_msg(dev, golden):
    """runtime.GraphedModule on a net that samples (PointNet2ClsMsg): the FPS start indices are drawn per call like the
    reference draws them, so a replay equals the eager forward under the same seed -- for different seeds too."""
    from pointnet12_b200.model.pointnet2 import PointNet2ClsMsg
    from pointnet12_b200.runtime import GraphedModule

    net = _seeded(PointNet2ClsMsg(), 1234, dev)
    x = cuda(syn.modelnet_batch(32, 1024), dev)
    runner = GraphedModule(net)
    for seed in (0, 1, 2):
        torch.manual_seed(seed)
        with torch.no_grad():
            want_logp, want_l3 = net(x)
            want_logp, want_l3 = want_logp.clone(), want_l3.clone()
        torch.manual_seed(seed)
        logp, l3 = runner(x)
        assert torch.equal(logp, want_logp) and torch.equal(l3, want_l3)
    g = golden("cls_msg_b32")
    torch.manual_seed(0)
    assert rel_err(runner(x)[0], g["logp"]) < LOGP_TOL


@pytest.mark.parametrize("block", ["8", "32"])
def test_three_nn_block_size_hook(dev, block):
    """PN12_NN_BLOCK (read once per process) forces the block size of the 3-NN block search: 8 and 32 points per block give the
    all-pairs scan's indices and weights like the default 16 (own process: the hook is latched at first use)."""
    import os
    import subprocess
    import sys

    code = (
        "import torch, numpy as np\n"
        "from pointnet12_b200 import ops, synthetic as syn\n"
        "dev = torch.device('cuda', 0)\n"
        "x = torch.from_numpy(syn.kitti_batch(2, 6000, config=6)).to(dev).permute(0, 2, 1)[:, :, :3]\n"
        "for S in (1024, 100):\n"
        "    st = torch.zeros((2,), dtype=torch.long, device=dev)\n"
        "    c = ops.index_points(x, ops.fps(x, S, st)).contiguous()\n"
        "    grid = ops.ball_grid(x, 0.1)\n"
        "    bi, bw = ops.three_nn(x, c, order=grid, method='blocks')\n"
        "    si, sw = ops.three_nn(x, c, method='scan')\n"
        "    assert torch.equal(bi, si) and torch.equal(bw, sw), S\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PN12_NN_BLOCK=block, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_pipelined_runner_picks_a_sampling_shape_that_fits(dev, ckpt_path):
    """With batches in flight level-1 sampling runs on as few CTAs as hold the cloud in registers (2 x 256 threads x 48 points
    up to N = 24576); a larger cloud must move to 3, 4 or 8 CTAs (or the automatic shape) instead of failing, and the results
    stay torch.equal to the one-batch-at-a-time runner's."""
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    deep = GraphedSemSeg(net, depth=8)
    assert deep.fps1_shape(24000) == (2, 256, 2) and deep.fps1_shape(30000) == (3, 256, 2) and deep.fps1_shape(40000) == (4, 256, 2)
    assert deep.fps1_shape(98304) == (8, 256, 2) and deep.fps1_shape(120000) is None
    assert GraphedSemSeg(net, depth=1).fps1_shape(24000) is None
    for N in (30000, 2048, 512):          # (small clouds: no bucket grid below 4096 points, fewer points than centroids at 512)
        xs = [cuda(syn.kitti_batch(2, N, config=2, first=2 * i), dev) for i in range(3)]
        torch.manual_seed(5)
        want = GraphedSemSeg(net, depth=1).run_pipelined(xs)
        torch.manual_seed(5)
        got = deep.run_pipelined(xs)
        assert all(torch.equal(a, b) for a, b in zip(got, want)), N
    torch.cuda.synchronize()
