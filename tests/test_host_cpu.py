"""CPU-only checks of the host side: the C ABI loads and exports every declared symbol, argument validation
works without a GPU, CPU tensors are refused, state_dict / checkpoint compatibility, and the data-parallel
sharding helpers under a world_size-2 gloo group."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

from pointnet12_b200 import _native as nv
from pointnet12_b200 import dist as pdist


def test_library_exports_every_declared_symbol():
    lib = nv.lib()
    declared = nv.declared_symbols()
    assert len(declared) >= 19 and "pn_fps_f32" in declared and "pn_fp_mlp_bf16x3" in declared
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, f"libpn12_b200.so does not export {missing}"
    assert lib.pn_version() >= 100


def test_argument_validation_needs_no_gpu():
    lib = nv.lib()
    assert lib.pn_fps_f32(None, 0, 0, 0, 1, 16, 4, None, None, None, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    # launch options travel with the call (pn_launch_opts); a bad cluster size is refused before anything is launched
    ctas, smem = C.c_int(), C.c_size_t()
    bad = nv.LaunchOpts()
    bad.fps_cluster = 5
    assert lib.pn_fps_launch_info(8, 24000, 1024, C.byref(bad), C.byref(ctas), C.byref(smem)) == -1
    assert b"fps_cluster" in lib.pn_last_error_string()
    assert lib.pn_fps_launch_info(8, 24000, 1024, None, C.byref(ctas), C.byref(smem)) == 0 and ctas.value == 64
    four = nv.LaunchOpts()
    four.fps_cluster, four.fps_threads, four.fps_exchange = 4, 256, 2
    assert lib.pn_fps_launch_info(8, 24000, 1024, C.byref(four), C.byref(ctas), C.byref(smem)) == 0 and ctas.value == 32
    # no process-wide setters are left in the ABI
    assert not [s for s in nv.declared_symbols() if "_set_" in s]
    d = nv.MlpDesc()
    d.nlayers = 2
    d.cin[0], d.cout[0], d.relu[0] = 128, 128, 1
    d.cin[1], d.cout[1], d.relu[1] = 128, 19, 0
    assert lib.pn_mlp_blob_bytes(C.byref(d)) == 128 * 128 * 4 + 32 * 128 * 4 + (128 + 32) * 4
    d.cin[1] = 64                                  # does not chain
    assert lib.pn_mlp_blob_bytes(C.byref(d)) == 0 and b"cin[l]" in lib.pn_last_error_string()
    d.cin[1], d.cout[0], d.cin[1] = 512, 512, 512   # hidden layer wider than 256
    assert lib.pn_mlp_blob_bytes(C.byref(d)) == 0


def test_cpu_tensors_are_refused():
    from pointnet12_b200.model import pointnet_util as U
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        U.square_distance(torch.zeros(1, 16, 3), torch.zeros(1, 16, 3))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        U.index_points(torch.zeros(1, 16, 3), torch.zeros(1, 4, dtype=torch.long))
    net = PointNet2SemSeg(19, feature_dims=1).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(torch.zeros(1, 4, 2048))


def test_checkpoint_state_dict_contract(ckpt_path):
    """The reference's checkpoint loads strict=True into the drop-in modules (names, shapes, dtypes)."""
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg
    from pointnet12_b200.model.utils import ModuleWrapper

    sd = torch.load(ckpt_path, map_location="cpu")
    net = ModuleWrapper(PointNet2SemSeg(19, feature_dims=1))
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    own = net.state_dict()
    assert list(own.keys()) == list(sd.keys())
    assert all(own[k].shape == sd[k].shape and own[k].dtype == sd[k].dtype for k in sd)
    assert sum(p.numel() for p in net.parameters()) == 968787


def test_bn_folding_matches_unfolded():
    from pointnet12_b200.model.pointnet_util import FoldedLayers, fold_conv_bn

    torch.manual_seed(0)
    conv, bn = torch.nn.Conv1d(7, 5, 1), torch.nn.BatchNorm1d(5).eval()
    bn.running_mean.normal_()
    bn.running_var.uniform_(0.5, 2)
    bn.weight.data.normal_()
    bn.bias.data.normal_()
    x = torch.randn(3, 7, 11)
    w, b = fold_conv_bn(conv, bn)
    got = torch.einsum("oc,bcn->bon", w, x) + b[None, :, None]
    assert torch.allclose(got, bn(conv(x)), atol=1e-5)
    f = FoldedLayers()
    first = f.get([conv], [bn])
    assert f.get([conv], [bn]) is first                 # cached
    bn.running_mean.add_(1.0)                           # any change refolds
    assert f.get([conv], [bn]) is not first


def test_shard_range_partitions():
    for n, world in [(8, 1), (8, 2), (8, 4), (8, 8), (7, 4), (3, 8), (64, 8)]:
        spans = [pdist.shard_range(n, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [hi - lo for lo, hi in spans]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        pdist.shard_range(8, 2, 2)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        assert pdist.env_world() == (rank, world, rank)
        from pointnet12_b200 import synthetic as syn

        glob = torch.from_numpy(syn.kitti_batch(5, 256, config=8))          # uneven: 3 + 2 clouds
        mine = pdist.shard_batch(glob, rank, world)
        lo, hi = pdist.shard_range(5, rank, world)
        assert mine.shape[0] == hi - lo and torch.equal(mine, glob[lo:hi])
        labels = (mine[:, 0, :] * 1000).long()                              # stand-in for per-rank predictions
        allv = pdist.gather_labels(labels, 5)
        assert torch.equal(allv, (glob[:, 0, :] * 1000).long())
        ms = pdist.max_over_ranks([1.0 + rank, 5.0 - rank])
        assert ms == [float(world), 5.0]
        # training step, data-parallel exchange: every rank's flat gradient is summed by ONE all-reduce and the 1/world
        # factor is returned for the Adam kernel (train.FlatAdam; the update itself is a CUDA kernel, not run here)
        from pointnet12_b200.train import FlatAdam

        torch.manual_seed(0)
        lin = torch.nn.Sequential(torch.nn.Conv1d(4, 8, 1), torch.nn.BatchNorm1d(8))
        opt = FlatAdam(lin.parameters(), lr=1e-3, weight_decay=1e-4)
        assert opt.flat.numel() == sum(p.numel() for p in lin.parameters())
        assert all(p.data_ptr() >= opt.flat.data_ptr() for p in lin.parameters())        # parameters live in the flat buffer
        opt.zero_grad()
        lin(torch.randn(2, 4, 5)).sum().backward()                                        # autograd accumulates in place
        assert opt.grad.abs().sum() > 0 and all(p.grad.data_ptr() >= opt.grad.data_ptr() for p in lin.parameters())
        opt.grad.fill_(1.0 + rank)
        scale = opt.all_reduce()
        assert scale == 1.0 / world and torch.equal(opt.grad, torch.full_like(opt.grad, sum(1.0 + r for r in range(world))))
        out.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        out.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_sharding_world_size_2_gloo():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    results = dict(out.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert results == {0: "ok", 1: "ok"}, results


def test_reference_import_path_aliases():
    """`from model.pointnet2 import PointNet2SemSeg` (the reference's spelling) resolves to the drop-in."""
    import model.pointnet2 as m2
    import model.pointnet_util as mu
    from pointnet12_b200.model import pointnet2, pointnet_util

    assert m2.PointNet2SemSeg is pointnet2.PointNet2SemSeg
    assert mu.farthest_point_sample is pointnet_util.farthest_point_sample
    for name in ("square_distance", "index_points", "farthest_point_sample", "query_ball_point", "sample_and_group",
                 "sample_and_group_all", "PointNetSetAbstraction", "PointNetSetAbstractionMsg",
                 "PointNetFeaturePropagation"):
        assert hasattr(mu, name)


def test_train_mode_refuses_cpu_tensors():
    """train() mode has no CPU fallback either: every trainable net refuses CPU tensors before any work is done."""
    from pointnet12_b200.model.pointnet import PointNetSeg
    from pointnet12_b200.model.pointnet2 import PointNet2ClsSsg, PointNet2PartSegSsg, PointNet2SemSeg
    from pointnet12_b200.train import cross_entropy

    for net, x in ((PointNet2SemSeg(19, feature_dims=1), torch.zeros(1, 4, 2048)), (PointNet2ClsSsg(), torch.zeros(2, 3, 1024)),
                   (PointNet2PartSegSsg(50), torch.zeros(2, 3, 1024)), (PointNetSeg(19, 4, True), torch.zeros(2, 4, 512))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            net.train()(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cross_entropy(torch.zeros(1, 8, 19), torch.zeros(1, 8, dtype=torch.long))


def test_training_abi_argument_validation_needs_no_gpu():
    """The training / pre-processing entry points validate their arguments before any launch (no GPU needed)."""
    lib = nv.lib()
    assert lib.pn_version() >= 300
    # planning helpers
    assert lib.pn_train_gemm_supported(128, 128) == 1 and lib.pn_train_gemm_supported(4, 32) == 1
    assert lib.pn_train_gemm_supported(259, 256) == 0            # 288 x 256 x 4 bytes of weights > 128 KB
    assert lib.pn_train_gemm_supported(128, 512) == 0            # more than 256 output channels
    assert lib.pn_train_gemm_scratch_bytes(67, 64) == 96 * 64 * 4 and lib.pn_train_gemm_scratch_bytes(259, 256) == 0
    assert lib.pn_scan_workspace_bytes(8, 120000) == 8 * 59 * 4 and lib.pn_scan_workspace_bytes(0, 5) == 0
    # null pointers / bad shapes are refused with a message, nothing is launched
    assert lib.pn_bn_stats_f32(None, 128, 10, 128, None, None, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    buf = (C.c_float * 4)()
    p = C.cast(buf, C.c_void_p)
    assert lib.pn_bn_stats_f32(p, 2, 10, 4, p, p, None) == -1    # leading dimension smaller than the row
    assert lib.pn_bn_bwd_stats_f32(p, 4, 10, 4, p, 4, p, 3, p, p, p, p, 1, p, p, None) == -1 and b"multiple of K" in lib.pn_last_error_string()
    assert lib.pn_grad_weight_f32(p, 4, p, 4, 0, 4, 4, p, 4, None, None) == -1
    assert lib.pn_dropout_f32(p, 4, 1, 4, C.c_float(1.5), p, None, None, p, 4, None) == -1       # p must be < 1
    assert lib.pn_adam_f32(p, p, p, p, 4, C.c_float(1e-3), C.c_float(0.9), C.c_float(0.999), C.c_float(1e-8), C.c_float(0.0), 0,
                           C.c_float(1.0), None) == -1 and b"step" in lib.pn_last_error_string()
    assert lib.pn_seg_metrics_f32(p, 100, p, 1, 100, None, p, None) == -1                       # more than 64 classes
    q = C.c_void_p(1 << 20)          # a 128-byte aligned address; validation fails before anything is dereferenced
    assert lib.pn_train_gemm_bf16x3(p, 259, 10, 259, None, None, 0, p, 0, None, 256, p, 256, None, None, q, None) == -2
    assert b"does not fit" in lib.pn_last_error_string()
    assert lib.pn_train_gemm_bf16x3(p, 4, 10, 4, p, None, 0, p, 0, None, 4, p, 4, None, None, q, None) == -1   # scale without shift
    assert lib.pn_train_gemm_bf16x3(p, 4, 10, 4, None, None, 0, p, 0, None, 4, p, 4, None, None, C.c_void_p((1 << 20) + 4), None) == -3
    assert lib.pn_scan_sample_f32(p, p, p, 1, p, 4, p, p, 8, None, None, C.c_float(0.0), C.c_float(0.0), None, p, p, None) == -1
    assert b"choice indices or a Philox seed" in lib.pn_last_error_string()
    assert lib.pn_chamfer_f32(p, 3, 3, 1, p, 3, 3, 1, 1, 1, 1, 9, None, p, None) == -1            # D <= 8


def _simulate_pacer(gpu_ms, host_ms, depth, steps, factor=0.92, seed_est=None):
    """Discrete-event model of the host-output loop: a GPU that finishes one batch every gpu_ms (FIFO, a batch cannot finish
    before gpu_ms after its submit), a host that needs host_ms per submit and waits for batch k before submitting batch k + depth.
    Returns (pacer, submit times)."""
    from pointnet12_b200.runtime import Pacer

    now = [0.0]
    pacer = Pacer(factor, clock=lambda: now[0])
    pacer.per_batch = seed_est
    done_at, submits, pending = [], [], []
    gpu_free = 0.0
    for k in range(steps):
        now[0] = max(now[0], pacer.next_submit_time())
        pacer.submitted()                      # (as in GraphedSemSeg.submit: the spacing counts from the start of a submit's host work)
        submits.append(now[0])
        now[0] += host_ms * 1e-3
        gpu_free = max(gpu_free, now[0]) + gpu_ms * 1e-3
        done_at.append(gpu_free)
        pending.append(k)
        if len(pending) >= depth:
            j = pending.pop(0)
            t0 = now[0]
            now[0] = max(now[0], done_at[j])
            pacer.completed(now[0] - t0)
    return pacer, submits


def test_pacer_follows_the_gpu_rate_and_never_throttles():
    """The submit pacing of the host-output loop (runtime.Pacer): with a GPU-bound loop the estimate settles on the GPU's time per
    batch and the submits end up evenly spaced just below it; an estimate that is far too large (a hiccup, another workload
    before) decays instead of throttling the loop; a host-bound loop is never slowed down."""
    # GPU-bound: 0.40 ms per batch, host 0.10 ms per submit
    pacer, submits = _simulate_pacer(gpu_ms=0.40, host_ms=0.10, depth=6, steps=400)
    assert 0.33e-3 < pacer.per_batch < 0.42e-3                            # (it hovers just below the GPU's 0.40 ms)
    gaps = [b - a for a, b in zip(submits[-50:-1], submits[-49:])]
    assert min(gaps) > 0.30e-3 and max(gaps) < 0.50e-3                   # no bursts, no stalls
    total = submits[-1] / len(submits)
    assert total < 0.41e-3                                                # throughput = the GPU's
    # a stale estimate five times too large decays geometrically: after 400 batches the loop runs at the GPU's rate again
    pacer, submits = _simulate_pacer(gpu_ms=0.40, host_ms=0.10, depth=6, steps=400, seed_est=2.0e-3)
    assert pacer.per_batch < 0.45e-3
    tail = (submits[-1] - submits[-101]) / 100
    assert tail < 0.41e-3
    # host-bound (0.6 ms per submit against 0.4 ms of GPU time): pacing must not add to it
    pacer, submits = _simulate_pacer(gpu_ms=0.40, host_ms=0.60, depth=6, steps=200)
    assert (submits[-1] - submits[-101]) / 100 < 0.61e-3
    # disabled estimate: first window of a fresh pacer never waits
    from pointnet12_b200.runtime import Pacer
    assert Pacer(0.92).next_submit_time() == 0.0


def test_pipelined_sampling_shape_follows_cloud_size():
    """Host logic of runtime.GraphedSemSeg.fps1_shape (no GPU needed): the fewest 8-warp CTAs whose threads hold the cloud in
    registers at 48 points each, from 2 (deep pipelines) or 3 upwards; the automatic shape for one batch at a time and beyond
    8 x 256 x 48 points."""
    import torch

    from pointnet12_b200.runtime import GraphedSemSeg

    net = torch.nn.Linear(2, 2)
    one, mid, deep = GraphedSemSeg(net, depth=1), GraphedSemSeg(net, depth=4), GraphedSemSeg(net, depth=10)
    assert one.fps1_shape(24000) is None and one.pace == 0.0
    assert [mid.fps1_shape(n) for n in (512, 24000, 36864, 36865, 49152, 49153, 98304, 98305)] == \
        [(3, 256, 2), (3, 256, 2), (3, 256, 2), (4, 256, 2), (4, 256, 2), (8, 256, 2), (8, 256, 2), None]
    assert [deep.fps1_shape(n) for n in (24000, 24576, 24577, 120000)] == [(2, 256, 2), (2, 256, 2), (3, 256, 2), None]
    for n in (24000, 30000, 60000, 98304):            # every chosen shape respects the kernel's limits (fps.cu: <= 48 points per thread,
        c, t, _ = deep.fps1_shape(n)                  # cluster x warps <= 64 slots)
        assert -(-(-(-n // c)) // t) <= 48 and c * (t // 32) <= 64


def test_runner_weight_change_detection_cheap_and_exact_for_inplace_updates(monkeypatch):
    """runtime.GraphedSemSeg._check_weights (host logic, no GPU): in a tight pipelined loop only the version counters are summed,
    and every in-place update (optimizer step, load_state_dict, copy_) is still caught at the next submit; a pointer change is
    caught by the full check after a pause; one batch at a time the full signature is taken on every call."""
    import time

    import torch

    from pointnet12_b200.runtime import GraphedSemSeg

    monkeypatch.setattr(torch.cuda, "synchronize", lambda dev=None: None)
    net = torch.nn.Sequential(torch.nn.Linear(4, 4), torch.nn.BatchNorm1d(4))
    r = GraphedSemSeg(net, depth=4)
    r._check_weights(None)
    r._graphs = {"shape": "graphs"}
    for _ in range(5):
        r._check_weights(None)
    assert r._graphs                                            # nothing changed: graphs kept
    with torch.no_grad():
        net[0].weight.mul_(2.0)                                 # in-place: version bump, same pointer
    r._check_weights(None)
    assert not r._graphs
    r._graphs = {"shape": "graphs"}
    net.load_state_dict({k: v.clone() + 1 for k, v in net.state_dict().items()})
    r._check_weights(None)
    assert not r._graphs
    r._graphs = {"shape": "graphs"}
    net[0].weight.data = net[0].weight.data.clone()             # pointer change without a version bump of the old storage
    time.sleep(0.003)                                           # ... seen by the full check that follows any pause
    r._check_weights(None)
    assert not r._graphs
    one = GraphedSemSeg(net, depth=1)
    one._check_weights(None)
    one._graphs = {"shape": "graphs"}
    net[1].running_mean.data = net[1].running_mean.data.clone()
    one._check_weights(None)                                    # depth 1: always the full signature
    assert not one._graphs
