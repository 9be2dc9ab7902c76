"""The sampling, ball-query and 3-NN kernels against the CPU oracle on clouds built to reach their edges (pointnet12_b200/
synthetic.py): ties between DISTINCT points and exact arithmetic (the 2^-5 lattice), points exactly on the radius and one ulp
either side (the boundary sets), sampling that runs out of distinct points, zero extent along an axis, metre-scale clouds
offset by 1000 m and points beyond the reference's initial FPS distance of 1e10.  Every test first asserts, with the
oracle, that its input reaches the edge it is named for; indices are then compared bit for bit, tie rows included (the
oracle defines them by (distance, index))."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pointnet12_b200 import synthetic as syn
from test_geometry_edges_cpu import fps64, on_radius_pairs, xyz_of          # the float64 restatements the CPU file pins
from test_gpu_parity import LOGP_TOL, TC_TOL, _rand_layers                   # the parity suite's tolerances and chains

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (run with -m 'not gpu' on CPU boxes)")
    from pointnet12_b200 import ops

    assert ops.device_check()[1] == 10, "kernels are built for sm_100a"
    return torch.device("cuda", 0)


def cuda(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def views(pts_dev):
    """[B,4,N] -> strided point-major views (xyz [B,N,3], feat [B,N,1]) as the reference makes them."""
    pm = pts_dev.permute(0, 2, 1)
    return pm[:, :, :3], pm[:, :, 3:]


def rel_err(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))

R_LATTICE = 3 * syn.LATTICE_STEP      # r**2 = 9/1024 exactly: hundreds of pairs on the radius
FPS_SHAPES = [(1, 1024, 0), (2, 512, 1), (4, 256, 1), (8, 128, 1), (8, 512, 1), (16, 128, 1), (16, 256, 1), (2, 128, 2),
              (2, 256, 2), (4, 64, 2), (4, 128, 2), (8, 64, 2), (8, 128, 2), (8, 256, 2), (16, 64, 2), (16, 128, 2), (8, 128, 3),
              (4, 128, 3), (16, 64, 3), (16, 512, 0), (8, 512, 0), (2, 1024, 0), (4, 512, 0)]


def cloud(family: str, B: int, N: int) -> np.ndarray:
    """[B, 4, N] of one edge family."""
    if family == "lattice":
        return syn.lattice_batch(B, N, seed=N)
    if family.startswith("few"):
        return syn.few_distinct_batch(B, N, int(family[3:]), seed=N)
    if family == "flat":
        return syn.flat_batch(B, N, "z")
    if family == "line":
        return syn.flat_batch(B, N, "yz")
    if family == "offset":
        return syn.offset_batch(B, N)
    if family == "outlier":
        return syn.outlier_batch(B, N)
    raise ValueError(family)


def mix(N: int) -> np.ndarray:
    """One cloud each of the lattice, 300 distinct points, the outlier cloud and the plane: [4, 4, N]."""
    return np.concatenate([cloud(f, 1, N) for f in ("lattice", "few300", "outlier", "flat")])


def assert_fps_edges(pts: np.ndarray, want: np.ndarray, start: np.ndarray) -> None:
    """The oracle's sampling of mix(N) reaches every edge: ties between distinct points (lattice), no distinct point left
    (300 points), the 1e10 cap (the nearer far point wins the tie), zero extent (plane)."""
    x = xyz_of(pts)
    npoint = want.shape[1]
    idx64, ties = fps64(x[0], min(npoint, 256), int(start[0]))
    assert np.array_equal(idx64, want[0, :len(idx64)]) and ties > len(idx64) // 2
    if npoint > 300:
        assert (want[1, 300:] == 0).all()
    assert x[2, want[2, 1], 0] == -syn.OUTLIER_FAR[0] and x[2, want[2, 2], 0] == syn.OUTLIER_FAR[1]
    assert np.ptp(x[3, :, 2]) == 0


_CACHE = {}


def fps_case(N: int, npoint: int):
    """(points, starts, oracle indices) of mix(N), cached over the module."""
    key = (N, npoint)
    if key not in _CACHE:
        pts = mix(N)
        st = np.array([N // 3, 7, N - 1, 0], dtype=np.int64)
        want = orc.farthest_point_sample(xyz_of(pts), npoint, st)
        assert_fps_edges(pts, want, st)
        _CACHE[key] = pts, st, want
    return _CACHE[key]


# ------------------------------------------------------------------------------------------------ farthest-point sampling
@pytest.mark.parametrize("family", ["lattice", "few1", "few3", "few300", "flat", "line", "offset", "outlier"])
def test_fps_edge_clouds(dev, family):
    """ops.fps on its automatic shape, B = 2, N = 24000, 1024 samples."""
    from pointnet12_b200 import ops

    pts = cloud(family, 2, 24000)
    x = xyz_of(pts)
    st = np.array([11, 23999], dtype=np.int64)
    want = orc.farthest_point_sample(x, 1024, st)
    if family == "lattice":
        idx64, ties = fps64(x[0], 1024, int(st[0]))
        assert np.array_equal(idx64, want[0]) and ties > 900
    elif family.startswith("few"):
        assert (want[:, int(family[3:]):] == 0).all()
    elif family in ("flat", "line"):
        assert (np.ptp(x[..., 2], axis=1) == 0).all() and (family == "flat" or (np.ptp(x[..., 1], axis=1) == 0).all())
    elif family == "offset":
        assert ((x.astype(np.float64) ** 2).sum(-1) > 1e6).all()
    else:
        assert (x[np.arange(2), want[:, 1], 0] == -syn.OUTLIER_FAR[0]).all()
    got = ops.fps(views(cuda(pts, dev))[0], 1024, cuda(st, dev))
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("cluster,threads,exchange", FPS_SHAPES)
def test_fps_every_cluster_shape_on_edges(dev, cluster, threads, exchange):
    """Every cluster size / CTA width / exchange mechanism of test_fps_every_cluster_shape, on mix(8000), 512 samples."""
    from pointnet12_b200 import ops

    pts, st, want = fps_case(8000, 512)
    got = ops.fps(views(cuda(pts, dev))[0], 512, cuda(st, dev), config=(cluster, threads, exchange))
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("config", [(2, 256, 2), (3, 256, 3)])
def test_fps_few_wide_ctas_on_edges(dev, config):
    """The level-1 shapes of the deep pipelines (2 or 3 CTAs x 8 warps holding a 24000-point cloud in registers)."""
    from pointnet12_b200 import ops

    pts, st, want = fps_case(24000, 1024)
    got = ops.fps(views(cuda(pts, dev))[0], 1024, cuda(st, dev), config=config)
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("config", [None, (0, 512, 0), (0, 256, 0), (0, 0, 1)])
def test_fps_bucket_pruned_on_edges(dev, config):
    """ops.fps_sorted (bucket pruning over the cell-sorted cloud; (0, 0, 1): pruning off) on mix(24000)."""
    from pointnet12_b200 import ops

    pts, st, want = fps_case(24000, 1024)
    x = views(cuda(pts, dev))[0]
    got = ops.fps_sorted(x, ops.ball_grid(x, 0.1), 1024, cuda(st, dev), config=config)
    assert np.array_equal(got.cpu().numpy(), want)


def test_fps_progress_words_on_edges(dev):
    """fps(..., progress=): the published words are (index << 32 | 1), equal to the returned indices."""
    from pointnet12_b200 import ops

    pts, st, want = fps_case(24000, 1024)
    progress = torch.zeros((4, 1024), dtype=torch.int64, device=dev)
    got = ops.fps(views(cuda(pts, dev))[0], 1024, cuda(st, dev), progress=progress)
    torch.cuda.synchronize()
    p = progress.cpu().numpy()
    assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(p >> 32, want) and ((p & 0xFFFFFFFF) == 1).all()


@pytest.mark.parametrize("N", [3072, 3073])
@pytest.mark.parametrize("npoint", [1, 500, "N"])
def test_fps_npoint_edges_around_single_cta(dev, N, npoint):
    """N = 3072 (one CTA per cloud) / 3073 (a cluster); one sample, more samples than distinct points (500 > 300) and N."""
    from pointnet12_b200 import ops

    npoint = N if npoint == "N" else npoint
    pts = np.concatenate([cloud("lattice", 1, N), cloud("few300", 1, N)])
    st = np.array([N - 1, 1], dtype=np.int64)
    x = xyz_of(pts)
    want = orc.farthest_point_sample(x, npoint, st)
    assert (want[:, 0] == st).all()
    idx64, ties = fps64(x[0], npoint, int(st[0]))
    assert np.array_equal(idx64, want[0]) and (ties > npoint // 2 or npoint == 1)
    if npoint > 300:
        assert (want[1, 300:] == 0).all()
    if npoint == N:
        assert len(np.unique(want[0])) == N
    got = ops.fps(views(cuda(pts, dev))[0], npoint, cuda(st, dev))
    assert np.array_equal(got.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------ ball query
def fps_queries(pts: np.ndarray, S: int) -> np.ndarray:
    x = xyz_of(pts)
    sel = orc.farthest_point_sample(x, S, np.zeros(len(x), dtype=np.int64))
    return np.ascontiguousarray(np.stack([x[b][sel[b]] for b in range(len(x))]))


def grid_plan(x: np.ndarray, radius: float):
    """Cells per axis and the cell of every point of one cloud under the plan of ball_grid.cu (restated in float64: coarse
    checks only) -> (g [3], cell [N, 3])."""
    lo, hi = x.min(0).astype(np.float64), x.max(0).astype(np.float64)
    m2 = (np.maximum(np.abs(lo), np.abs(hi)) ** 2).sum()
    h0 = np.sqrt(radius ** 2 + m2 / 262144) * 1.001
    ext = hi - lo
    g = np.where(ext / h0 < 31, np.floor(ext / h0).astype(int) + 1, 32)
    h = np.where(g == 32, np.maximum(h0, ext / 32 * 1.001), h0)
    return g, np.minimum(((x - lo) / h).astype(int), g - 1)


def dense_threshold(N: int) -> int:
    """gq_auto_threshold of ball_grid.cu: more candidates than this in the 27 cells send a query to the ordered scan."""
    t = 64
    while t * t < 1024 * N:
        t += 64
    return t


BALL_CASES = [("lattice", 4095, R_LATTICE, 1), ("lattice", 4096, R_LATTICE, 32), ("lattice", 4096, R_LATTICE, 128),
              ("lattice", 4095, R_LATTICE, 128), ("few1", 4096, 0.1, 32), ("few300", 8192, 0.1, 128), ("flat", 8192, 0.1, 32),
              ("line", 8192, 0.2, 32), ("offset", 8192, 0.2, 32), ("offset", 8192, 0.5, 128), ("outlier", 8192, 0.1, 32)]


@pytest.mark.parametrize("method", ["auto", "scan", "grid", "grid-cells", "grid-scan"])
@pytest.mark.parametrize("family,N,radius,K", BALL_CASES)
def test_ball_query_edge_clouds(dev, method, family, N, radius, K):
    """Every ball-query method on FPS centroids and on points of the cloud itself (N = 4095 / 4096 straddle GRID_MIN_POINTS)."""
    from pointnet12_b200 import ops

    pts = cloud(family, 2, N)
    x = xyz_of(pts)
    q = np.ascontiguousarray(np.concatenate([fps_queries(pts, 128), x[:, :128]], axis=1))
    want = orc.query_ball_point(radius, K, x, q)
    if family == "lattice":
        assert on_radius_pairs(x, q, radius) > 100
    elif family == "few1":
        assert (np.ptp(x, axis=1) == 0).all()
    elif family in ("flat", "line"):
        assert (np.ptp(x[..., 2], axis=1) == 0).all()
    elif family == "offset":     # the expansion formula and the exact distance disagree on membership
        d = orc.square_distance(q, x)
        exact = ((q[:, :, None, :].astype(np.float64) - x[:, None].astype(np.float64)) ** 2).sum(-1)
        assert ((d <= np.float32(radius ** 2)) != (exact <= radius ** 2)).sum() > 10
    elif family == "outlier":    # 32 cells along x (the cap), and the cloud's body in one cell: the dense path
        for b in range(2):
            g, cell = grid_plan(x[b], radius)
            assert g[0] == 32 and np.unique(cell, axis=0, return_counts=True)[1].max() > dense_threshold(N)
    got = ops.ball_query(radius, K, views(cuda(pts, dev))[0], cuda(q, dev), method=method)
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("method", ["auto", "scan", "grid", "grid-cells", "grid-scan"])
@pytest.mark.parametrize("radius", [0.1, 0.2, 0.4, 0.8])
def test_ball_query_boundary_sets(dev, method, radius):
    """Points whose squared distance to the query (the origin) is fp32(radius**2) and one ulp either side: the first two
    levels are in the ball, the third is not; the threshold is fp32(radius**2), not fp32(fp32(radius)**2)."""
    from pointnet12_b200 import ops

    pts = syn.boundary_batch(2, 4096, radius, seed=int(radius * 10))
    x = xyz_of(pts)
    q = np.ascontiguousarray(x[:, :1])
    d = orc.square_distance(q, x)[:, 0]
    r2 = np.float32(radius ** 2)
    assert np.float32(np.float32(radius) ** 2) == np.nextafter(r2, np.float32(1))
    assert ((d == r2).sum(1) == 24).all() and ((d == np.nextafter(r2, np.float32(1))).sum(1) == 24).all()
    for K in (32, 128):
        want = orc.query_ball_point(radius, K, x, q)
        if K == 128:
            assert all(len(set(want[b, 0])) == 49 for b in range(2))
        got = ops.ball_query(radius, K, views(cuda(pts, dev))[0], cuda(q, dev), method=method)
        assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("radius", [0.1, 0.2, 0.4, 0.8, R_LATTICE])
def test_public_path_radius_on_boundary_rows(dev, radius):
    """pointnet_util.query_ball_point and sample_and_group (the first centroid is the origin: start index 0) derive the
    threshold from the python radius like the reference; the grouped rows are bit-exact."""
    from pointnet12_b200.model import pointnet_util as U

    if radius == R_LATTICE:
        pts = syn.lattice_batch(2, 4096, side=16, seed=5)     # every site taken: the whole shell of radius 3/32
        pts[:, :3] -= pts[:, :3, :1]          # point 0 at the origin; still on the lattice
    else:
        pts = syn.boundary_batch(2, 4096, radius, seed=3)
    x = xyz_of(pts)
    q = np.ascontiguousarray(x[:, :1])
    assert on_radius_pairs(x, q, radius) >= 2 * (24 if radius != R_LATTICE else 6)
    xyz, feat = views(cuda(pts, dev))
    got = U.query_ball_point(radius, 128, xyz, cuda(q, dev))
    assert np.array_equal(got.cpu().numpy(), orc.query_ball_point(radius, 128, x, q))
    st = np.zeros(2, dtype=np.int64)
    w_xyz, w_points, w_fps, w_idx = orc.sample_and_group(64, radius, 32, x, np.ascontiguousarray(pts.transpose(0, 2, 1)[:, :, 3:]), st)
    new_xyz, new_points = U.sample_and_group(64, radius, 32, xyz, feat, start_idx=torch.from_numpy(st))
    assert np.array_equal(new_xyz.cpu().numpy(), w_xyz) and np.array_equal(new_points.cpu().numpy(), w_points)


def streamed_beside_fps(pts: np.ndarray, S: int, K: int, r: float):
    """Sampling from start 0 publishes its centroids while ball_query_stream answers them on a second stream; the follow-up
    query over the done flags completes the rest -> (oracle sampling, sampling, done flags, completed query)."""
    from pointnet12_b200 import ops

    dev = torch.device("cuda", 0)
    B, _, N = pts.shape
    xyz = views(cuda(pts, dev))[0]
    want_fps = orc.farthest_point_sample(xyz_of(pts), S, np.zeros(B, dtype=np.int64))
    grid = ops.ball_grid(xyz, r)
    fps_ctas, fps_smem = ops.fps_launch_info(B, N, S)
    ctas = (148 - fps_ctas) // B * B
    progress = torch.zeros((B, S), dtype=torch.int64, device=dev)
    done = torch.zeros((B, S), dtype=torch.int32, device=dev)
    out = torch.full((B, S, K), -7, dtype=torch.int64, device=dev)
    start = torch.zeros(B, dtype=torch.long, device=dev)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(dev)
    fps_idx = ops.fps(xyz, S, start, progress=progress)      # sampling first: its clusters need whole groups of free SMs
    with torch.cuda.stream(side):
        ops.ball_query_stream(r, K, xyz, grid, progress, done, out, ctas, 227 * 1024 - fps_smem + 1024)
    torch.cuda.synchronize()
    done_h = done.cpu().numpy()
    got = ops.ball_query(r, K, xyz, ops.index_points(xyz, fps_idx), grid=grid, done=done, out=out)
    return want_fps, fps_idx.cpu().numpy(), done_h, got.cpu().numpy()


def test_ball_query_streamed_beside_fps_on_lattice(dev):
    """The level-1 query fed by the running sampling kernel, on the lattice at r = 3/32 (ties in every sampling step, pairs
    on the radius); the streamed kernel answers rows itself, and with the follow-up query the result is the oracle's."""
    B, N, S, K, r = 4, 24000, 512, 32, R_LATTICE
    pts = syn.lattice_batch(B, N, seed=41)
    x = xyz_of(pts)
    want_fps, fps_idx, done, got = streamed_beside_fps(pts, S, K, r)
    assert np.array_equal(fps_idx, want_fps)
    q = np.ascontiguousarray(np.stack([x[b][want_fps[b]] for b in range(B)]))
    assert on_radius_pairs(x[:1], q[:1], r) > 100
    assert int(done.sum()) > 0, "the streamed kernel never ran beside the sampling kernel"
    assert np.array_equal(got, orc.query_ball_point(r, K, x, q))


@pytest.mark.parametrize("radius", [0.1, 0.2, 0.4, 0.8])
def test_ball_query_streamed_boundary_rows(dev, radius):
    """The streamed query derives its own threshold (ops.ball_query_stream): on the boundary sets, row 0 is the origin (start
    index 0) with 24 points on fp32(radius**2) and 24 one ulp above, where fp32(fp32(radius)**2) lies.  That row must come from
    the streamed kernel and equal the oracle's."""
    B, N, S, K = 4, 24000, 512, 32
    pts = syn.boundary_batch(B, N, radius, seed=int(radius * 100))
    x = xyz_of(pts)
    d = orc.square_distance(x[:, :1], x)[:, 0]
    r2 = np.float32(radius ** 2)
    above = np.nextafter(r2, np.float32(1))
    assert np.float32(np.float32(radius) ** 2) == above
    assert ((d == r2).sum(1) == 24).all() and ((d == above).sum(1) == 24).all()
    for b in range(B):       # the first K hits differ between the two thresholds
        assert not np.array_equal(np.flatnonzero(d[b] <= r2)[:K], np.flatnonzero(d[b] <= above)[:K])
    want_fps, fps_idx, done, got = streamed_beside_fps(pts, S, K, radius)
    assert np.array_equal(fps_idx, want_fps) and (want_fps[:, 0] == 0).all()
    assert (done[:, 0] == 1).all(), "row 0 was not answered by the streamed kernel"
    q = np.ascontiguousarray(np.stack([x[b][want_fps[b]] for b in range(B)]))
    assert np.array_equal(got, orc.query_ball_point(radius, K, x, q))


# ------------------------------------------------------------------------------------------------ 3-NN
@pytest.mark.parametrize("family", ["lattice", "few300", "flat", "offset"])
@pytest.mark.parametrize("S", [3, 31, 32, 33, 4096, 4097, 8192])
def test_three_nn_edge_clouds(dev, family, S):
    """scan and the block search (bucket-ordered, raw order, capped background grid) on S coarse points drawn from the fine
    cloud; S crosses the block-size switch (16 -> 32 points above 4096).  Indices equal the oracle's on every row, ties
    between the 3rd and 4th neighbour included; the weights are bit-identical between the methods."""
    from pointnet12_b200 import ops

    N, B = 12000, 2
    pts = cloud(family, B, N)
    x1 = xyz_of(pts)
    rng = np.random.default_rng(S)
    sel = np.stack([rng.choice(N, S, replace=False) for _ in range(B)])
    if family == "few300":       # coarse points 0 and 1: two copies of one point
        for b in range(B):
            twin = np.flatnonzero((x1[b] == x1[b][sel[b, 0]]).all(1))
            sel[b, 1] = twin[twin != sel[b, 0]][0]
    x2 = np.ascontiguousarray(np.stack([x1[b][sel[b]] for b in range(B)]))
    widx, ww, wd, tie = orc.three_nn(x1, x2)
    if family == "lattice":      # equal distances to distinct coarse points: in the top three, or between the 3rd and 4th
        assert (tie | (wd[..., 0] == wd[..., 1]) | (wd[..., 1] == wd[..., 2])).any() and (S == 3 or tie.any())
    elif family == "few300":
        assert all(len(np.unique(x2[b], axis=0)) < S for b in range(B))
    elif family == "flat":
        assert (np.ptp(x1[..., 2], axis=1) == 0).all()
    elif family == "offset":
        assert ((x1.astype(np.float64) ** 2).sum(-1) > 1e6).all()
    fine, coarse = views(cuda(pts, dev))[0], cuda(x2, dev)
    si, sw = ops.three_nn(fine, coarse, method="scan")
    assert np.array_equal(si.cpu().numpy(), widx)
    assert np.abs(sw.cpu().numpy() - ww).max() < 1e-6
    grid = ops.ball_grid(fine, 0.1)
    for order, background in ((grid, False), (None, False), (grid, True)):
        bi, bw = ops.three_nn(fine, coarse, order=order, method="blocks", background=background)
        assert torch.equal(bi, si) and torch.equal(bw, sw), (order is not None, background)


@pytest.mark.parametrize("block", ["8", "32"])
def test_three_nn_block_size_hook_on_edges(dev, block):
    """PN12_NN_BLOCK = 8 / 32 (own process: the hook is latched at first use) on the lattice and on 300 distinct points:
    the oracle's indices, ties included, and the scan's weights."""
    code = (
        "import torch, numpy as np\n"
        "from oracle import oracle as orc\n"
        "from pointnet12_b200 import ops, synthetic as syn\n"
        "dev = torch.device('cuda', 0)\n"
        "for pts in (syn.lattice_batch(2, 6000, seed=3), syn.few_distinct_batch(2, 6000, 300, seed=3)):\n"
        "    x = torch.from_numpy(pts).to(dev).permute(0, 2, 1)[:, :, :3]\n"
        "    xh = pts.transpose(0, 2, 1)[:, :, :3]\n"
        "    for S in (1024, 100):\n"
        "        c = np.ascontiguousarray(xh[:, np.random.default_rng(S).choice(6000, S, replace=False)])\n"
        "        widx = orc.three_nn(xh, c)[0]\n"
        "        cd = torch.from_numpy(c).to(dev)\n"
        "        bi, bw = ops.three_nn(x, cd, order=ops.ball_grid(x, 0.1), method='blocks')\n"
        "        si, sw = ops.three_nn(x, cd, method='scan')\n"
        "        assert torch.equal(bi, si) and torch.equal(bw, sw), S\n"
        "        assert np.array_equal(bi.cpu().numpy(), widx), S\n"
        "print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PN12_NN_BLOCK=block, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ consumers of the indices
def grouped_on_radius(x: np.ndarray, q: np.ndarray, idx: np.ndarray, radius: float) -> int:
    """Entries of the ball-query rows idx [B, S, K] whose oracle square_distance to their centroid is exactly fp32(radius**2)."""
    d = orc.square_distance(q, x)
    return int((np.take_along_axis(d, idx, axis=2) == np.float32(radius ** 2)).sum())


@pytest.mark.parametrize("family", ["lattice", "few3", "few300"])
def test_grouping_on_edge_indices(dev, family):
    """index_points / group (both channel orders) / sample_and_group / sample_and_group_all, bit-exact."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model import pointnet_util as U

    pts = cloud(family, 2, 4096)
    x = xyz_of(pts)
    feat = np.ascontiguousarray(pts.transpose(0, 2, 1)[:, :, 3:])
    st = np.array([1, 4095], dtype=np.int64)
    r = 0.1 if family != "lattice" else R_LATTICE
    w_xyz, w_points, w_fps, w_idx = orc.sample_and_group(512, r, 32, x, feat, st)
    if family.startswith("few"):
        assert (w_fps[:, int(family[3:]):] == 0).all()
    else:                        # grouped points on the radius, and rows padded with their first hit
        assert grouped_on_radius(x, w_xyz, w_idx, r) > 0 and (w_idx[..., -1] == w_idx[..., 0]).any()
    d_xyz, d_feat = views(cuda(pts, dev))
    assert np.array_equal(ops.index_points(d_xyz, cuda(w_fps, dev)).cpu().numpy(), orc.index_points(x, w_fps))
    for msg in (False, True):
        got = ops.group(d_xyz, d_feat, cuda(w_xyz, dev), cuda(w_idx, dev), msg_order=msg)
        assert np.array_equal(got.cpu().numpy(), orc.group(x, feat, w_xyz, w_idx, msg_order=msg))
    new_xyz, new_points = U.sample_and_group(512, r, 32, d_xyz, d_feat, start_idx=torch.from_numpy(st))
    assert np.array_equal(new_xyz.cpu().numpy(), w_xyz) and np.array_equal(new_points.cpu().numpy(), w_points)
    nx, allp = U.sample_and_group_all(d_xyz, d_feat)
    wx, wp = orc.sample_and_group_all(x, feat)
    assert np.array_equal(nx.cpu().numpy(), wx) and np.array_equal(allp.cpu().numpy(), wp)


@pytest.mark.parametrize("family", ["lattice", "few300"])
def test_chains_on_edge_indices(dev, family):
    """sa_mlp_max_tc on the ball-query indices and fp_mlp_tc on the 3-NN indices / weights of the edge clouds (repeated
    rows, padding with the first hit, equal weights of identical coarse points), within TC_TOL of the oracle."""
    from pointnet12_b200 import ops

    pts = cloud(family, 2, 4096)
    x = xyz_of(pts)
    feat = np.ascontiguousarray(pts.transpose(0, 2, 1)[:, :, 3:])
    r = 0.1 if family != "lattice" else R_LATTICE
    q, _, fps_idx, gidx = orc.sample_and_group(512, r, 32, x, feat, np.array([0, 9]))
    B, S, K = gidx.shape
    idx, w, _, tie = orc.three_nn(x, q)
    if family == "lattice":      # ball rows with points on the radius, 3-NN rows with a tie between the 3rd and 4th
        assert grouped_on_radius(x, q, gidx, r) > 0 and tie.any()
    else:                        # sampling ran out: repeated centroids, so equal weights of identical coarse points
        assert (fps_idx[:, 300:] == 0).all() and (w[..., 0] == w[..., 1]).any()
    layers = _rand_layers([(4, 64), (64, 64), (64, 128)], seed=3)
    g = orc.group(x, feat, q, gidx, msg_order=False)
    want = orc.group_max(orc.linear(orc.linear(orc.linear(g.reshape(B * S * K, -1), *layers[0][:2], None, True),
                                               *layers[1][:2], None, True), *layers[2][:2], None, True), K).reshape(B, S, -1)
    chain = ops.PackedChain([(cuda(w, dev), cuda(b, dev), rl) for w, b, rl in layers])
    got = ops.sa_mlp_max_tc(chain, cuda(x, dev), cuda(feat, dev), cuda(q, dev), cuda(gidx, dev), False)
    assert rel_err(got, want) < TC_TOL
    p2 = np.random.default_rng(1).normal(size=(B, S, 64)).astype(np.float32)
    fl = _rand_layers([(65, 128), (128, 64)], seed=4)
    rows = np.concatenate([feat, orc.three_interpolate(p2, idx, w)], -1).reshape(B * x.shape[1], -1)
    want = orc.linear(orc.linear(rows, *fl[0][:2], None, True), *fl[1][:2], None, True).reshape(B, x.shape[1], -1)
    chain = ops.PackedChain([(cuda(wt, dev), cuda(b, dev), rl) for wt, b, rl in fl])
    got = ops.fp_mlp_tc(chain, cuda(feat, dev), cuda(p2, dev), cuda(idx, dev), cuda(w, dev), ops.OUT_ROWS)
    assert rel_err(got, want) < TC_TOL


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("family", ["few3", "few300", "flat", "lattice"])
def test_semseg_edge_clouds_vs_oracle(dev, ckpt_state, ckpt_path, family):
    """PointNet2SemSeg eval forward (B = 2, N = 4096): the sampling, ball-query and 3-NN indices of every level, taken from
    the primitives level by level with the same starts, equal the oracle's trace bit for bit; log-probs within 1e-3."""
    from pointnet12_b200 import ops
    from pointnet12_b200.model.utils import load_pointnet

    B, N = 2, 4096
    pts = cloud(family, B, N)
    rng = np.random.default_rng(N)
    st = [rng.integers(0, n, B) for n in (N, 1024, 256, 64)]
    trace = {}
    want = orc.pointnet2_semseg(ckpt_state, pts, st, trace)
    if family.startswith("few"):
        assert (trace["sa1.fps_idx"][:, int(family[3:]):] == 0).all()
    if family == "lattice":
        assert trace["fp1.nn_tie"].any()
    cur = views(cuda(pts, dev))[0]
    xs = [cur]
    for lvl, (npoint, radius) in enumerate([(1024, 0.1), (256, 0.2), (64, 0.4), (16, 0.8)], 1):
        fps = ops.fps(cur, npoint, cuda(st[lvl - 1], dev))
        assert np.array_equal(fps.cpu().numpy(), trace[f"sa{lvl}.fps_idx"]), f"sampling, level {lvl}"
        new_xyz = ops.index_points(cur, fps)
        ball = ops.ball_query(radius, 32, cur, new_xyz)
        assert np.array_equal(ball.cpu().numpy(), trace[f"sa{lvl}.group_idx"]), f"ball query, level {lvl}"
        cur = new_xyz
        xs.append(cur)
    grid = ops.ball_grid(xs[0], 0.1)
    for name, (a, b) in (("fp4", (3, 4)), ("fp3", (2, 3)), ("fp2", (1, 2)), ("fp1", (0, 1))):
        idx, _ = ops.three_nn(xs[a], xs[b], order=grid if a == 0 else None)
        assert np.array_equal(idx.cpu().numpy(), trace[name + ".nn_idx"]), name
    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    with torch.no_grad():
        got = net(cuda(pts, dev), fps_starts=[cuda(s, dev) for s in st]).cpu().numpy()
    assert rel_err(got, want) < LOGP_TOL


def test_graphed_deep_pipeline_on_lattice(dev, ckpt_path):
    """GraphedSemSeg(depth = 8) -- level-1 sampling on 2 CTAs per cloud holding the cloud in registers, the level-1 query
    after sampling -- torch.equal to the sequential runner on 24000-point lattice batches."""
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    net = load_pointnet("pointnet2", 19, ckpt_path, device=dev)
    deep = GraphedSemSeg(net, depth=8)
    assert deep.fps1_shape(24000) == (2, 256, 2)
    xs = [cuda(syn.lattice_batch(4, 24000, seed=50 + i), dev) for i in range(3)]
    torch.manual_seed(4)
    want = GraphedSemSeg(net, depth=1).run_pipelined(xs)
    torch.manual_seed(4)
    got = deep.run_pipelined(xs)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ function-level API
@pytest.mark.parametrize("family", ["offset", "lattice"])
def test_square_distance_edges(dev, family):
    from pointnet12_b200.model import pointnet_util as U

    pts = cloud(family, 2, 4096)
    x = xyz_of(pts)
    a, b = np.ascontiguousarray(x[:, :300]), x[:, 1000:3000]
    got = U.square_distance(cuda(a, dev), views(cuda(pts, dev))[0][:, 1000:3000]).cpu().numpy()
    assert np.array_equal(got, orc.square_distance(a, b))


def test_chamfer_argmin_first_of_equal_minima(dev):
    """On the lattice every distance is exact, so equal minima are real: chamfer_argmin returns the first of them."""
    from pointnet12_b200 import ops

    x = xyz_of(syn.lattice_batch(2, 6000, seed=8))
    p1 = np.ascontiguousarray(x[:, :2000] + np.float32(syn.LATTICE_STEP / 2))     # between the sites: many equal minima
    p2 = np.ascontiguousarray(x[:, 2000:])
    d = ((p1[:, :, None, :].astype(np.float64) - p2[:, None].astype(np.float64)) ** 2).sum(-1)
    want = d.argmin(-1)
    assert ((d == d.min(-1, keepdims=True)).sum(-1) > 1).mean() > 0.1
    _, got = ops.chamfer_argmin(cuda(p1, dev), cuda(p2, dev))
    assert np.array_equal(got.cpu().numpy(), want)
