"""The edge clouds of pointnet12_b200/synthetic.py reach the edges they are built for (checked with the CPU oracle), and on the
lattice, where fp32 arithmetic is exact, the oracle agrees with a plain float64 restatement of the reference's sampling,
ball query and 3-NN with its tie rules: the first maximum (pointnet_util.py:83), ascending index (:102-106) and
(distance, index) (:295-297).  tests/test_gpu_geometry_edges.py runs the CUDA kernels on the same clouds."""
import numpy as np
import pytest

from oracle import oracle as orc
from pointnet12_b200 import synthetic as syn

RADII = (0.1, 0.2, 0.4, 0.8)


def xyz_of(pts: np.ndarray) -> np.ndarray:
    """[B, 4, N] -> point-major xyz view [B, N, 3]."""
    return pts.transpose(0, 2, 1)[:, :, :3]


# ------------------------------------------------------------------------------------------------ float64 restatements
def fps64(xyz: np.ndarray, npoint: int, start: int):
    """pointnet_util.py:63-84 in float64 for one cloud -> (indices, steps whose maximum is shared by DISTINCT points)."""
    p = xyz.astype(np.float64)
    dist = np.full(len(p), 1e10)
    far, out, ties = int(start), [], 0
    for _ in range(npoint):
        out.append(far)
        dist = np.minimum(dist, ((p - p[far]) ** 2).sum(1))
        best = np.flatnonzero(dist == dist.max())
        ties += len(np.unique(p[best], axis=0)) > 1
        far = int(best[0])
    return np.array(out), ties


def ball64(xyz: np.ndarray, q: np.ndarray, radius: float, K: int) -> np.ndarray:
    """pointnet_util.py:87-107 in float64 for one cloud: first K points with d <= radius**2 in index order, padded with the
    first (N if none)."""
    d = ((q[:, None, :].astype(np.float64) - xyz[None].astype(np.float64)) ** 2).sum(-1)
    out = np.empty((len(q), K), dtype=np.int64)
    for s in range(len(q)):
        hit = np.flatnonzero(d[s] <= np.float32(radius ** 2))[:K]
        first = hit[0] if len(hit) else len(xyz)
        out[s] = np.concatenate([hit, np.full(K - len(hit), first)])
    return out


def nn64(xyz1: np.ndarray, xyz2: np.ndarray):
    """The 3 nearest of xyz2 for every point of xyz1 ordered by (distance, index) in float64 -> (idx [N, 3], tie [N]: the 3rd
    and the 4th nearest are at the same distance)."""
    d = ((xyz1[:, None, :].astype(np.float64) - xyz2[None].astype(np.float64)) ** 2).sum(-1)
    order = np.argsort(d, axis=1, kind="stable")
    tie = np.take_along_axis(d, order[:, 2:3], 1)[:, 0] == np.take_along_axis(d, order[:, 3:4], 1)[:, 0] \
        if xyz2.shape[0] > 3 else np.zeros(len(xyz1), dtype=bool)
    return order[:, :3], tie


def on_radius_pairs(xyz: np.ndarray, q: np.ndarray, radius: float) -> int:
    """Pairs whose oracle square_distance is exactly fp32(radius**2)."""
    return int((orc.square_distance(q, xyz) == np.float32(radius ** 2)).sum())


# ------------------------------------------------------------------------------------------------ the edges are there
@pytest.fixture(scope="module")
def lattice():
    return syn.lattice_batch(2, 24000, seed=0)


def test_lattice_is_exact_and_distinct(lattice):
    x = xyz_of(lattice)
    for b in range(2):
        assert len(np.unique(x[b], axis=0)) == 24000
        assert np.array_equal(np.round(x[b] / syn.LATTICE_STEP) * syn.LATTICE_STEP, x[b])
    sq = orc.square_distance(x[:1, :300], x[:1])[0].astype(np.float64)
    exact = ((x[0, :300, None, :].astype(np.float64) - x[0, None].astype(np.float64)) ** 2).sum(-1)
    assert np.array_equal(sq, exact)


def test_lattice_fps_ties_between_distinct_points(lattice):
    x = xyz_of(lattice)
    got, ties = fps64(x[0], 1024, 17)
    assert ties > 900                        # almost every step has several distinct points at the maximum
    assert np.array_equal(orc.farthest_point_sample(x[:1], 1024, np.array([17])), got[None])


def test_lattice_ball_query_on_radius(lattice):
    x = xyz_of(lattice)
    r = 3 * syn.LATTICE_STEP
    assert np.float32(r ** 2) == np.float32(np.float32(r) ** 2) == r ** 2
    q = x[:1, :200]
    assert on_radius_pairs(x[:1], q, r) > 200
    for K in (1, 32, 128):
        assert np.array_equal(orc.query_ball_point(r, K, x[:1], q)[0], ball64(x[0], q[0], r, K))


def test_lattice_three_nn_ties(lattice):
    x = xyz_of(lattice)
    fine = x[0, :6000]
    coarse = np.ascontiguousarray(x[0, orc.farthest_point_sample(x[:1], 512, np.array([0]))[0]])
    widx, _, _, tie = orc.three_nn(fine[None], coarse[None])
    idx64, tie64 = nn64(fine, coarse)
    assert np.array_equal(widx[0], idx64)
    assert np.array_equal(tie[0], tie64)
    assert tie64.mean() > 0.05


def test_radius_squared_differs_from_squared_fp32_radius():
    for r in RADII:
        assert np.float32(r ** 2) != np.float32(np.float32(r) ** 2), r


@pytest.mark.parametrize("radius", RADII)
def test_boundary_set_straddles_the_radius(radius):
    pts = syn.boundary_batch(2, 4096, radius, seed=1)
    x = xyz_of(pts)
    assert (x[:, 0] == 0).all()
    d = orc.square_distance(x[:, :1], x)[:, 0]
    r2 = np.float32(radius ** 2)
    below, above = np.nextafter(r2, np.float32(0)), np.nextafter(r2, np.float32(1))
    for b in range(2):
        assert [(d[b] == v).sum() for v in (below, r2, above)] == [24, 24, 24]
        assert (d[b][d[b] > above] > 4 * radius ** 2).all()
    ball = orc.query_ball_point(radius, 128, x, x[:, :1])
    for b in range(2):
        assert len(set(ball[b, 0])) == 1 + 48 and not (d[b][ball[b, 0]] > r2).any()


@pytest.mark.parametrize("m", [1, 3, 300])
def test_few_distinct_exhausts_sampling(m):
    pts = syn.few_distinct_batch(2, 4096, m, seed=m)
    x = xyz_of(pts)
    assert all(len(np.unique(pts[b].T, axis=0)) == m for b in range(2))
    idx = orc.farthest_point_sample(x, 1024, np.array([5, 4000]))
    assert all(len(np.unique(x[b][idx[b]], axis=0)) == m for b in range(2))
    assert (idx[:, m:] == 0).all()           # every distance is 0: the first maximum is index 0


@pytest.mark.parametrize("axes", ["z", "yz"])
def test_flat_clouds_have_zero_extent(axes):
    x = xyz_of(syn.flat_batch(2, 4096, axes))
    for a in range(3):
        assert (np.ptp(x[..., a], axis=1) == 0).all() == ("xyz"[a] in axes)


def test_offset_cloud_has_large_norms():
    x = xyz_of(syn.offset_batch(2, 4096))
    n2 = (x.astype(np.float64) ** 2).sum(-1)
    assert n2.min() > 1e6 and np.ptp(x[..., 0], axis=1).min() > 20
    # the expansion formula is off the exact squared distance by much more than a small radius squared
    q = x[:, :64]
    err = np.abs(orc.square_distance(q, x).astype(np.float64)
                 - ((q[:, :, None, :].astype(np.float64) - x[:, None].astype(np.float64)) ** 2).sum(-1))
    assert err.max() > 0.05


def test_outlier_beyond_the_initial_distance():
    pts = syn.outlier_batch(2, 24000)
    x = xyz_of(pts)
    st = np.array([3, 20000])
    for b in range(2):
        far = np.flatnonzero(np.abs(x[b, :, 0]) >= syn.OUTLIER_FAR[0])
        assert len(far) == 2 and x[b, far[0], 0] < 0 < x[b, far[1], 0]
        assert (((x[b, far] - x[b, st[b]]).astype(np.float64) ** 2).sum(-1) > 1e10).all()
        mid = np.linalg.norm(x[b].astype(np.float64), axis=1)
        assert ((mid > 900) & (mid < 1100)).sum() == 4
    idx = orc.farthest_point_sample(x, 8, st)
    for b in range(2):           # capped at 1e10, both far points tie and the lower index (the nearer one) wins
        assert x[b, idx[b, 1], 0] == -syn.OUTLIER_FAR[0] and x[b, idx[b, 2], 0] == syn.OUTLIER_FAR[1]
