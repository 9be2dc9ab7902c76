"""Synthetic input clouds for parity tests and benchmarks (no dataset ships with the repo).

`kitti_cloud` makes a "KITTI-shaped" scan as SURVEY.md section 8(d) defines it: rays cast from the
sensor origin inside the reference's "inview" field of view (azimuth +-40 deg, `kitti_utils.py:222`;
HDL-64 elevation span) against a ground plane, two side walls and a dozen boxes, then the reference's
normalisation (`data_utils/SemKITTI_Loader.py:23-30`: x/70, y/70, z/3, (refl-0.5)*2, clip to [-1,1])
and its resample-with-replacement to a fixed point budget (`SemKITTI_Loader.py:110-113`), which is
what creates the duplicate points / distance ties the sampling kernels must break like the reference.

Only numpy is used so the same arrays can be rebuilt anywhere from a seed; the golden fixtures under
tests/golden/ store a checksum of the inputs they were generated from.
"""
from __future__ import annotations

import hashlib

import numpy as np

SENSOR_HEIGHT = 1.73   # metres above the ground plane
MAX_RANGE = 80.0


def _ray_scene_depth(dirs: np.ndarray, rng: np.random.Generator) -> np.ndarray:
    """Distance along each unit ray to the first surface of a random street scene."""
    n = dirs.shape[0]
    t = np.full(n, MAX_RANGE, dtype=np.float64)
    dx, dy, dz = dirs[:, 0], dirs[:, 1], dirs[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        # ground plane z = -SENSOR_HEIGHT
        tg = np.where(dz < 0, -SENSOR_HEIGHT / dz, np.inf)
        t = np.minimum(t, tg)
        # two side walls
        yl = rng.uniform(6.0, 15.0)
        yr = -rng.uniform(6.0, 15.0)
        tl = np.where(dy > 0, yl / dy, np.inf)
        tr = np.where(dy < 0, yr / dy, np.inf)
        t = np.minimum(t, np.minimum(tl, tr))
        # 12 axis-aligned boxes standing on the ground (slab test)
        for _ in range(12):
            cx = rng.uniform(5.0, 60.0)
            cy = rng.uniform(-6.0, 6.0)
            sx = rng.uniform(0.3, 4.5)
            sy = rng.uniform(0.3, 2.0)
            sz = rng.uniform(1.2, 4.0)
            lo = np.array([cx - sx / 2, cy - sy / 2, -SENSOR_HEIGHT])
            hi = np.array([cx + sx / 2, cy + sy / 2, -SENSOR_HEIGHT + sz])
            t0 = lo[None, :] / dirs
            t1 = hi[None, :] / dirs
            tn = np.minimum(t0, t1).max(axis=1)
            tf = np.maximum(t0, t1).min(axis=1)
            hit = (tn <= tf) & (tf > 0) & (tn > 0)
            t = np.where(hit, np.minimum(t, tn), t)
    return t


def kitti_cloud(n_points: int, seed: int) -> np.ndarray:
    """One normalised scan, shape [4, n_points] float32 = (x/70, y/70, z/3, (refl-0.5)*2)."""
    rng = np.random.default_rng(seed)
    az = np.deg2rad(rng.uniform(-40.0, 40.0, n_points))
    el = np.deg2rad(rng.uniform(-24.8, 2.0, n_points))
    dirs = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], axis=1)
    depth = _ray_scene_depth(dirs, rng)
    pts = dirs * depth[:, None] + rng.normal(0.0, 0.02, (n_points, 3))
    refl = rng.beta(2.0, 5.0, n_points)
    pcd = np.concatenate([pts, refl[:, None]], axis=1).astype(np.float32)
    # reference normalisation (SemKITTI_Loader.py:23-30)
    pcd[:, 0] /= 70
    pcd[:, 1] /= 70
    pcd[:, 2] /= 3
    pcd[:, 3] = (pcd[:, 3] - 0.5) * 2
    pcd = np.clip(pcd, -1, 1)
    # resample with replacement to the fixed budget (SemKITTI_Loader.py:110-113)
    choice = rng.choice(n_points, n_points, replace=True)
    pcd = pcd[choice]
    return np.ascontiguousarray(pcd.T, dtype=np.float32)


def kitti_batch(batch: int, n_points: int, config: int = 2, first: int = 0) -> np.ndarray:
    """[B, 4, N] float32 batch; cloud b of config c uses seed 1000*c + b (SURVEY.md section 8d)."""
    return np.stack([kitti_cloud(n_points, 1000 * config + first + b) for b in range(batch)], axis=0)


def modelnet_batch(batch: int, n_points: int = 1024, seed: int = 4000) -> np.ndarray:
    """[B, 3, N] float32: Gaussian blobs scaled into the unit sphere (ModelNet40-shaped, config C4)."""
    rng = np.random.default_rng(seed)
    pts = rng.normal(0.0, 1.0, (batch, n_points, 3))
    pts /= np.linalg.norm(pts, axis=2).max(axis=1)[:, None, None]
    return np.ascontiguousarray(pts.transpose(0, 2, 1), dtype=np.float32)


# ------------------------------------------------------------------------------------------------ clouds at the geometry edges
# Inputs built to reach the decisions where the sampling, ball-query and 3-NN kernels can go wrong: ties between DISTINCT
# points, points exactly on the radius, sampling that runs out of distinct points, zero extent along an axis, large |p|^2 in
# the expansion formula and points beyond the reference's initial FPS distance of 1e10 (pointnet_util.py:74).
LATTICE_STEP = 2.0 ** -5


def lattice_batch(batch: int, n_points: int, side: int = 29, seed: int = 0) -> np.ndarray:
    """[B, 4, N]: N distinct sites of the integer lattice {-side//2 .. side-1-side//2}^3 scaled by 2^-5, in shuffled index
    order; the 4th channel is uniform in [-1, 1).  Every coordinate is k / 32 with |k| < 32, so the reference's distance
    formulas are exact in fp32 (equal to float64): ties between distinct points are real, and r**2 is exact for r = k / 32."""
    if n_points > side ** 3:
        raise ValueError(f"a {side}^3 lattice has fewer than {n_points} sites")
    rng = np.random.default_rng(seed)
    out = np.empty((batch, 4, n_points), dtype=np.float32)
    for b in range(batch):
        site = rng.choice(side ** 3, n_points, replace=False)
        ijk = np.stack([site % side, site // side % side, site // side ** 2], axis=0) - side // 2
        out[b, :3] = ijk * LATTICE_STEP
        out[b, 3] = rng.uniform(-1.0, 1.0, n_points)
    return out


def few_distinct_batch(batch: int, n_points: int, distinct: int, seed: int = 0) -> np.ndarray:
    """[B, 4, N]: `distinct` different points (uniform in [-1, 1)^4) resampled to N, each of them present at least once."""
    rng = np.random.default_rng(seed)
    out = np.empty((batch, 4, n_points), dtype=np.float32)
    for b in range(batch):
        base = rng.uniform(-1.0, 1.0, (4, distinct)).astype(np.float32)
        pick = np.concatenate([np.arange(distinct), rng.integers(0, distinct, n_points - distinct)])
        out[b] = base[:, rng.permutation(pick)]
    return out


def flat_batch(batch: int, n_points: int, axes: str = "z", config: int = 30) -> np.ndarray:
    """kitti_batch with the coordinates named in `axes` ("z": a plane, "yz": a line) set to one constant per axis."""
    out = kitti_batch(batch, n_points, config=config)
    for a in axes:
        out[:, "xyz".index(a)] = np.float32(-0.375 if a == "z" else 0.125)
    return out


def offset_batch(batch: int, n_points: int, config: int = 31) -> np.ndarray:
    """kitti_batch back in metres (x 70, y 70, z 3) and shifted by +1000 m in x: |p|^2 ~ 1e6, so the expansion formula of
    the reference's square_distance cancels and rounds by ~0.1 m^2."""
    out = kitti_batch(batch, n_points, config=config)
    out[:, 0] = out[:, 0] * np.float32(70) + np.float32(1000)
    out[:, 1] *= np.float32(70)
    out[:, 2] *= np.float32(3)
    return out


OUTLIER_FAR = (2.0e5, 3.0e5)


def outlier_batch(batch: int, n_points: int, config: int = 32) -> np.ndarray:
    """kitti_batch with 4 points moved to |p| ~ 1e3 and two to x = -2e5 and x = +3e5, the nearer one at the lower index.
    Both far points are more than 1e5 from any start point, so their squared distance exceeds the reference's initial
    1e10 (pointnet_util.py:74): after the first pick the running minimum caps both at 1e10 and the tie goes to the lower
    index, where an uncapped kernel would take the farther point."""
    out = kitti_batch(batch, n_points, config=config)
    rng = np.random.default_rng(config)
    for b in range(batch):
        pos = rng.choice(n_points, 6, replace=False)
        d = rng.normal(size=(3, 4))
        out[b, :3, pos[:4]] = (1000.0 * d / np.linalg.norm(d, axis=0)).T.astype(np.float32)
        lo, hi = np.sort(pos[4:])
        out[b, :3, lo] = np.float32([-OUTLIER_FAR[0], 0.0, 0.0])
        out[b, :3, hi] = np.float32([OUTLIER_FAR[1], 0.0, 0.0])
    return out


def boundary_batch(batch: int, n_points: int, radius: float, per_level: int = 24, seed: int = 0) -> np.ndarray:
    """[B, 4, N] for a ball query centred at the ORIGIN, which is point 0 of every cloud: `per_level` points each whose
    squared norm ((x*x + y*y) + z*z in fp32 -- the reference's square_distance from the origin) is exactly fp32(radius**2),
    one ulp below it and one ulp above it, and background points farther than 2 * radius.  The fine structure decides
    membership: `sqrdists > radius ** 2` (pointnet_util.py:102) keeps the first two levels and drops the third, and a
    threshold of fp32(fp32(radius) ** 2) -- one ulp higher at radius 0.1, 0.2, 0.4 and 0.8 -- would keep all three."""
    rng = np.random.default_rng(seed)
    r2 = np.float32(radius ** 2)
    targets = (np.nextafter(r2, np.float32(0)), r2, np.nextafter(r2, np.float32(1e30)))
    out = np.empty((batch, 4, n_points), dtype=np.float32)
    for b in range(batch):
        pts = []
        for t in targets:
            for _ in range(per_level):
                pts.append(_on_sphere(float(radius), t, rng))
        pts = np.array(pts, dtype=np.float32)
        nb = n_points - 1 - len(pts)
        d = rng.normal(size=(nb, 3))
        far = d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(2.0 * radius + 0.05, 2.0 * radius + 1.0, (nb, 1))
        xyz = np.concatenate([pts, far.astype(np.float32)])[rng.permutation(n_points - 1)]
        out[b, :3, 0] = 0.0
        out[b, :3, 1:] = xyz.T
        out[b, 3] = rng.uniform(-1.0, 1.0, n_points)
    return out


def sqnorm_f32(p) -> np.float32:
    """(x*x + y*y) + z*z rounded like the reference's fp32 tensor ops."""
    x, y, z = (np.float32(v) for v in p)
    return np.float32(np.float32(x * x + y * y) + np.float32(z * z))


def _on_sphere(radius: float, target: np.float32, rng: np.random.Generator) -> np.ndarray:
    """A point with sqnorm_f32(p) == target exactly: random x, y, then z found among the floats next to the real root."""
    while True:
        u = rng.normal(size=3)
        u *= radius / np.linalg.norm(u)
        x, y = np.float32(u[0]), np.float32(u[1])
        xy = np.float32(x * x + y * y)
        if not float(xy) < 0.9 * float(target):
            continue
        z = np.float32(np.sqrt(float(target) - float(xy)))
        for _ in range(64):
            s = sqnorm_f32((x, y, z))
            if s == target:
                return np.array([x, y, z if u[2] >= 0 else -z], dtype=np.float32)
            z = np.nextafter(z, np.float32(1e30) if s < target else np.float32(0))


def checksum(arr: np.ndarray) -> str:
    """Stable digest of an array's bytes (dtype and shape included)."""
    h = hashlib.sha256()
    h.update(str(arr.dtype).encode())
    h.update(str(arr.shape).encode())
    h.update(np.ascontiguousarray(arr).tobytes())
    return h.hexdigest()[:16]


def random_state_dict(shapes: dict, seed: int) -> dict:
    """Deterministic weights for nets whose checkpoint is not shipped (PointNetSeg, PointNet2ClsMsg).

    `shapes` maps state_dict names to shapes.  Values depend only on (sorted name order, seed), not on
    module construction order, so the reference model (oracle/gen_golden.py), the oracle and the CUDA
    modules all get identical numbers.  BatchNorm running statistics are perturbed away from their
    (0, 1) defaults so that BN folding is actually exercised (SURVEY.md section 8a-11).
    """
    rng = np.random.default_rng(seed)
    out = {}
    for name in sorted(shapes):
        shape = tuple(shapes[name])
        leaf = name.rsplit(".", 1)[-1]
        if leaf == "num_batches_tracked":
            out[name] = np.zeros(shape, dtype=np.int64)
        elif leaf == "running_mean":
            out[name] = rng.normal(0.0, 0.1, shape).astype(np.float32)
        elif leaf == "running_var":
            out[name] = rng.uniform(0.5, 1.5, shape).astype(np.float32)
        elif leaf == "weight" and len(shape) == 1:          # BatchNorm gamma
            out[name] = rng.uniform(0.5, 1.5, shape).astype(np.float32)
        elif leaf == "weight":                              # conv / linear: fan-in scaled uniform
            fan_in = int(np.prod(shape[1:]))
            bound = float(np.sqrt(3.0 / fan_in))
            out[name] = rng.uniform(-bound, bound, shape).astype(np.float32)
        else:                                               # biases (conv, linear, BatchNorm beta)
            out[name] = rng.normal(0.0, 0.1, shape).astype(np.float32)
    return out


# SemanticKITTI raw label id -> training class 0..19 (0 = ignored): the `learning_map` table of the dataset's public
# semantic-kitti.yaml, which the reference reads at data_utils/kitti_utils.py:152-155.
SEMANTIC_KITTI_LEARNING_MAP = {
    0: 0, 1: 0, 10: 1, 11: 2, 13: 5, 15: 3, 16: 5, 18: 4, 20: 5, 30: 6, 31: 7, 32: 8, 40: 9, 44: 10, 48: 11, 49: 12, 50: 13,
    51: 14, 52: 0, 60: 9, 70: 15, 71: 16, 72: 17, 80: 18, 81: 19, 99: 0, 252: 1, 253: 7, 254: 6, 255: 8, 256: 5, 257: 5,
    258: 4, 259: 5}


def raw_scan(n_points: int, seed: int):
    """A synthetic RAW SemanticKITTI scan in the dataset's wire format: points [M, 4] float32 (x, y, z in metres over the
    full 360 degrees, reflectance in [0, 1]) and labels [M] uint32 (semantic id in the low 16 bits, instance id above).
    Points whose azimuth / elevation lies within 1e-5 rad of a field-of-view bound of the in-view filter (+-40, +-20 degrees)
    get label 0 (dropped by every implementation), so the filter decision never hinges on the last ulp of atan2."""
    rng = np.random.default_rng(seed)
    az = np.deg2rad(rng.uniform(-180.0, 180.0, n_points))
    el = np.deg2rad(rng.uniform(-24.8, 24.0, n_points))
    r = rng.uniform(1.5, 80.0, n_points)
    pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el),
                    rng.uniform(0.0, 1.0, n_points)], axis=1).astype(np.float32)
    ids = np.array(sorted(SEMANTIC_KITTI_LEARNING_MAP), dtype=np.uint32)
    sem = ids[rng.integers(0, len(ids), n_points)]
    x, y, z = (pts[:, i].astype(np.float64) for i in range(3))
    h, v = np.arctan2(y, x), np.arctan2(z, np.sqrt(x * x + y * y + z * z))
    edge = np.zeros(n_points, dtype=bool)
    for ang, bound in ((h, 40.0), (h, -40.0), (v, 20.0), (v, -20.0)):
        edge |= np.abs(ang - np.deg2rad(bound)) < 1e-5
    sem[edge] = 0
    inst = rng.integers(0, 200, n_points).astype(np.uint32)
    return pts, (sem | (inst << 16)).astype(np.uint32)
