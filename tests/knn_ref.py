"""CPU reference and adversarial clouds for the kNN + covariance kernels (csrc/knn_cov.cu, csrc/grid_search.cuh).  Test
infrastructure only.

`raw_cov_from_list` restates the covariance kernel's statistics (cov_point) in numpy float64, summing in the order of a
given neighbour list.  numpy float64 arithmetic is unfused and knn_cov.cu is compiled with -fmad=false, so applied to the
GPU's own neighbour list (ngicp_cov_neighbors) it reproduces the unregularised covariances bit for bit.

`knn_distances` gives the exact ascending k nearest squared distances (nanoflann's metric, float32).

The generators build seeded clouds, each aimed at a branch of the kernels that ordinary voxelised scans almost never
reach.  They return (n, 8) float32 PointXYZI records; `O` is the oracle module (oracle/oracle.py).
"""
import numpy as np

from direct_lidar_odometry_b200 import synth

BRUTE_MAX_POINTS = 30000   # above this, distances come from the kd-tree (checked against brute force on a sample)
TILE_MIN_POINTS = 131072   # knn_tile_min_points: AUTO runs clouds from this size on the tile path


def raw_cov_from_list(xyz, idx) -> np.ndarray:
    """Unregularised covariance of each row's neighbour list, (m, 6) float64 = xx, xy, xz, yy, yz, zz.

    cov_point restated: mean = sum(x) / k in list order; then sum((x - mean)(x - mean)^T) / k in list order, as six
    upper-triangle terms.  A -1 entry counts as a zero column minus the mean (what the reference's zero-initialised
    neighbour matrix holds)."""
    p = np.asarray(xyz, dtype=np.float32)[:, :3].astype(np.float64)
    idx = np.asarray(idx)
    m, k = idx.shape
    valid = idx >= 0
    cols = [np.where(valid[:, j, None], p[np.where(valid[:, j], idx[:, j], 0)], 0.0) for j in range(k)]
    mean = np.zeros((m, 3))
    for c in cols:
        mean = mean + c
    mean = mean / float(k)
    acc = np.zeros((m, 6))
    for c in cols:
        d = c - mean
        x, y, z = d[:, 0], d[:, 1], d[:, 2]
        acc = acc + np.stack([x * x, x * y, x * z, y * y, y * z, z * z], axis=1)
    return acc / float(k)


def cov6(covs) -> np.ndarray:
    """The six upper-triangle terms of (n, 4, 4) or (n, 3, 3) covariance matrices."""
    c = np.asarray(covs)
    return np.stack([c[:, 0, 0], c[:, 0, 1], c[:, 0, 2], c[:, 1, 1], c[:, 1, 2], c[:, 2, 2]], axis=1)


def sqdist_f32(q, p) -> np.ndarray:
    """nanoflann's squared distance in float32, in its order: (dx*dx + dy*dy) + dz*dz, unfused."""
    q = np.asarray(q, dtype=np.float32)
    p = np.asarray(p, dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        dx, dy, dz = q[..., 0] - p[..., 0], q[..., 1] - p[..., 1], q[..., 2] - p[..., 2]
        return (dx * dx + dy * dy) + dz * dz


def knn_distances(O, xyz, queries, k, sample: int = 512, seed: int = 0) -> np.ndarray:
    """Exact ascending k nearest squared distances (nq, k) of `queries` in the finite cloud `xyz` (-1 past the cloud's
    size, like nanoflann's short result).  Brute force up to BRUTE_MAX_POINTS points; above, the oracle's kd-tree, whose
    distances are checked bit for bit against brute force on a seeded sample of the queries."""
    q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32)[:, :3])
    if xyz.shape[0] <= BRUTE_MAX_POINTS:
        return O.Cloud(xyz, backend=O.BACKEND_BRUTE).knn(q, k)[1]
    d2 = O.Cloud(xyz).knn(q, k)[1]
    pick = np.random.default_rng(seed).choice(q.shape[0], size=min(sample, q.shape[0]), replace=False)
    ref = O.Cloud(xyz, backend=O.BACKEND_BRUTE).knn(q[pick], k)[1]
    if not np.array_equal(d2[pick].view(np.uint32), ref.view(np.uint32)):
        raise AssertionError("kd-tree distances differ from brute force")
    return d2


# ------------------------------------------------------------------------------------------------ generators
def _xyzi(p) -> np.ndarray:
    p = np.asarray(p, dtype=np.float32)
    out = np.zeros((p.shape[0], 8), dtype=np.float32)
    out[:, :3] = p[:, :3]
    out[:, 3] = 1.0
    return out


def _shuffled(cloud, seed):
    """Original indices in random order, so that index order and cell order disagree (ties are broken by sorted slot)."""
    return np.ascontiguousarray(cloud[np.random.default_rng(seed).permutation(cloud.shape[0])])


def scan(O, i: int = 0, leaf: float = 0.25) -> np.ndarray:
    """A synthetic OS1-64 scan, crop-boxed and voxelised (sensor frame), as DLO feeds S2S."""
    T = synth.trajectory_pose(i)
    return O.voxel_filter(synth.crop_box_negative(synth.os1_like(i, T)), leaf)


def lattice(nx: int = 60, ny: int = 60, nz: int = 8, step: float = 0.1, seed: int = 1) -> np.ndarray:
    """Integer grid x 0.1 m: exact distance ties at almost every point, at the k-th place and inside the k list.
    Targets the tile kernel's tie hand-off to the warp search, the lattice-order fix-ups (cov_rest_kernel), and the
    shared fb_list filling from both ends."""
    g = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), axis=-1).reshape(-1, 3)
    return _shuffled(_xyzi(g * step), seed)


def dupes(O, r: int) -> np.ndarray:
    """A voxelised scan (1 m leaf) with every point repeated r times: zero distances, and for r > k ties at the k-th
    place on every point."""
    return np.ascontiguousarray(np.repeat(scan(O, 0, 1.0), r, axis=0))


HOT_COPIES = 600
HOT_CLUSTER = 2000


def hot_cell(O, seed: int = 2) -> np.ndarray:
    """A voxelised scan plus HOT_COPIES copies of one point and a HOT_CLUSTER-point cluster in a 2 cm cube next to it: a
    cell holding more than the tile capacity (TQ_CMAX slots), so its tile overflows and its points take the warp search."""
    base = scan(O, 3, 0.25)
    rng = np.random.default_rng(seed)
    hot = np.array([6.0, -3.0, 0.5], dtype=np.float32)
    copies = np.repeat(hot[None, :], HOT_COPIES, axis=0)
    cluster = hot[None, :] + rng.uniform(0.0, 0.02, size=(HOT_CLUSTER, 3)).astype(np.float32)
    return _shuffled(np.vstack([base, _xyzi(copies), _xyzi(cluster)]), seed)


def flat(n: int = 20000, extent: float = 20.0, seed: int = 3) -> np.ndarray:
    """Random points on z = 0: a grid one cell thick (the plan kernel's stride loop over many boxes) and exactly
    coplanar neighbourhoods."""
    rng = np.random.default_rng(seed)
    return _xyzi(np.c_[rng.uniform(-extent, extent, size=(n, 2)), np.zeros(n)])


def line(per_segment: int = 3000, seed: int = 4) -> np.ndarray:
    """Points on four 3-D segments: collinear neighbourhoods, where the PLANE regularisation is basis dependent."""
    rng = np.random.default_rng(seed)
    ends = np.array([[[-10, -10, 0], [10, 10, 2]], [[-5, 8, 1], [7, -6, 4]], [[0, 0, -3], [0, 0, 9]],
                     [[12, -12, 3], [14, 12, 3]]], dtype=np.float64)
    parts = []
    for a, b in ends:
        t = rng.uniform(0.0, 1.0, size=(per_segment, 1))
        parts.append(a + t * (b - a))
    return _shuffled(_xyzi(np.vstack(parts)), seed)


def sparse(O, k: int, n_isolated: int = 64, n_groups: int = 32, seed: int = 5) -> np.ndarray:
    """A voxelised scan plus, above it, isolated points and groups of exactly k+1 points, metres apart: boxes whose
    surroundings hold fewer than 2k points (the plan's slow items), tile radius growth up to TQ_SMAX, and the rest
    kernel's warp search."""
    rng = np.random.default_rng(seed)
    base = scan(O, 6, 0.25)
    iso = np.c_[rng.uniform(-60, 60, size=(n_isolated, 2)), rng.uniform(25, 45, size=n_isolated)]
    centres = np.c_[rng.uniform(-60, 60, size=(n_groups, 2)), rng.uniform(50, 70, size=n_groups)]
    groups = (centres[:, None, :] + rng.normal(0.0, 0.05, size=(n_groups, k + 1, 3))).reshape(-1, 3)
    return _shuffled(np.vstack([base, _xyzi(iso), _xyzi(groups)]), seed)


def raw_submap(O, keyframes: int = 6) -> np.ndarray:
    """Six unvoxelised keyframes in the world frame (DLO with its voxel filter off): above TILE_MIN_POINTS points, so
    AUTO runs them on the tile path, with dense rings near each sensor (the plan splits boxes)."""
    keys = []
    for j in range(keyframes):
        i = j * 33
        T = synth.trajectory_pose(i)
        keys.append(synth.transform_xyzi(synth.crop_box_negative(synth.os1_like(i, T)), T.astype(np.float32)))
    return np.ascontiguousarray(np.vstack(keys))


FAR_SHIFT = (20000.0, -2000.0, 30.0)


def far(submap) -> np.ndarray:
    """The S2M submap shifted by (+20 km, -2 km, +30 m): coordinates quantised to millimetres, far from the origin."""
    p = submap[:, :3].astype(np.float64) + np.asarray(FAR_SHIFT)
    out = submap.copy()
    out[:, :3] = p.astype(np.float32)
    return out


def nan_rows(cloud, frac: float = 0.01, seed: int = 7):
    """`cloud` with a fraction of its rows made non-finite (NaN, +Inf or -Inf in one or all coordinates): non-finite
    queries and candidates inside tiles.  Returns (cloud, mask of the finite rows)."""
    rng = np.random.default_rng(seed)
    out = cloud.copy()
    n = out.shape[0]
    rows = rng.choice(n, size=max(1, int(frac * n)), replace=False)
    kinds = rng.integers(0, 4, size=rows.size)
    vals = np.array([np.nan, np.inf, -np.inf], dtype=np.float32)
    for r, kind in zip(rows, kinds):
        if kind == 3:
            out[r, :3] = np.nan
        else:
            out[r, kind] = vals[rng.integers(0, 3)]
    return out, np.isfinite(out[:, :3]).all(axis=1)
