"""CPU restatement of pcl::Registration::getFitnessScore(max_range) (PCL registration.hpp), the reference the GPU
fitness score (ngicp_fitness_score / ngicp_fitness_batch) is tested against.  Test infrastructure only.

PCL: transformPointCloud(*input_, input_transformed, final_transformation_) in float; per point
tree_->nearestKSearch(pt, 1); `if (nn_dists[0] <= max_range) { fitness_score += nn_dists[0]; nr++; }`, summed serially
in double; `fitness_score / nr`, or DBL_MAX when nr == 0.  The SQUARED float distance is compared with max_range as
given, as a double, with <=.
"""
import sys

import numpy as np

DBL_MAX = sys.float_info.max


def transform_f32(src_xyz, T) -> np.ndarray:
    """Eigen's float transform in its operation order, per row ((m0*x + m1*y) + (m2*z + m3)).  numpy float32
    arithmetic is unfused, so the bits are the device's."""
    p = np.asarray(src_xyz, dtype=np.float32)[:, :3]
    T = np.asarray(T, dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        rows = [(T[r, 0] * p[:, 0] + T[r, 1] * p[:, 1]) + (T[r, 2] * p[:, 2] + T[r, 3]) for r in range(3)]
    return np.ascontiguousarray(np.stack(rows, axis=1).astype(np.float32))


def score_from_d2(d2: np.ndarray, max_range: float = DBL_MAX):
    """PCL's filter and serial double sum over per-point nearest squared distances (NaN = no neighbour / non-finite
    point, never counted).  Returns (score, count)."""
    with np.errstate(invalid="ignore"):
        sel = np.asarray(d2, dtype=np.float32).astype(np.float64) <= max_range
    vals = np.asarray(d2, dtype=np.float32)[sel].astype(np.float64)
    if vals.size == 0:
        return DBL_MAX, 0
    return float(np.add.accumulate(vals)[-1]) / vals.size, int(vals.size)


def nearest_d2(q: np.ndarray, target) -> np.ndarray:
    """Per query the squared distance to the nearest target point through the oracle's kd-tree (`target`: an
    oracle.Cloud or None for an empty target); NaN where the query is not finite or nothing was found."""
    d2 = np.full(q.shape[0], np.nan, dtype=np.float32)
    ok = np.isfinite(q).all(axis=1)
    if target is None or target.n == 0 or not ok.any():
        return d2
    idx, d = target.knn(np.ascontiguousarray(q[ok]), 1)
    d2[ok] = np.where(idx[:, 0] >= 0, d[:, 0], np.float32(np.nan))
    return d2


def fitness_score(src_xyz, target, T, max_range: float = DBL_MAX):
    """getFitnessScore(max_range) of `src_xyz` (n, >=3) against `target` (oracle.Cloud, or None when empty) at the
    4x4 transform T.  Returns (score, count)."""
    return score_from_d2(nearest_d2(transform_f32(src_xyz, T), target), max_range)


def brute_nearest_d2(q: np.ndarray, tgt_xyz: np.ndarray, block: int = 256) -> np.ndarray:
    """Exhaustive float32 nearest squared distance in nanoflann's order ((dx*dx + dy*dy) + dz*dz); NaN for non-finite
    queries."""
    t = np.asarray(tgt_xyz, dtype=np.float32)[:, :3]
    out = np.full(q.shape[0], np.nan, dtype=np.float32)
    for a in range(0, q.shape[0], block):
        qq = q[a:a + block]
        with np.errstate(over="ignore", invalid="ignore"):
            dx = qq[:, None, 0] - t[None, :, 0]
            dy = qq[:, None, 1] - t[None, :, 1]
            dz = qq[:, None, 2] - t[None, :, 2]
            d = (dx * dx + dy * dy) + dz * dz
        out[a:a + block] = d.min(axis=1)
    out[~np.isfinite(q).all(axis=1)] = np.nan
    return out
