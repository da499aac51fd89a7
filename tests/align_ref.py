"""CPU restatement of the registration linearisation (csrc/align.cu: K4 linearize_block / finish_point, K5 error_point)
and the clouds built to reach its rare branches.  Test infrastructure only.

K4 per source point: q = float(T) * p (fitness_ref.transform_f32); the exact 1-NN of q among the target points under
nanoflann's float metric (knn_ref.sqdist_f32); a correspondence iff q is finite and float64(d) < thr^2 (thr^2 in double),
else corr = -1 and sqd = FLT_MAX; M = (C_B + R C_A R^T)^-1 restated in gicp_math.cuh's operation order (sym3_rcr, then
sym3_inverse); then the 28 gicp_accumulate terms.  numpy float64 arithmetic is unfused and align.o is built with
-fmad=false, so applied to the GPU's own correspondences and covariances M and every term are the device's bits.

Sums (H, b, err) run in a different order on the device (per warp, per block, per pass).  They are checked against the
exact sum (math.fsum) with the order-independent bound |gpu - exact| <= gamma(n-1) * sum|t_i| per component, where
gamma(k) = k u / (1 - k u), u = 2^-53 and n is the number of contributing points.
"""
import math

import numpy as np

from direct_lidar_odometry_b200 import synth
import fitness_ref
import knn_ref

FLT_MAX = np.float32(np.finfo(np.float32).max)
U = 2.0 ** -53
KMAX = 32                   # widest tie set the kd-tree pass resolves; wider ones fall back to brute force
transform_f32 = fitness_ref.transform_f32


def gamma(k: int) -> float:
    return k * U / (1.0 - k * U) if k > 0 else 0.0


# ------------------------------------------------------------------------------------------------ exact 1-NN
def _brute_ties(q, tgt, rows):
    """(dmin, tie lists) of q[rows] by exhaustive search."""
    t = np.asarray(tgt, dtype=np.float32)[:, :3]
    dmin = np.empty(len(rows), dtype=np.float32)
    ties = []
    for j, r in enumerate(rows):
        d = knn_ref.sqdist_f32(q[r][None, :], t)
        m = d.min()
        dmin[j] = m
        ties.append(np.nonzero(d == m)[0].astype(np.int32) if np.isfinite(m) else np.zeros(0, np.int32))
    return dmin, ties


class NN1:
    """Exact 1-NN of every query: `d` (nq,) float32 minimum distance (+inf when the query is not finite or every
    distance overflows), `ties` (nq, w) int32 every target index at that distance, -1 padded, `nties` (nq,)."""

    def __init__(self, O, tgt, q, sample: int = 256, seed: int = 0):
        q = np.ascontiguousarray(np.asarray(q, dtype=np.float32)[:, :3])
        tgt = np.asarray(tgt, dtype=np.float32)
        nq = q.shape[0]
        fin = np.isfinite(q).all(axis=1)
        d = np.full(nq, np.inf, dtype=np.float32)
        lists = [np.zeros(0, np.int32)] * nq
        rows = np.nonzero(fin)[0]
        if rows.size:
            k = min(KMAX, tgt.shape[0])
            idx, d2 = O.Cloud(tgt).knn(q[rows], k)
            # a result set that stayed empty (every distance overflows) leaves its entries unset: recompute the first
            # entry's distance and hand such rows, and rows whose tie set is wider than k, to brute force
            first = knn_ref.sqdist_f32(q[rows], tgt[np.maximum(idx[:, 0], 0), :3])
            wide = (idx[:, 0] < 0) | (first != d2[:, 0]) | ~np.isfinite(first)
            for j, r in enumerate(rows):
                if wide[j]:
                    continue
                eq = d2[j] == d2[j, 0]
                if eq[-1] and k < tgt.shape[0]:          # the k-th is still tied: tie set wider than k
                    wide[j] = True
                    continue
                d[r] = d2[j, 0]
                lists[r] = np.sort(idx[j][eq])
            redo = rows[wide]
            if redo.size:
                bd, bt = _brute_ties(q, tgt, redo)
                for r, m, t in zip(redo, bd, bt):
                    d[r], lists[r] = m, t
            # the kd-tree against brute force on a sample of the queries
            pick = np.random.default_rng(seed).choice(rows, size=min(sample, rows.size), replace=False)
            bd, bt = _brute_ties(q, tgt, pick)
            for r, m, t in zip(pick, bd, bt):
                ok = (m == d[r]) if np.isfinite(m) else not np.isfinite(d[r])
                if not ok or not np.array_equal(t, lists[r]):
                    raise AssertionError(f"kd-tree 1-NN differs from brute force at query {r}")
        self.d = d
        self.nties = np.array([t.size for t in lists], dtype=np.int64)
        w = max(1, int(self.nties.max()) if nq else 1)
        self.ties = np.full((nq, w), -1, dtype=np.int32)
        for r, t in enumerate(lists):
            self.ties[r, :t.size] = t

    def has_corr(self, thr: float) -> np.ndarray:
        thr2 = float(thr) * float(thr)
        with np.errstate(invalid="ignore"):
            return np.isfinite(self.d) & (self.d.astype(np.float64) < thr2)

    def in_ties(self, corr) -> np.ndarray:
        return (self.ties == np.asarray(corr)[:, None]).any(axis=1)


# ------------------------------------------------------------------------------------------------ M and the terms
def sym6(covs) -> np.ndarray:
    """(n, 4, 4) or (n, 3, 3) -> (n, 6) xx, xy, xz, yy, yz, zz."""
    return knn_ref.cov6(covs)


def sym3_rcr(B, R, A):
    """gicp_math.cuh sym3_rcr: B + R A R^T, row by row in its order.  B, A (n, 6); R (3, 3) or (n, 3, 3)."""
    R = np.broadcast_to(np.asarray(R, dtype=np.float64), (B.shape[0], 3, 3))
    a0, a1, a2, a3, a4, a5 = (A[:, j] for j in range(6))
    RA = np.empty((B.shape[0], 3, 3))
    for r in range(3):
        r0, r1, r2 = R[:, r, 0], R[:, r, 1], R[:, r, 2]
        RA[:, r, 0] = r0 * a0 + r1 * a1 + r2 * a2
        RA[:, r, 1] = r0 * a1 + r1 * a3 + r2 * a4
        RA[:, r, 2] = r0 * a2 + r1 * a4 + r2 * a5
    o = np.empty_like(B)
    for j, (ra, rb) in enumerate(((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))):
        o[:, j] = B[:, j] + RA[:, ra, 0] * R[:, rb, 0] + RA[:, ra, 1] * R[:, rb, 1] + RA[:, ra, 2] * R[:, rb, 2]
    return o


def sym3_inverse(s):
    """gicp_math.cuh sym3_inverse, cofactors over the determinant in its order."""
    s0, s1, s2, s3, s4, s5 = (s[:, j] for j in range(6))
    with np.errstate(divide="ignore", invalid="ignore"):
        c00 = s3 * s5 - s4 * s4
        c01 = s2 * s4 - s1 * s5
        c02 = s1 * s4 - s2 * s3
        det = s0 * c00 + s1 * c01 + s2 * c02
        idt = 1.0 / det
        return np.stack([c00 * idt, c01 * idt, c02 * idt, (s0 * s5 - s2 * s2) * idt, (s1 * s2 - s0 * s4) * idt,
                         (s0 * s3 - s1 * s1) * idt], axis=1)


def mahal6(src_cov6, tgt_cov6, R, corr) -> np.ndarray:
    """(n, 6) M of every row with corr >= 0 (zeros elsewhere), from the given correspondences."""
    corr = np.asarray(corr)
    m = corr >= 0
    out = np.zeros((corr.size, 6))
    if m.any():
        out[m] = sym3_inverse(sym3_rcr(tgt_cov6[corr[m]], R, src_cov6[m]))
    return out


def mat4(m6) -> np.ndarray:
    """(n, 6) -> (n, 4, 4) with the 4th row and column zero (mahalanobis_ layout)."""
    m6 = np.asarray(m6)
    out = np.zeros((m6.shape[0], 4, 4))
    for j, (r, c) in enumerate(((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))):
        out[:, r, c] = out[:, c, r] = m6[:, j]
    return out


def transformed_a(src, T):
    """T p_A in double: R[r,0] px + R[r,1] py + R[r,2] pz + t[r], left to right (finish_point, error_point)."""
    p = np.asarray(src, dtype=np.float32)[:, :3].astype(np.float64)
    T = np.asarray(T, dtype=np.float64)
    return np.stack([T[r, 0] * p[:, 0] + T[r, 1] * p[:, 1] + T[r, 2] * p[:, 2] + T[r, 3] for r in range(3)], axis=1)


def terms(src, tgt, T, corr, m6) -> np.ndarray:
    """(m, 28) gicp_accumulate terms of the rows with corr >= 0: packed upper-triangle H (21), b (6), error."""
    corr = np.asarray(corr)
    sel = corr >= 0
    a = transformed_a(np.asarray(src)[sel], T)
    tp = np.asarray(tgt, dtype=np.float32)[corr[sel], :3].astype(np.float64)
    e = tp - a
    M = np.asarray(m6)[sel]
    m00, m01, m02, m11, m12, m22 = (M[:, j] for j in range(6))
    ax, ay, az = a[:, 0], a[:, 1], a[:, 2]
    ms00, ms01, ms02 = m01 * az - m02 * ay, -m00 * az + m02 * ax, m00 * ay - m01 * ax
    ms10, ms11, ms12 = m11 * az - m12 * ay, -m01 * az + m12 * ax, m01 * ay - m11 * ax
    ms20, ms21, ms22 = m12 * az - m22 * ay, -m02 * az + m22 * ax, m02 * ay - m12 * ax
    me0 = m00 * e[:, 0] + m01 * e[:, 1] + m02 * e[:, 2]
    me1 = m01 * e[:, 0] + m11 * e[:, 1] + m12 * e[:, 2]
    me2 = m02 * e[:, 0] + m12 * e[:, 1] + m22 * e[:, 2]
    cols = [az * ms10 - ay * ms20, az * ms11 - ay * ms21, az * ms12 - ay * ms22, -ms00, -ms10, -ms20,    # row 0
            -az * ms01 + ax * ms21, -az * ms02 + ax * ms22, -ms01, -ms11, -ms21,                          # row 1
            ay * ms02 - ax * ms12, -ms02, -ms12, -ms22,                                                   # row 2
            m00, m01, m02, m11, m12, m22,                                                                 # rows 3-5
            az * me1 - ay * me2, -az * me0 + ax * me2, ay * me0 - ax * me1, -me0, -me1, -me2,
            e[:, 0] * me0 + e[:, 1] * me1 + e[:, 2] * me2]
    return np.stack(cols, axis=1) if sel.any() else np.zeros((0, 28))


def error_terms(src, tgt, T, corr, m6) -> np.ndarray:
    """error_point (K5) per contributing row: e^T M e with e = q_B - T p_A, in its order."""
    corr = np.asarray(corr)
    sel = corr >= 0
    a = transformed_a(np.asarray(src)[sel], T)
    tp = np.asarray(tgt, dtype=np.float32)[corr[sel], :3].astype(np.float64)
    e0, e1, e2 = tp[:, 0] - a[:, 0], tp[:, 1] - a[:, 1], tp[:, 2] - a[:, 2]
    M = np.asarray(m6)[sel]
    m0 = M[:, 0] * e0 + M[:, 1] * e1 + M[:, 2] * e2
    m1 = M[:, 1] * e0 + M[:, 3] * e1 + M[:, 4] * e2
    m2 = M[:, 2] * e0 + M[:, 4] * e1 + M[:, 5] * e2
    return e0 * m0 + e1 * m1 + e2 * m2


def exact_sums(t) -> tuple:
    """(exact column sums, order-independent error bound per column) of per-point terms (m, c)."""
    t = np.asarray(t, dtype=np.float64)
    if t.ndim == 1:
        t = t[:, None]
    s = np.array([math.fsum(t[:, j]) for j in range(t.shape[1])])
    bound = gamma(max(t.shape[0] - 1, 0)) * np.abs(t).sum(axis=0)
    return s, bound


def unpack_H(red21) -> np.ndarray:
    H = np.zeros((6, 6))
    k = 0
    for r in range(6):
        for c in range(r, 6):
            H[r, c] = H[c, r] = red21[k]
            k += 1
    return H


def pack_H(H) -> np.ndarray:
    return np.array([H[r, c] for r in range(6) for c in range(r, 6)])


# ------------------------------------------------------------------------------------------------ clouds
def f32_pose(T) -> np.ndarray:
    """A pose whose entries are exact floats: the double and float transforms every path applies agree."""
    return np.asarray(T, dtype=np.float32).astype(np.float64)


def perturbed(rot_deg: float = 0.4, shift=(0.08, -0.03, 0.02)) -> np.ndarray:
    return f32_pose(synth.perturb_pose(np.eye(4), shift, rot_deg))


def lattice(n, step: float, offset=(0.0, 0.0, 0.0)) -> np.ndarray:
    """Integer grid n = (nx, ny, nz) times `step` (a power of two: exact coordinates) plus `offset`, shuffled."""
    g = np.stack(np.meshgrid(*(np.arange(k) for k in n), indexing="ij"), axis=-1).reshape(-1, 3).astype(np.float64)
    return knn_ref._shuffled(knn_ref._xyzi(g * step + np.asarray(offset)), 11)


def lattice_half():
    """Target: a 0.125 m lattice.  Source: the lattice shifted by exactly half a step on every axis, at the identity:
    every interior source point has 8 tied nearest targets, edge points 4 or 2."""
    tgt = lattice((40, 40, 10), 0.125)
    src = lattice((39, 39, 9), 0.125, (0.0625, 0.0625, 0.0625))
    return src, tgt, np.eye(4)


def _ulps(x, n):
    """x moved by n float32 ulps."""
    x = np.float32(x)
    for _ in range(abs(n)):
        x = np.nextafter(x, np.float32(np.inf if n > 0 else -np.inf))
    return x


def _hit(p, v, rng):
    """A float32 point at squared float distance exactly v from target point p (searched over a few ulps), or None."""
    for _ in range(64):
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        base = (p.astype(np.float64) + u * math.sqrt(float(v))).astype(np.float32)
        for dx in range(-3, 4):
            for dy in range(-3, 4):
                c = np.array([_ulps(base[0], dx), _ulps(base[1], dy), base[2]], dtype=np.float32)
                if knn_ref.sqdist_f32(c, p) == v:
                    return c
    return None


def straddle_values(thr: float):
    """The float squared distances next to thr^2: prev(f), f, next(f) with f the float nearest to thr^2 (double)."""
    f = np.float32(float(thr) * float(thr))
    return np.nextafter(f, np.float32(0)), f, np.nextafter(f, np.float32(np.inf))


def straddlers(thr: float, per_value: int = 96, seed: int = 8):
    """Target: a 2 m lattice (exact coordinates, isolated points).  Source: for each of the three float squared
    distances next to thr^2, `per_value` points at exactly that distance from a lattice point, plus as many points at
    random distances inside and outside thr; at the identity."""
    rng = np.random.default_rng(seed)
    tgt = lattice((12, 12, 4), 2.0)
    xyz = tgt[:, :3]
    pts = []
    for v in straddle_values(thr):
        made = 0
        while made < per_value:
            c = _hit(xyz[rng.integers(xyz.shape[0])], v, rng)
            if c is not None:
                pts.append(c)
                made += 1
    for _ in range(3 * per_value):
        p = xyz[rng.integers(xyz.shape[0])].astype(np.float64)
        u = rng.normal(size=3)
        pts.append((p + u / np.linalg.norm(u) * rng.uniform(0.05, 1.5 * thr)).astype(np.float32))
    return knn_ref._shuffled(knn_ref._xyzi(np.array(pts)), seed), tgt, np.eye(4)


def far_sources(O, shifts=(50.0, 200.0, 1000.0), per_shift: int = 200, seed: int = 9):
    """A voxelised scan against its neighbour scan, plus `per_shift` of its points moved by each shift (m) beyond the
    target's bounding box along a random axis: unbounded searches that must cross empty space."""
    rng = np.random.default_rng(seed)
    tgt = knn_ref.scan(O, 0)
    src = knn_ref.scan(O, 1)
    lo, hi = tgt[:, :3].min(0), tgt[:, :3].max(0)
    extra = []
    for s in shifts:
        rows = src[rng.choice(src.shape[0], per_shift, replace=False)].copy()
        ax = rng.integers(0, 3, size=per_shift)
        sign = rng.choice([-1.0, 1.0], size=per_shift)
        for j in range(per_shift):
            rows[j, ax[j]] = (hi[ax[j]] + s) if sign[j] > 0 else (lo[ax[j]] - s)
        extra.append(rows)
    return np.ascontiguousarray(np.vstack([src] + extra)), tgt


def overflow_rows(cloud, frac: float = 0.01, seed: int = 10):
    """`cloud` with a fraction of rows moved to (s, s, s), s = +-3e38: finite points whose squared distance to every
    target point is +inf, and whose float transform overflows under a rotation that adds two of them up.  Returns
    (cloud, mask of the untouched rows)."""
    rng = np.random.default_rng(seed)
    out = cloud.copy()
    rows = rng.choice(out.shape[0], size=max(1, int(frac * out.shape[0])), replace=False)
    for r in rows:
        out[r, :3] = np.float32(3e38) * np.float32(rng.choice([-1.0, 1.0]))
    keep = np.ones(out.shape[0], dtype=bool)
    keep[rows] = False
    return out, keep


# ------------------------------------------------------------------------------------------------ properties
def straddle_counts(nn: NN1, thr: float):
    """Points whose exact float distance is prev(thr^2), the float nearest thr^2, next(thr^2)."""
    return tuple(int((nn.d == v).sum()) for v in straddle_values(thr))


def tail_bound(nn: NN1, cell: float, thr: float) -> np.ndarray:
    """Points whose exact NN lies farther than twice the cell edge but within thr: the radius-1 cube around the query
    cannot settle them (its faces are at most 2 cells away), so they must go through the tail queue."""
    with np.errstate(invalid="ignore"):
        d = nn.d.astype(np.float64)
        return np.isfinite(d) & (d > (2.0 * cell) ** 2) & (d < float(thr) * float(thr))


def transform_overflows(src, T) -> np.ndarray:
    """Finite source rows whose float transform is not finite."""
    s = np.asarray(src, dtype=np.float32)[:, :3]
    return np.isfinite(s).all(axis=1) & ~np.isfinite(transform_f32(s, T)).all(axis=1)

