"""Exact restatement of the voxel grid stage (K0, csrc/voxel.cu) and clouds built to reach its edges.  TEST
INFRASTRUCTURE ONLY.

`voxel_filter` restates pcl::VoxelGrid<PointXYZI>::applyFilter as SURVEY.md App. B1 states it, every operation in
float32 and in PCL's order: inv = 1.0f / leaf; getMinMax3D over the finite points; the index-range guard; min_b /
div_b; ijk = (int)(floor(p * inv) - (float)min_b); idx wrapped to uint32 and sorted stable ascending; centroids as
sequential float32 running sums in ascending input index, divided by the float count.  The guard is PCL's made exact
(`grid_setup`, the rule of vox_grid_setup in csrc/voxel.cu and of the CPU oracle).  Sums are formed by a loop over run
positions, never by np.sum / np.add.reduceat, whose summation order is pairwise or unspecified.

Around it: the negative CropBox, removeNaN, transformPointCloud in synth.transform_xyzi's order, fromROSMsg
(oracle.from_ros_msg) and the voxel of every input point (`assign`, the library's voxel_assignment).

`cases()` returns the seeded clouds, each built for one property (see its docstring); `old_guard` and
`old_keys_signed_order` restate the rule the oracle used before, for the property checks.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

F32 = np.float32
INT32_MAX = 2**31 - 1
TWO31 = F32(2.0**31)
NAN = np.array(0x7FC00000, dtype=np.uint32).view(F32)[()]       # one payload everywhere: the bits stay comparable


def as_xyzi(pts) -> np.ndarray:
    """(n,3|4|8) -> contiguous (n,8) float32 PointXYZI records {x,y,z,1,intensity,0,0,0} (4 columns: the 4th is the
    intensity; 8 columns are taken as they are)."""
    pts = np.asarray(pts, dtype=F32)
    if pts.ndim == 2 and pts.shape[1] == 8:
        return np.ascontiguousarray(pts)
    out = np.zeros((pts.shape[0], 8), dtype=F32)
    out[:, :3] = pts[:, :3]
    out[:, 3] = 1.0
    if pts.shape[1] >= 4:
        out[:, 4] = pts[:, 3]
    return out


# ------------------------------------------------------------------------------------------------ the grid
def grid_setup(mn, mx, inv):
    """PCL's min_b / div_b with the exact guard.  Returns (overflow, min_b, div_b) as Python ints.  Overflow (the cloud
    passes through) when an axis extent (max - min) * inv is not finite or >= 2^31, dx*dy*dz > INT32_MAX without
    wrapping, floor(min * inv) or floor(max * inv) is outside int32, div_b exceeds INT32_MAX, floor(max * inv) -
    (float)min_b rounds past max_b - min_b, or the div_b product is >= 2^32."""
    dxyz, cells, minb, div = 1, 1, [], []
    with np.errstate(all="ignore"):
        for a in range(3):
            ext = F32(F32(mx[a]) - F32(mn[a])) * inv
            if not ext < TWO31:
                return 1, [0, 0, 0], [1, 1, 1]
            dxyz *= int(ext) + 1
            if dxyz > INT32_MAX:
                return 1, [0, 0, 0], [1, 1, 1]
            flo, fhi = np.floor(F32(mn[a]) * inv), np.floor(F32(mx[a]) * inv)
            if not (flo >= -TWO31) or not (fhi < TWO31):
                return 1, [0, 0, 0], [1, 1, 1]
            span = int(fhi) - int(flo)
            if span >= INT32_MAX or int(F32(fhi - flo)) > span:
                return 1, [0, 0, 0], [1, 1, 1]
            cells *= span + 1
            if cells >= 2**32:
                return 1, [0, 0, 0], [1, 1, 1]
            minb.append(int(flo))
            div.append(span + 1)
    return 0, minb, div


def old_guard(mn, mx, inv):
    """The guard the oracle and the kernels had before: PCL's int64 dx*dy*dz > INT32_MAX only.  Returns (overflow,
    exact dx*dy*dz as a Python int or None where (int64)ext itself is out of range, min_b, div_b); min_b / div_b only
    where every floor is inside int32 (x86 and PTX disagree on the rest)."""
    with np.errstate(all="ignore"):
        ext = [F32(F32(mx[a]) - F32(mn[a])) * inv for a in range(3)]
        dprod = None
        if all(np.isfinite(e) and e < F32(2.0**63) for e in ext):
            dprod = 1
            for e in ext:
                dprod *= int(e) + 1
        wrapped = None if dprod is None else ((dprod + 2**63) % 2**64) - 2**63
        over = wrapped is not None and wrapped > INT32_MAX
        flo = [np.floor(F32(mn[a]) * inv) for a in range(3)]
        fhi = [np.floor(F32(mx[a]) * inv) for a in range(3)]
    minb = div = None
    if all(-TWO31 <= v < TWO31 for v in flo + fhi):
        minb = [int(v) for v in flo]
        div = [int(fhi[a]) - int(flo[a]) + 1 for a in range(3)]
    return over, dprod, minb, div


def keys_of(xyz, inv, minb, div) -> np.ndarray:
    """uint32 voxel index of finite points: (int)(floor(p * inv) - (float)min_b) per axis, i + j*div0 + k*div0*div1 mod
    2^32 (the guard keeps every term in range)."""
    with np.errstate(all="ignore"):
        fl = np.floor(np.asarray(xyz, F32) * inv) - np.asarray(minb, dtype=np.int64).astype(F32)
    ijk = fl.astype(np.int64)
    return ((ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * (div[0] * div[1])) & 0xFFFFFFFF).astype(np.uint64)


def bbox(xyz):
    fin = np.isfinite(xyz).all(axis=1)
    return fin, xyz[fin].min(axis=0), xyz[fin].max(axis=0)


def voxel_filter(pts, leaf):
    """pcl::VoxelGrid<PointXYZI>::filter.  Returns (records (m,8), assign (n,) or None, status): status 1 is the
    pass-through (records = the input records; no voxel of a point is defined then)."""
    pts = as_xyzi(pts)
    n = pts.shape[0]
    xyz = pts[:, :3]
    fin = np.isfinite(xyz).all(axis=1)
    assign = np.full(n, -1, dtype=np.int32)
    if not fin.any():
        return np.zeros((0, 8), F32), assign, 0
    inv = F32(1.0) / F32(leaf)
    over, minb, div = grid_setup(xyz[fin].min(axis=0), xyz[fin].max(axis=0), inv)
    if over:
        return pts.copy(), None, 1
    idx = np.nonzero(fin)[0]
    key = keys_of(xyz[idx], inv, minb, div)
    order = np.argsort(key, kind="stable")
    sk, members = key[order], idx[order]
    starts = np.r_[0, np.nonzero(np.diff(sk))[0] + 1]
    lens = np.diff(np.r_[starts, sk.size])
    m = starts.size
    # run-position loop over the runs ordered by length: position j adds the j-th member of every run longer than j
    by_len = np.argsort(-lens, kind="stable")
    st, ln = starts[by_len], lens[by_len]
    vals = np.ascontiguousarray(pts[:, [0, 1, 2, 4]])
    acc = np.zeros((m, 4), F32)
    neg = -ln
    with np.errstate(all="ignore"):
        for j in range(int(ln[0])):
            act = int(np.searchsorted(neg, -j, side="left"))        # runs with ln > j (ln descending)
            acc[:act] += vals[members[st[:act] + j]]
        sums = np.empty_like(acc)
        sums[by_len] = acc
        cent = sums / lens.astype(F32)[:, None]
    out = np.zeros((m, 8), F32)
    out[:, :3] = cent[:, :3]
    out[:, 3] = 1.0
    out[:, 4] = cent[:, 3]
    assign[members] = np.repeat(np.arange(m, dtype=np.int32), lens)
    return out, assign, 0


def cropped(pts, crop) -> np.ndarray:
    """Negative pcl::CropBox(+-crop): a point with min <= p <= max on all three axes is dropped (NaN compares false)."""
    xyz = as_xyzi(pts)[:, :3]
    c = F32(crop)
    return ((xyz >= -c) & (xyz <= c)).all(axis=1)


def transform(pts, T) -> np.ndarray:
    """pcl::transformPointCloud in synth.transform_xyzi's order: ((m00 x + m01 y) + m02 z) + m03, float32."""
    from direct_lidar_odometry_b200 import synth
    with np.errstate(all="ignore"):
        return synth.transform_xyzi(as_xyzi(pts), np.asarray(T, dtype=F32))


def pipeline(pts, leaf, crop=None, T=None, compact_on_overflow=True):
    """What ngicp_preprocess / ngicp_transform_voxel_filter / ngicp_preprocess_pointcloud2 compute (and, with
    compact_on_overflow=False and no crop / transform, ngicp_voxel_filter): [transform] -> removeNaN + [negative
    CropBox] -> voxel grid.  Where the grid passes the cloud through, the output is the surviving points in input order
    ({x,y,z,1,intensity,0,0,0}); a removed point's voxel is -1.  Returns (records, assign or None, status)."""
    pts = as_xyzi(pts)
    if T is not None:
        pts = transform(pts, T)
    work = pts.copy()
    if crop is not None:
        work[cropped(work, crop), 0] = NAN          # a cropped point is treated as non-finite: no bbox, no voxel
    if not compact_on_overflow:
        assert crop is None and T is None
        return voxel_filter(work, leaf)
    rec, assign, st = voxel_filter(work, leaf) if leaf > 0 else (None, None, 1)
    if st == 0:
        return rec, assign, 0
    keep = np.isfinite(work[:, :3]).all(axis=1)
    out = np.zeros((int(keep.sum()), 8), F32)
    out[:, :3] = work[keep, :3]
    out[:, 3] = 1.0
    out[:, 4] = work[keep, 4]
    assign = np.full(pts.shape[0], -1, np.int32)
    assign[keep] = np.arange(out.shape[0], dtype=np.int32)
    return out, assign, (1 if leaf > 0 else 0)


def from_ros_msg(msg) -> np.ndarray:
    from oracle.oracle import from_ros_msg as f
    return f(msg)


def key_bits(pts, leaf, crop=None, T=None):
    """Radix key width the library sorts for this cloud (cells < 2^bits, cells = div_b product); None on overflow."""
    pts = as_xyzi(pts)
    if T is not None:
        pts = transform(pts, T)
    pts = pts.copy()
    if crop is not None:
        pts[cropped(pts, crop), 0] = NAN
    fin = np.isfinite(pts[:, :3]).all(axis=1)
    if not fin.any():
        return 1
    over, _, div = grid_setup(pts[fin, :3].min(axis=0), pts[fin, :3].max(axis=0), F32(1.0) / F32(leaf))
    if over:
        return None
    return max(1, (div[0] * div[1] * div[2]).bit_length())


# ------------------------------------------------------------------------------------------------ generators
@dataclass
class Case:
    name: str
    pts: np.ndarray                 # (n, 8) float32 records
    leaf: float
    crop: float | None = None       # for the preprocess entry points
    meta: dict = field(default_factory=dict)


def _records(xyz, rng, intensity=None):
    xyz = np.asarray(xyz, F32)
    it = rng.uniform(0, 1, xyz.shape[0]).astype(F32) if intensity is None else intensity
    return as_xyzi(np.c_[xyz, it].astype(F32))


def _cells(dims, n, rng, extra=()):
    """Points at cell centres (i + 0.5) of a dims[0] x dims[1] x dims[2] grid at leaf 1: div_b == dx == dims.  Both
    corners, points in the highest keys, a few NaN rows (the invalid key)."""
    d = np.asarray(dims, np.int64)
    ijk = (rng.random((n, 3)) * d).astype(np.int64)
    top = d - 1 - (rng.random((n // 8, 3)) * np.minimum(d, 4)).astype(np.int64)
    ijk = np.vstack([np.zeros((1, 3), np.int64), d[None] - 1, top, ijk] + [np.asarray(e, np.int64)[None] for e in extra])
    xyz = ijk.astype(np.float64) + 0.5
    pts = _records(xyz, rng)
    pts = pts[rng.permutation(pts.shape[0])]
    pts[rng.choice(pts.shape[0], 5, replace=False), 1] = NAN
    return pts


def faces(leaf, seed=0, n=6000):
    """A lattice at k * leaf (k in [-40, 40], float32 product) with every coordinate moved 0, +1 or -1 ulp, plus rows
    of +-0.0 and subnormals: many p * inv land one ulp below (or on, or above) an integer, where floor decides the
    voxel, and negative coordinates separate floor from truncation."""
    rng = np.random.default_rng(seed)
    k = rng.integers(-40, 41, size=(n, 3)).astype(F32)
    xyz = k * F32(leaf)
    step = rng.integers(-1, 2, size=xyz.shape)
    xyz = np.where(step > 0, np.nextafter(xyz, F32(np.inf)), np.where(step < 0, np.nextafter(xyz, F32(-np.inf)), xyz)).astype(F32)
    sub = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.1754942e-38, -1.1754942e-38], F32)
    special = sub[rng.integers(0, sub.size, size=(64, 3))]
    special[:8, 0] = sub
    return _records(np.vstack([xyz, special]), rng)


PASS_EDGES = {          # div_b product -> dims; the fused kernel's 1->2, 2->3 and 3->4 radix passes (9-bit digits)
    511: (7, 73, 1), 512: (8, 8, 8), 2**18 - 1: (133, 27, 73), 2**18: (64, 64, 64),
    2**27 - 1: (7, 73, 262657), 2**27: (512, 512, 512),
}
GUARD_EDGES = {         # dx*dy*dz at the nearest reachable values either side of INT32_MAX (a prime)
    "below_2^31-2": (1386, 4681, 331), "above_2^31": (2048, 1024, 1024), "cube_1291": (1291, 1291, 1291),
}


def band(seed=0, n=2000):
    """A 1290-leaf cube, corners at 0.9 and 1290.8: dx*dy*dz = 1290^3 <= INT32_MAX but div_b = 1291 per axis, so keys
    run past 2^31 (points in the highest keys included): a signed sort orders them differently from PCL's unsigned."""
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(0.9, 1290.8, size=(n, 3)).astype(F32)
    top = rng.uniform(1285.0, 1290.8, size=(n // 8, 3)).astype(F32)
    xyz = np.vstack([np.full((1, 3), 0.9, F32), np.full((1, 3), 1290.8, F32), top, xyz])
    pts = _records(xyz, rng)
    pts[rng.choice(pts.shape[0], 5, replace=False), 2] = NAN
    return pts


SLAB_Z = float(2**30 + 128)


def slab_wrap(seed=0, n=2000):
    """x, y in [0.5, 1.4], z in [0.5, 2^30 + 128] at leaf 1: dx*dy*dz = 2^30 + 129 passes PCL's guard, div_b = (2, 2,
    2^30 + 129) and the product 2^32 + 516 wraps: the old invalid key 516 is the key of the finite points at z ~ 129.5."""
    rng = np.random.default_rng(seed)
    xy = rng.uniform(0.5, 1.4, size=(n, 2))
    z = np.where(rng.random(n) < 0.5, rng.uniform(0.5, 300.0, n), rng.uniform(0.5, SLAB_Z, n))
    xyz = np.c_[xy, z].astype(F32)
    pin = np.array([[0.5, 0.5, 0.5], [1.4, 1.4, SLAB_Z], [0.5, 0.5, 129.5], [0.7, 0.6, 129.2]], F32)
    pts = _records(np.vstack([pin, xyz]), rng)
    pts = pts[rng.permutation(pts.shape[0])]
    pts[rng.choice(pts.shape[0], 7, replace=False), 0] = NAN
    return pts


def round_up(seed=0, n=1000):
    """x from -0.5 to 2^24 + 2 at leaf 1: min_b = -1, max_b = 2^24 + 2, and the last cell's float index
    (2^24 + 2) - (-1.0f) rounds to 2^24 + 4 = div_b: that point's key equals div_b's product, the invalid key, although
    dx*dy*dz and the product are far below every int32 / uint32 bound."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-0.5, 2.0**24 + 2, n)
    xyz = np.c_[x, rng.uniform(0.5, 0.6, (n, 2))].astype(F32)
    xyz = np.vstack([np.array([[-0.5, 0.5, 0.5], [2.0**24 + 2, 0.6, 0.6]], F32), xyz])
    pts = _records(xyz, rng)
    pts[3, 1] = NAN
    return pts


def far(stray=None, offset=None, seed=0, n=3000):
    """A cloud within +-40 m plus one stray return at (f, -f/2, f/4), or the whole cloud moved by `offset` so that
    |min * inv| > 2^31 at leaf 0.25.  PCL's int64 dx*dy*dz wraps (or the conversion is already out of range) and the
    floors are out of int32: x86 gives INT_MIN where PTX saturates."""
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(-40, 40, size=(n, 3)).astype(F32)
    if offset is not None:
        xyz = (xyz + F32(offset)).astype(F32)
    if stray is not None:
        xyz[17] = (stray, -stray * 0.5, stray * 0.25)
    return _records(xyz, rng)


def scan_like(n, seed=0):
    """A lidar-like cloud: ground plane, walls and clutter within +-40 m, no points inside the +-1 m box."""
    rng = np.random.default_rng(seed)
    r = rng.uniform(2.0, 40.0, n)
    th = rng.uniform(-np.pi, np.pi, n)
    z = np.where(rng.random(n) < 0.4, -1.7 + rng.normal(0, 0.02, n), rng.uniform(-1.7, 6.0, n))
    return _records(np.c_[r * np.cos(th), r * np.sin(th), z], rng)


def hot_voxel(seed=0, n_scan=60000, n_hot=20000):
    """A scan with 20k points in one 0.25 m voxel scattered through it: the run spans many fused-kernel chunks."""
    rng = np.random.default_rng(seed)
    scan = scan_like(n_scan, seed)
    hot = _records(F32(10.0) + rng.uniform(0.01, 0.24, size=(n_hot, 3)).astype(F32), rng)
    pts = np.vstack([scan, hot])
    return pts[rng.permutation(pts.shape[0])]


def size_cloud(n, seed=0):
    rng = np.random.default_rng(seed + n)
    xyz = rng.uniform(-40, 40, size=(n, 3)).astype(F32)
    xyz[:, 2] *= F32(0.1)
    return _records(xyz, rng)


def sizes(sms=148):
    """Around warp / block / fused-chunk sizes, the fused kernel's smallest grid, its limit (sms * 4096) and just past
    it (the multi-kernel fallback)."""
    return [1, 31, 32, 33, 1023, 1024, 1025, 4096, 4097, sms * 1024 - 1, sms * 1024 + 1, sms * 4096, sms * 4096 + 1]


def dirty(seed=0, n=5000):
    """NaN / +-Inf in one coordinate at a time, NaN / +-Inf intensity on finite xyz (one voxel gets +Inf and -Inf:
    a NaN centroid intensity)."""
    rng = np.random.default_rng(seed)
    pts = scan_like(n, seed)
    pts[0::29, 0] = NAN
    pts[1::31, 1] = np.inf
    pts[2::37, 2] = -np.inf
    pts[3::41, 1] = NAN
    pts[4::43, 0] = -np.inf
    pts[5::47, 2] = NAN
    pts[6::53, 4] = NAN
    pts[7::59, 4] = np.inf
    pts[8::61, 4] = -np.inf
    pts[100, :3] = pts[101, :3] = (20.1, 20.1, 3.1)
    pts[100, 4], pts[101, 4] = np.inf, -np.inf
    return pts


def lonely(seed=0, n=3000):
    """Every point non-finite but one."""
    rng = np.random.default_rng(seed)
    pts = scan_like(n, seed)
    kind = rng.integers(0, 3, n)
    pts[np.arange(n), kind] = np.where(rng.random(n) < 0.5, NAN, np.inf)
    pts[1234, :3] = (3.3, -4.4, 0.5)
    return pts


def crop_faces(seed=0, n=4000):
    """For the +-1 m negative crop box: points exactly on its faces and edges (dropped), one ulp outside a face (kept),
    and dropped points at x < 0 while everything kept has x > 1: counting a cropped point would move min_b."""
    rng = np.random.default_rng(seed)
    keep = rng.uniform(-40, 40, size=(n, 3)).astype(F32)
    keep[:, 0] = rng.uniform(2.0, 40.0, n)
    on = rng.uniform(-1, 1, size=(300, 3)).astype(F32)
    ax = rng.integers(0, 3, 300)
    on[np.arange(300), ax] = np.where(rng.random(300) < 0.5, F32(1.0), F32(-1.0))
    on[:8] = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], F32)
    on[on[:, 0] > F32(0.0), 0] *= F32(-1.0)                         # inside the box and at x <= 0
    inside = rng.uniform(-0.95, -0.05, size=(300, 3)).astype(F32)
    out_face = rng.uniform(-1, 1, size=(100, 3)).astype(F32)
    out_face[:, 0] = np.nextafter(F32(1.0), F32(2.0))               # just outside +x: kept
    xyz = np.vstack([keep, on, inside, out_face])
    pts = _records(xyz, rng)
    return pts[rng.permutation(pts.shape[0])]


def cases(sms=148, with_sizes=True):
    """Every generator, seeded.  meta['gen'] names the generator; the GPU test runs each through every path."""
    out = []
    for leaf in (0.1, 0.3, 0.25):
        out.append(Case(f"faces_{leaf}", faces(leaf, seed=int(leaf * 100)), leaf, meta=dict(gen="faces")))
    for prod, dims in PASS_EDGES.items():
        out.append(Case(f"pass_{prod}", _cells(dims, 3000, np.random.default_rng(prod)), 1.0, meta=dict(gen="pass", prod=prod)))
    out.append(Case("band", band(), 1.0, meta=dict(gen="band")))
    out.append(Case("slab_wrap", slab_wrap(), 1.0, meta=dict(gen="slab_wrap")))
    out.append(Case("round_up", round_up(), 1.0, meta=dict(gen="round_up")))
    for name, dims in GUARD_EDGES.items():
        out.append(Case(f"guard_{name}", _cells(dims, 2000, np.random.default_rng(sum(dims))), 1.0,
                        meta=dict(gen="guard", prod=int(np.prod(dims, dtype=np.int64)))))
    for f in (1e13, 1e20, 3e38):
        out.append(Case(f"far_{f:g}", far(stray=f), 0.25, meta=dict(gen="far")))
    out.append(Case("far_offset", far(offset=6.0e8), 0.25, meta=dict(gen="far_offset")))
    out.append(Case("hot_voxel", hot_voxel(), 0.25, crop=1.0, meta=dict(gen="hot")))
    out.append(Case("dirty", dirty(), 0.5, crop=1.0, meta=dict(gen="dirty")))
    out.append(Case("lonely", lonely(), 0.25, meta=dict(gen="lonely")))
    out.append(Case("crop_faces", crop_faces(), 0.5, crop=1.0, meta=dict(gen="crop")))
    if with_sizes:
        for n in sizes(sms):
            out.append(Case(f"n{n}", size_cloud(n), 0.4, meta=dict(gen="size", n=n)))
    return out
