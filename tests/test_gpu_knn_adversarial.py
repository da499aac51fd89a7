"""The kNN + covariance kernels (csrc/knn_cov.cu: plan -> tile -> rest -> covariance launches, and the one-warp-per-point
search) on clouds built to reach their rare branches — exact distance ties everywhere, duplicated points, a cell over the
tile capacity, one-cell-thick and collinear clouds, isolated points, raw submaps, coordinates far from the origin,
non-finite rows — at every k the tile kernel handles differently (1, 2, 3 < 4 <= 5, 10 and 20 specialised, the rest
generic, 31 and 32 at the warp-wide limit).  tests/knn_ref.py holds the references and the generators.

On every point, for both kernel families:
  1. the k squared distances of ngicp_cov_neighbors equal the exact sorted k distances bit for bit, ties included;
  2. the neighbour list is valid: distinct in-range indices, distances that recompute bit for bit and never decrease;
  3. with REG_NONE the covariance equals the restated statistics summed over the GPU's own list in its reported order,
     bit for bit (the summation order is the order cov_neighbors reports, also after tie fix-ups and the rest search);
  4. where all k+1 distances are distinct, the covariance equals the oracle's bit for bit (REG_NONE) and within 1e-5
     relative (REG_PLANE, where the plane is resolvable); PLANE eigenvalue magnitudes are {1e-3, 1, 1};
  5. tile and warp covariances are bit-identical on those points.
Plus: covariance slices of a tile-path run add up to the full result, non-finite rows change nothing for the finite
points, and NGICP_KNN_STATS shows that each cloud reaches the branch it was built for.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import knn_ref as R
from util import make_small_submap

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
COV_RTOL = 1e-5
K_ALL = (1, 2, 3, 5, 10, 16, 20, 31, 32)
KMAX = max(K_ALL)
SMALL = ("lattice", "dupes_2", "dupes_k", "dupes_k1", "hot_cell", "flat", "line", "sparse")


@pytest.fixture(scope="module")
def G():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from direct_lidar_odometry_b200 import NanoGICP
    return NanoGICP


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    oracle.load(prefer_ref=False)
    return oracle


class Clouds:
    """Generated clouds, their exact KMAX+1 distances and oracle covariances, built once per module."""

    def __init__(self, O):
        self.O = O
        self.pts, self.d2, self.tree, self.covs = {}, {}, {}, {}

    def key(self, name, k):
        return {"dupes_k": f"dupes_{k}", "dupes_k1": f"dupes_{k + 1}", "sparse": f"sparse_{k}"}.get(name, name)

    def get(self, key):
        if key not in self.pts:
            O = self.O
            if key == "lattice":
                c = R.lattice()
            elif key.startswith("dupes_"):
                c = R.dupes(O, int(key[6:]))
            elif key.startswith("sparse_"):
                c = R.sparse(O, int(key[7:]))
            elif key == "hot_cell":
                c = R.hot_cell(O)
            elif key == "flat":
                c = R.flat()
            elif key == "line":
                c = R.line()
            elif key == "raw_submap":
                c = R.raw_submap(O)
            elif key == "submap":
                c = make_small_submap(O)[0]
            elif key == "far":
                c = R.far(self.get("submap"))
            else:
                raise KeyError(key)
            self.pts[key] = c
        return self.pts[key]

    def ref_d2(self, key):
        if key not in self.d2:
            c = self.get(key)
            self.d2[key] = R.knn_distances(self.O, np.ascontiguousarray(c[:, :3]), c, min(KMAX + 1, c.shape[0]))
        return self.d2[key]

    def oracle_covs(self, key, k, method):
        if (key, k, method) not in self.covs:
            if key not in self.tree:
                self.tree[key] = self.O.Cloud(self.get(key))
            self.covs[(key, k, method)] = self.tree[key].covariances(k, method)
        return self.covs[(key, k, method)]


@pytest.fixture(scope="module")
def clouds(O):
    return Clouds(O)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32 if a.dtype == np.float32 else np.uint64)


def gpu_run(G, cloud, k, path, method, cell=None, table=None):
    """(covariances (n,4,4), neighbour indices (n,k), squared distances (n,k)) of one calculateSourceCovariances."""
    from direct_lidar_odometry_b200 import _lib
    g = G()
    g.setCorrespondenceRandomness(k)
    g.setRegularizationMethod(method)
    g.setKnnPath(path)
    if cell is not None:
        g.setGridCellSize(cell)
    if table is not None:
        g.setGridTableCells(table)
    g.setInputSource(cloud)
    assert g.calculateSourceCovariances() is True
    covs = g.getSourceCovariances()
    idx, d2 = g.cov_neighbors(_lib.SOURCE)
    return covs, idx, d2


def check_lists(cloud, k, idx, d2, ref_d2, rows):
    """Checks 1 and 2 on the rows `rows` (bool mask)."""
    n = cloud.shape[0]
    I, D = idx[rows], d2[rows]
    assert np.array_equal(bits(D), bits(ref_d2[rows][:, :k])), \
        f"distances differ on {int((bits(D) != bits(ref_d2[rows][:, :k])).any(axis=1).sum())} points"
    assert I.min() >= 0 and I.max() < n, "neighbour index out of range (or -1 with n >= k)"
    srt = np.sort(I, axis=1)
    assert (srt[:, 1:] != srt[:, :-1]).all(), "a neighbour listed twice"
    xyz = cloud[:, :3]
    rec = R.sqdist_f32(xyz[np.nonzero(rows)[0]][:, None, :], xyz[I])
    assert np.array_equal(bits(rec.astype(np.float32)), bits(D)), "reported d2 does not recompute"
    assert (np.diff(D, axis=1) >= 0).all(), "d2 decreases along a list"


def check_raw_covs(cloud, covs, idx, rows):
    """Check 3: the REG_NONE covariance is the restated statistics over the GPU's own list, bit for bit."""
    assert np.abs(covs[:, 3, :]).max() == 0 and np.abs(covs[:, :, 3]).max() == 0
    assert np.array_equal(bits(covs[:, :3, :3]), bits(covs[:, :3, :3].transpose(0, 2, 1)))
    got = R.cov6(covs)[rows]
    ref = R.raw_cov_from_list(cloud, idx[rows])
    same = (bits(got) == bits(ref)).all(axis=1)
    assert same.all(), f"{int((~same).sum())} covariances are not the sum over the reported list in its order"


def tie_free(ref_d2, k):
    """Points whose k+1 nearest distances are all distinct: a unique list, the same for every correct kernel."""
    d = ref_d2[:, :k + 1]
    return (d[:, 1:] != d[:, :-1]).all(axis=1)


def check_plane(covs, oracle_plane, oracle_raw, ok):
    """Check 4 for REG_PLANE: within 1e-5 relative where resolvable; eigenvalue magnitudes {1e-3, 1, 1} within 1e-9
    there and within 1e-4 on every other point.

    On a singular neighbourhood (exactly coplanar: k = 3, the flat cloud; or duplicated points) the reference's SVD may
    pair the null direction of U with the opposite one of V, so U diag(1, 1, 1e-3) V^T has the eigenvalue -1e-3 there;
    the CPU oracle does this too, so the sign is checked through the parity with the oracle.  Where the plane is not
    defined at all (collinear or coincident neighbours) U and V also differ inside the degenerate subspace; the kernel
    keeps the upper triangle of that non-symmetric product, whose eigenvalues then miss {1e-3, 1, 1}: by up to 7e-5 on
    the `line` cloud at k = 3, about 1e-5 at larger k (B200)."""
    w = np.linalg.eigvalsh(oracle_raw[:, :3, :3])
    resolvable = ok & ((w[:, 1] - w[:, 0]) > 1e-6 * w[:, 2])
    if resolvable.any():
        num = np.linalg.norm((covs - oracle_plane)[resolvable].reshape(-1, 16), axis=1)
        den = np.linalg.norm(oracle_plane[resolvable].reshape(-1, 16), axis=1)
        assert (num / den).max() < COV_RTOL
    ev = np.sort(np.abs(np.linalg.eigvalsh(0.5 * (covs[:, :3, :3] + covs[:, :3, :3].transpose(0, 2, 1)))), axis=1)
    dev = np.abs(ev - [1e-3, 1, 1]).max(axis=1)
    assert dev[resolvable].max(initial=0.0) < 1e-9, float(dev[resolvable].max())
    assert dev.max() < 1e-4, float(dev.max())


def run_all_checks(G, O, clouds, key, k, tile_path, **grid):
    from direct_lidar_odometry_b200 import _lib
    cloud = clouds.get(key)
    n = cloud.shape[0]
    ref = clouds.ref_d2(key)
    ok = tie_free(ref, k)
    rows = np.ones(n, dtype=bool)
    raw_ref = clouds.oracle_covs(key, k, O.REG_NONE)
    plane_ref = clouds.oracle_covs(key, k, O.REG_PLANE)
    raw = {}
    for path in (tile_path, _lib.KNN_WARP):
        covs, idx, d2 = gpu_run(G, cloud, k, path, O.REG_NONE, **grid)
        where = f"{key} k={k} path={path}"
        try:
            check_lists(cloud, k, idx, d2, ref, rows)
            check_raw_covs(cloud, covs, idx, rows)
            same = (bits(R.cov6(covs)) == bits(R.cov6(raw_ref))).all(axis=1)
            assert same[ok].all(), f"{int((~same[ok]).sum())} tie-free covariances differ from the oracle"
            pcovs = gpu_run(G, cloud, k, path, O.REG_PLANE, **grid)[0]
            check_plane(pcovs, plane_ref, raw_ref, ok)
        except AssertionError as e:
            raise AssertionError(f"{where}: {e}") from e
        raw[path] = covs
    a, b = raw[tile_path], raw[_lib.KNN_WARP]
    assert np.array_equal(bits(a[ok]), bits(b[ok])), f"{key} k={k}: tile and warp covariances differ off ties"


# ---------------------------------------------------------------------------------------------- small clouds, every k
@pytest.mark.parametrize("k", K_ALL)
@pytest.mark.parametrize("name", SMALL)
def test_small_clouds_every_k(G, O, clouds, name, k):
    from direct_lidar_odometry_b200 import _lib
    key = clouds.key(name, k)
    run_all_checks(G, O, clouds, key, k, _lib.KNN_TILE)


# ---------------------------------------------------------------------------------------------- large clouds, thinned k
@pytest.mark.parametrize("key,k", [("raw_submap", 3), ("raw_submap", 10), ("raw_submap", 16), ("raw_submap", 20),
                                   ("far", 5), ("far", 10), ("far", 20), ("far", 31)])
def test_large_clouds(G, O, clouds, key, k):
    """Above TILE_MIN_POINTS AUTO takes the tile path (raw submaps); the far cloud is forced onto it."""
    from direct_lidar_odometry_b200 import _lib
    big = clouds.get(key).shape[0] >= R.TILE_MIN_POINTS
    run_all_checks(G, O, clouds, key, k, _lib.KNN_AUTO if big else _lib.KNN_TILE)


@pytest.mark.parametrize("cell,table,k", [(0.1, None, 10), (0.1, None, 16), (2.0, None, 20), (2.0, None, 5),
                                          (4.0, None, 20), (4.0, None, 2), (None, 4096, 10), (None, 4096, 32)])
def test_submap_forced_cell_edge(G, O, clouds, cell, table, k):
    """The S2M submap with a forced cell edge: tiny cells give empty space and deep radius growth, coarse cells dense
    boxes, plan splits and tile overflow; a tiny table makes the device grow the cell."""
    from direct_lidar_odometry_b200 import _lib
    run_all_checks(G, O, clouds, "submap", k, _lib.KNN_TILE, cell=cell, table=table)


# ---------------------------------------------------------------------------------------------- slices
@pytest.mark.parametrize("k", [10, 16])
@pytest.mark.parametrize("name", ["lattice", "hot_cell", "sparse"])
def test_tile_slices_sum_to_full(G, O, clouds, name, k):
    """calculateSourceCovariancesPart(p, 3) on the tile path: the three slices (zeros elsewhere) add up to the full
    result bit for bit, with the plan, the ties and the fix-ups of each slice restricted to it."""
    from direct_lidar_odometry_b200 import _lib
    cloud = clouds.get(clouds.key(name, k))
    g = G()
    g.setCorrespondenceRandomness(k)
    g.setKnnPath(_lib.KNN_TILE)
    g.setInputSource(cloud)
    g.calculateSourceCovariances()
    full = g.getSourceCovariances()
    acc = np.zeros_like(full)
    covered = np.zeros(cloud.shape[0], dtype=int)
    for p in range(3):
        g.calculateSourceCovariancesPart(p, 3)
        part = g.getSourceCovariances()
        covered += np.abs(part).reshape(-1, 16).sum(axis=1) > 0
        acc += part
    assert (covered == 1).all()
    assert np.array_equal(bits(acc), bits(full)), float(np.abs(acc - full).max())


# ---------------------------------------------------------------------------------------------- non-finite rows
@pytest.mark.parametrize("k", [3, 10, 16])
def test_nan_rows(G, O, clouds, k):
    """raw_submap with 1 % of its rows non-finite: for the finite points, distances equal those of the same cloud with
    the non-finite rows removed, their lists never hold a non-finite row, their covariances equal the clean cloud's bit
    for bit off ties and are never NaN."""
    from direct_lidar_odometry_b200 import _lib
    clean_all = clouds.get("raw_submap")
    dirty, fin = R.nan_rows(clean_all)
    clean = np.ascontiguousarray(dirty[fin])
    fidx = np.nonzero(fin)[0]                  # dirty row of every clean row
    ref = R.knn_distances(O, np.ascontiguousarray(clean[:, :3]), clean, k + 1)
    ok = tie_free(ref, k)
    for path in (_lib.KNN_AUTO, _lib.KNN_WARP):
        covs, idx, d2 = gpu_run(G, dirty, k, path, O.REG_NONE)
        ccovs, cidx, _ = gpu_run(G, clean, k, path, O.REG_NONE)
        D, I = d2[fin], idx[fin]
        assert np.array_equal(bits(D), bits(ref[:, :k])), f"path={path}: finite points' distances changed"
        assert I.min() >= 0 and fin[I].all(), f"path={path}: a finite point lists a non-finite neighbour"
        check_raw_covs(dirty, covs, idx, fin)
        assert np.isfinite(covs[fin]).all()
        assert np.array_equal(bits(covs[fin][ok]), bits(ccovs[ok])), f"path={path}: tie-free covariances changed"
        assert np.array_equal(I[ok], fidx[cidx[ok]])
        pcovs = gpu_run(G, dirty, k, path, O.REG_PLANE)[0]
        assert np.isfinite(pcovs[fin]).all()


# ---------------------------------------------------------------------------------------------- branches reached
_DRIVER = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import numpy as np
from oracle import oracle as O
O.load(prefer_ref=False)
import knn_ref as R
from util import make_small_submap
from direct_lidar_odometry_b200 import NanoGICP, _lib
name, k, path, cell = sys.argv[3], int(sys.argv[4]), int(sys.argv[5]), float(sys.argv[6])
if name == "lattice": c = R.lattice()
elif name == "hot_cell": c = R.hot_cell(O)
elif name == "sparse": c = R.sparse(O, k)
elif name == "sparse_base": c = R.scan(O, 6, 0.25)
elif name == "dupes": c = R.dupes(O, k + 1)
elif name == "flat": c = R.flat()
elif name == "line": c = R.line()
elif name == "raw_submap": c = R.raw_submap(O)
elif name == "nan_rows": c = R.nan_rows(R.raw_submap(O))[0]
elif name == "far": c = R.far(make_small_submap(O)[0])
else: c = make_small_submap(O)[0]
g = NanoGICP(0)
g.setCorrespondenceRandomness(k)
g.setKnnPath(path)
if cell > 0: g.setGridCellSize(cell)
g.setInputSource(c)
g.calculateSourceCovariances()
g.sync()
print(c.shape[0])
"""

_HEAD = re.compile(r"\[ngicp knn\] n=(\d+) k=(\d+) warp-search=(\d+) \([\d.]+%, ties (\d+)\) items=(\d+)")
_CTRL = re.compile(r"control: rest=(\d+) fix=(\d+) slow=(\d+) items=(\d+), items by box edge \d+ / \d+ / 1: (\d+) / (\d+) / (\d+)")


def knn_stats(name, k, path=2, cell=0.0):
    """Runs one tile-path covariance computation in a fresh process with NGICP_KNN_STATS set (the variable is read once
    per process) and parses its report."""
    env = dict(os.environ, NGICP_KNN_STATS="1")
    p = subprocess.run([sys.executable, "-c", _DRIVER, ROOT, TESTS, name, str(k), str(path), str(cell)], env=env,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stderr.splitlines() if l.startswith("[ngicp knn]")]
    print(f"{name} k={k} path={path} cell={cell}:\n  " + "\n  ".join(lines))
    h, c = _HEAD.search(p.stderr), _CTRL.search(p.stderr)
    assert h and c, p.stderr[-2000:]
    n, _, ws, ties, _ = (int(v) for v in h.groups())
    rest, fix, slow, items, e4, e2, e1 = (int(v) for v in c.groups())
    assert n == int(p.stdout.split()[-1])
    assert rest == ws and slow + items == e4 + e2 + e1
    return dict(n=n, warp_search=ws, ties=ties, rest=rest, fix=fix, slow=slow, items=items, e4=e4, e2=e2, e1=e1)


def test_branches_reached():
    """Each cloud reaches the kernel branch it was built for (NGICP_KNN_STATS report of launch_covariances)."""
    s = knn_stats("lattice", 10)
    assert s["fix"] > 0 and s["ties"] > 0 and 0.5 * s["n"] < s["rest"] + s["fix"] <= s["n"]
    s = knn_stats("lattice", 20)
    assert s["fix"] > 0 and s["ties"] > 0 and 0.5 * s["n"] < s["rest"] + s["fix"] <= s["n"]
    s = knn_stats("hot_cell", 10)
    assert s["warp_search"] - s["ties"] > 0                        # tile overflow
    s = knn_stats("submap", 20, cell=4.0)
    assert s["e1"] > 0 and s["e2"] > 0                              # the plan split boxes down to single cells
    base = knn_stats("sparse_base", 10)
    s = knn_stats("sparse", 10)
    assert s["slow"] > 0 and s["slow"] >= base["slow"] + 48          # the isolated points and groups: slow boxes
    s = knn_stats("submap", 20, cell=0.1)
    assert s["slow"] > 0
    s = knn_stats("raw_submap", 20, path=0)                          # AUTO takes the tile path above 131,072 points
    assert s["n"] > R.TILE_MIN_POINTS and s["items"] + s["slow"] > 0
    for name, k in (("dupes", 10), ("flat", 16), ("line", 16), ("far", 20), ("nan_rows", 16)):
        s = knn_stats(name, k)
        assert s["rest"] + s["fix"] <= s["n"]
