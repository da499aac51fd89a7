"""The registration linearisation (csrc/align.cu K4 linearize_block / finish_point, K5 error_point) point by point, on
clouds built to reach its rare branches, on every launch shape, against the exact CPU restatement in tests/align_ref.py.

Clouds: the voxelised scan pair at a perturbed pose; a lattice source shifted by exactly half a step (8-way distance
ties); a target whose points are all tripled (tied targets at one position); threshold straddlers at exactly
prev(thr^2), thr^2 and next(thr^2) for thr = 0.5 (thr^2 is a float) and 0.3 (it is not); forced cell edges of 0.1 and
0.05 m at thr = 1 m on the scan pair (the grid grows a forced edge its table cannot hold) and 0.05 m on the lattice
(every point goes through the shared-memory tail queue, which fills); an unbounded threshold with sources 50-1000 m
outside the target's box; NaN / Inf rows and (s, s, s), s = +-3e38 rows; thr = 0; sources of 1, 31,
33, 129 and 257 points against a ~90k-point submap; the scan-to-submap case.

Paths: the stepped linearize launch; the fused LM kernel (Gauss-Newton, max_iterations = 1, so its one linearisation is at
the guess: per-point state through ngicp_correspondences, H through final_hessian, the error through last_error); the
stepped align; the fused kernel with lanes per point and register variant forced (NGICP_ALIGN_LPP / NGICP_ALIGN_MINB, read
once per process: subprocesses); grids capped at 1 and 3 blocks (NGICP_ALIGN_MAX_BLOCKS: many round-robin passes); the
cluster-batched kernel with one-lane and two-lane pairs in one call.

On every point: corr >= 0 iff the query is finite and float64(d) < thr^2 for the exact nearest squared float distance d;
sqd is that d bit for bit (FLT_MAX without a correspondence); corr is one of the target points at distance d; M is
bit-identical to the restatement from the GPU's own corr.  Sums: H, b and err, and K5's error at a second pose on the
frozen correspondences, within gamma(n-1) * sum|t_i| of the exact sums.  Across paths: corr, sqd and M bit-identical —
one tie rule everywhere (strictly closer wins; among equals the earliest scanned row of the radius-1 cube, then the lowest
sorted slot; in the warp tail the lowest slot).

Queries whose squared distance to every target point overflows to +inf (a finite point near 3e38) get no correspondence
on the GPU.  The oracle (nanoflann's result-set semantics) keeps such a query when thr^2 > FLT_MAX (its result set still
holds FLT_MAX < thr^2) with a target index the search never set; the GPU does not follow it there.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import align_ref as A
import knn_ref as R
from util import make_small_submap

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = float(np.finfo(np.float32).max)
TINY = (1, 31, 33, 129, 257)
CASES = ("scan", "lattice_half", "lattice_cell_0.05", "dupes", "straddle_0.5", "straddle_0.3", "cell_0.1", "cell_0.05",
         "far_unbounded", "nonfinite", "nonfinite_unbounded", "thr0") + tuple(f"tiny_{n}" for n in TINY) + ("s2m",)
LOCAL_PATHS = ("stepped", "fused", "stepped_align")
FORCED = ((1, 1), (1, 2), (1, 3), (2, 2), (2, 3))     # (NGICP_ALIGN_LPP, NGICP_ALIGN_MINB)


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


class Case:
    def __init__(self, name, src, tgt, T, thr, k, cell=0.0, src_cov=None, tgt_cov=None, tgt_key=None):
        self.name, self.src, self.tgt, self.T, self.thr, self.k, self.cell = name, src, tgt, A.f32_pose(T), thr, k, cell
        self.src_cov, self.tgt_cov = src_cov, tgt_cov
        self.tgt_key = tgt_key or name

    def finish(self, O):
        self.q = A.transform_f32(self.src, self.T)
        self.nn = A.NN1(O, self.tgt, self.q)
        self.has = self.nn.has_corr(self.thr)
        self.cs6, self.ct6 = A.sym6(self.src_cov), A.sym6(self.tgt_cov)
        self.T2 = A.f32_pose(self.T @ A.perturbed(0.05, (0.01, 0.01, 0.0)))
        return self


def _covs(G, cloud, k):
    g = G()
    g.setCorrespondenceRandomness(k)
    g.setInputSource(cloud)
    g.calculateSourceCovariances()
    return g.getSourceCovariances()


class Cases:
    def __init__(self, G, O):
        self.G, self.O, self.c, self.memo = G, O, {}, {}

    def cov(self, key, cloud, k):
        if (key, k) not in self.memo:
            self.memo[(key, k)] = _covs(self.G, cloud, k)
        return self.memo[(key, k)]

    def __getitem__(self, name):
        if name not in self.c:
            self.c[name] = self._make(name).finish(self.O)
        return self.c[name]

    def _make(self, name):
        O, cov = self.O, self.cov
        if name in ("scan", "cell_0.1", "cell_0.05", "thr0", "nonfinite", "nonfinite_unbounded"):
            src, tgt = R.scan(O, 1), R.scan(O, 0)
            cs, ct = cov("scan1", src, 10), cov("scan0", tgt, 10)
            thr = {"thr0": 0.0, "nonfinite_unbounded": FLT_MAX}.get(name, 1.0)
            cell = float(name[5:]) if name.startswith("cell_") else 0.0
            if name.startswith("nonfinite"):
                src, _ = R.nan_rows(src)
                src, _ = A.overflow_rows(src)
            return Case(name, src, tgt, A.perturbed(), thr, 10, cell, cs, ct, tgt_key="scan0" if cell == 0 else name)
        if name.startswith("lattice_"):
            src, tgt, T = A.lattice_half()
            cell = 0.05 if name == "lattice_cell_0.05" else 0.0
            return Case(name, src, tgt, T, 1.0, 10, cell, cov("lh_src", src, 10), cov("lh_tgt", tgt, 10),
                        tgt_key="lattice_half" if cell == 0 else name)
        if name == "dupes":
            src, tgt = R.scan(O, 1, 1.0), R.dupes(O, 3)
            return Case(name, src, tgt, A.perturbed(), 1.0, 10, 0.0, cov("d_src", src, 10), cov("d_tgt", tgt, 10))
        if name.startswith("straddle_"):
            thr = float(name[9:])
            src, tgt, T = A.straddlers(thr)
            return Case(name, src, tgt, T, thr, 10, 0.0, cov(name + "s", src, 10), cov(name + "t", tgt, 10))
        if name == "far_unbounded":
            src, tgt = A.far_sources(O)
            return Case(name, src, tgt, np.eye(4), FLT_MAX, 10, 0.0, cov("far_src", src, 10), cov("scan0", tgt, 10),
                        tgt_key="scan0")
        submap, scan, Ts = self.s2m()
        ct = cov("submap", submap, 20)
        cs = cov("s2m_scan", scan, 20)
        guess = A.f32_pose(A.synth.perturb_pose(Ts, (0.1, -0.05, 0.02), 0.5))
        if name == "s2m":
            return Case(name, scan, submap, guess, 0.5, 20, 0.0, cs, ct, tgt_key="submap")
        n = int(name[5:])
        return Case(name, np.ascontiguousarray(scan[:n]), submap, guess, 1.0, 20, 0.0, cs[:n], ct, tgt_key="submap")

    def s2m(self):
        if "s2m" not in self.memo:
            self.memo["s2m"] = make_small_submap(self.O)
        return self.memo["s2m"]


@pytest.fixture(scope="module")
def cases(G, O):
    return Cases(G, O)


# ---------------------------------------------------------------------------------------------- running a path
def _handle(G, c, align_mode=0):
    g = G()
    g.setCorrespondenceRandomness(c.k)
    g.setMaxCorrespondenceDistance(c.thr)
    if c.cell > 0:
        g.setGridCellSize(c.cell)
    g.setOptimizer(0)                 # Gauss-Newton: final_hessian is H at the (only) linearisation
    g.setMaximumIterations(1)
    g.setAlignMode(align_mode)
    g.setInputTarget(c.tgt)
    g.setInputSource(c.src)
    g.setTargetCovariances(c.tgt_cov)
    g.setSourceCovariances(c.src_cov)
    return g


def _after_align(g, c):
    r = g.correspondences()
    r.update(H=g.getFinalHessian(), b=None, err=g.result.last_error, err2=g.compute_error(c.T2))
    return r


def run_path(G, c, path):
    if path == "stepped":
        g = _handle(G, c)
        r = g.linearize(c.T, per_point=True)
        r["mahal"] = r.pop("mahalanobis")
        r["err2"] = g.compute_error(c.T2)
        acc = g.correspondences()     # the accessor reports what linearize returned
        assert np.array_equal(acc["corr"], r["corr"]) and np.array_equal(acc["sqd"].view(np.uint32), r["sqd"].view(np.uint32))
        assert np.array_equal(acc["mahalanobis"].view(np.uint64), r["mahal"].view(np.uint64))
        r["cell"] = g.grid_info(1)["cell"]
        return r
    g = _handle(G, c, align_mode=1 if path == "stepped_align" else 0)
    g.align(c.T.astype(np.float32))
    r = _after_align(g, c)
    r["mahal"] = r.pop("mahalanobis")
    return r


def _where(mask, what):
    rows = np.nonzero(mask)[0]
    return f"{what} at {rows.size} rows, first {rows[:8].tolist()}"


def check_points(c, r, where):
    corr, sqd = r["corr"], r["sqd"]
    bad = (corr >= 0) != c.has
    assert not bad.any(), f"{c.name} / {where}: correspondence rule " + _where(bad, "differs")
    bad = c.has & (sqd.view(np.uint32) != c.nn.d.view(np.uint32))
    assert not bad.any(), f"{c.name} / {where}: sqd " + _where(bad, "is not the exact minimum")
    bad = ~c.has & (sqd != np.float32(FLT_MAX))
    assert not bad.any(), f"{c.name} / {where}: sqd " + _where(bad, "is not FLT_MAX without a correspondence")
    bad = c.has & ~c.nn.in_ties(corr)
    assert not bad.any(), f"{c.name} / {where}: corr " + _where(bad, "is not a nearest point")
    m6 = A.mahal6(c.cs6, c.ct6, c.T[:3, :3], corr)
    got = A.sym6(r["mahal"])
    bad = (got.view(np.uint64) != m6.view(np.uint64)).any(axis=1)
    assert not bad.any(), f"{c.name} / {where}: M " + _where(bad, "differs from the restatement")
    assert not r["mahal"][:, 3, :].any() and not r["mahal"][:, :, 3].any()
    return m6


def check_sums(c, r, m6, where):
    t = A.terms(c.src, c.tgt, c.T, r["corr"], m6)
    exact, bound = A.exact_sums(t)
    got = A.pack_H(r["H"])
    bad = np.abs(got - exact[:21]) > bound[:21]
    assert not bad.any(), f"{c.name} / {where}: H entries {np.nonzero(bad)[0].tolist()} outside the bound"
    if r.get("b") is not None:
        assert (np.abs(r["b"] - exact[21:27]) <= bound[21:27]).all(), f"{c.name} / {where}: b outside the bound"
    assert abs(r["err"] - exact[27]) <= bound[27], f"{c.name} / {where}: err {r['err']!r} vs {exact[27]!r} +- {bound[27]!r}"
    e = A.error_terms(c.src, c.tgt, c.T2, r["corr"], m6)
    ex, bd = A.exact_sums(e)
    assert abs(r["err2"] - ex[0]) <= bd[0], f"{c.name} / {where}: K5 error {r['err2']!r} vs {ex[0]!r} +- {bd[0]!r}"


def check_same(c, r, ref, where):
    for key, view in (("corr", np.int32), ("sqd", np.uint32), ("mahal", np.uint64)):
        bad = ref[key].view(view) != r[key].view(view)
        if bad.ndim > 1:
            bad = bad.reshape(bad.shape[0], -1).any(axis=1)
        assert not bad.any(), f"{c.name}: {key} of {where} differs from the stepped linearize " + _where(bad, "")


@pytest.fixture(scope="module")
def stepped(G, cases):
    memo = {}

    def get(name):
        if name not in memo:
            memo[name] = run_path(G, cases[name], "stepped")
        return memo[name]
    return get


# ---------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("path", LOCAL_PATHS)
@pytest.mark.parametrize("name", CASES)
def test_points_and_sums(G, cases, stepped, name, path):
    c = cases[name]
    r = stepped(name) if path == "stepped" else run_path(G, c, path)
    m6 = check_points(c, r, path)
    check_sums(c, r, m6, path)
    if path != "stepped":
        check_same(c, r, stepped(name), path)


@pytest.mark.parametrize("blocks", [1, 3])
def test_max_blocks_many_passes(G, cases, stepped, monkeypatch, blocks):
    """A grid capped at 1 or 3 blocks runs the round-robin chunk dealing over many passes (read at handle creation)."""
    monkeypatch.setenv("NGICP_ALIGN_MAX_BLOCKS", str(blocks))
    for name in ("scan", "lattice_half", "lattice_cell_0.05", "cell_0.05", "far_unbounded", "nonfinite", "tiny_257", "s2m"):
        c = cases[name]
        for path in ("stepped", "fused"):
            r = run_path(G, c, path)
            where = f"{path}, {blocks} blocks"
            check_sums(c, r, check_points(c, r, where), where)
            check_same(c, r, stepped(name), where)


_DRIVER = r"""
import sys
sys.path[:0] = [sys.argv[1]]
import numpy as np
from direct_lidar_odometry_b200 import NanoGICP
d = np.load(sys.argv[2])
out = {}
for nm in [str(s) for s in d["names"]]:
    g = NanoGICP(0)
    g.setCorrespondenceRandomness(int(d[nm + "|k"])); g.setMaxCorrespondenceDistance(float(d[nm + "|thr"]))
    if float(d[nm + "|cell"]) > 0: g.setGridCellSize(float(d[nm + "|cell"]))
    g.setOptimizer(0); g.setMaximumIterations(1)
    tk = str(d[nm + "|tgt_key"])
    g.setInputTarget(d[tk + "|tgt"]); g.setInputSource(d[nm + "|src"])
    g.setTargetCovariances(d[tk + "|tgt_cov"]); g.setSourceCovariances(d[nm + "|src_cov"])
    g.align(d[nm + "|T"].astype(np.float32))
    c = g.correspondences()
    out[nm + "|corr"], out[nm + "|sqd"], out[nm + "|mahal"] = c["corr"], c["sqd"], c["mahalanobis"]
    out[nm + "|H"], out[nm + "|err"] = g.getFinalHessian(), np.float64(g.result.last_error)
    out[nm + "|err2"] = np.float64(g.compute_error(d[nm + "|T2"]))
np.savez(sys.argv[3], **out)
"""


def test_forced_lanes_and_register_variants(cases, stepped, tmp_path):
    """Every compiled variant of the fused kernel — one or two lanes per point, 255 / 128 / 80 registers — on every cloud
    (NGICP_ALIGN_LPP / NGICP_ALIGN_MINB are read once per process)."""
    blob = {"names": np.array(CASES)}
    for name in CASES:
        c = cases[name]
        for key, v in (("k", c.k), ("thr", c.thr), ("cell", c.cell), ("tgt_key", c.tgt_key), ("src", c.src),
                       ("src_cov", c.src_cov), ("T", c.T), ("T2", c.T2)):
            blob[f"{name}|{key}"] = np.asarray(v)
        blob[f"{c.tgt_key}|tgt"], blob[f"{c.tgt_key}|tgt_cov"] = c.tgt, c.tgt_cov
    inp = tmp_path / "in.npz"
    np.savez(inp, **blob)
    for lpp, minb in FORCED:
        out = tmp_path / f"out_{lpp}_{minb}.npz"
        env = dict(os.environ, NGICP_ALIGN_LPP=str(lpp), NGICP_ALIGN_MINB=str(minb))
        p = subprocess.run([sys.executable, "-c", _DRIVER, ROOT, str(inp), str(out)], env=env, capture_output=True,
                           text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        d = np.load(out)
        for name in CASES:
            c = cases[name]
            r = {k: d[f"{name}|{k}"] for k in ("corr", "sqd", "mahal", "H", "err2")}
            r["err"], r["b"] = float(d[f"{name}|err"]), None
            where = f"fused, LPP {lpp}, MINB {minb}"
            check_sums(c, r, check_points(c, r, where), where)
            check_same(c, r, stepped(name), where)


def test_batch_mixes_one_and_two_lane_pairs(G, cases, stepped):
    """align_batch with scan-to-scan (one lane per point) and scan-to-submap pairs (two lanes) in one call: the
    cluster's virtual blocks leave every handle the state its single fused launch would."""
    from direct_lidar_odometry_b200 import nanogicp
    names = ("scan", "s2m", "tiny_257", "lattice_half", "far_unbounded", "cell_0.05", "tiny_1")
    hs = [_handle(G, cases[n]) for n in names]
    nanogicp.align_batch(hs, [cases[n].T.astype(np.float32) for n in names])
    for n, g in zip(names, hs):
        c = cases[n]
        r = _after_align(g, c)
        r["mahal"] = r.pop("mahalanobis")
        check_sums(c, r, check_points(c, r, "batch"), "batch")
        check_same(c, r, stepped(n), "batch")


@pytest.mark.parametrize("name", ["nonfinite", "nonfinite_unbounded"])
def test_non_finite_rows_change_nothing(G, cases, stepped, name):
    """NaN / Inf rows and 3e38 rows in the source leave every other point's correspondence, distance and M unchanged."""
    c = cases[name]
    clean = Case("clean", R.scan(cases.O, 1), c.tgt, c.T, c.thr, c.k, 0.0, c.src_cov, c.tgt_cov)
    clean.T2 = c.T2
    rc = run_path(G, clean, "stepped")
    r = stepped(name)
    fin = np.isfinite(c.src[:, :3]).all(axis=1) & (np.abs(c.src[:, :3]) < 1e38).all(axis=1)
    assert (~fin).sum() > 200 and (r["corr"][~fin] == -1).all()
    assert np.array_equal(r["corr"][fin], rc["corr"][fin])
    assert np.array_equal(r["sqd"][fin].view(np.uint32), rc["sqd"][fin].view(np.uint32))
    assert np.array_equal(r["mahal"][fin].view(np.uint64), rc["mahal"][fin].view(np.uint64))


def test_thr_zero_gives_nothing(cases, stepped):
    r = stepped("thr0")
    assert (r["corr"] == -1).all() and (r["sqd"] == np.float32(FLT_MAX)).all()
    assert not r["H"].any() and not r["b"].any() and r["err"] == 0.0 and r["err2"] == 0.0


def test_slab_bounds_count_once(G, cases, stepped):
    """set_owner_slab: source points whose transformed x lies exactly on the bound are counted by exactly one of the
    complementary slabs [lo, b) and [b, hi); the two slabs' points together are the unfiltered correspondences."""
    c = cases["lattice_half"]
    b = float(np.float32(0.0625 + 0.125 * 19))
    on = c.q[:, 0] == np.float32(b)
    assert on.sum() > 100
    full = stepped("lattice_half")
    parts = []
    for lo, hi in ((-3e38, b), (b, 3e38)):
        g = _handle(G, c)
        g.set_owner_slab(0, lo, hi)
        r = g.linearize(c.T, per_point=True)
        parts.append(r)
    a, bb = parts[0]["corr"] >= 0, parts[1]["corr"] >= 0
    assert not (a & bb).any() and np.array_equal(a | bb, full["corr"] >= 0)
    assert bb[on].all() and not a[on].any()
    for r, m in ((parts[0], a), (parts[1], bb)):
        assert np.array_equal(r["corr"][m], full["corr"][m])
    # the slab sums add up to the whole: each within its own bound of the exact sum of its points
    m6 = A.mahal6(c.cs6, c.ct6, c.T[:3, :3], full["corr"])
    for r in parts:
        t = A.terms(c.src, c.tgt, c.T, r["corr"], m6)
        exact, bound = A.exact_sums(t)
        assert (np.abs(A.pack_H(r["H"]) - exact[:21]) <= bound[:21]).all()


def test_clouds_reach_their_branches(cases, stepped):
    """Each cloud has the property it was built for, measured from the exact reference (printed as a table)."""
    rows = []
    for name in CASES:
        c = cases[name]
        r = stepped(name)
        cell = r["cell"]                 # the grid's actual edge: a forced edge grows when the table cannot hold it
        ties = int((c.has & (c.nn.nties >= 2)).sum())
        strad = sum(A.straddle_counts(c.nn, c.thr)) if 0 < c.thr < FLT_MAX else 0
        tail = int(A.tail_bound(c.nn, cell, c.thr if c.thr > 0 else 0.0).sum())
        nonfin = int((~np.isfinite(c.q).all(axis=1) | ~np.isfinite(c.nn.d)).sum())
        lpp = 2 if c.tgt.shape[0] >= 4 * c.src.shape[0] else 1
        rows.append((name, c.src.shape[0], c.tgt.shape[0], ties, strad, tail, nonfin, lpp, cell))
        if name.startswith("lattice_") or name == "dupes":
            assert ties > 0.5 * c.has.sum()
        if name == "lattice_cell_0.05":     # every point is tail-bound: every block's queue holds all of its points
            assert cell == np.float32(0.05) and tail == c.src.shape[0]
        if name.startswith("straddle_"):
            assert strad >= 3 * 96
        if name in ("cell_0.1", "cell_0.05"):
            assert cell < 0.5 and tail > 0
        if name == "far_unbounded":
            assert tail >= 600
        if name.startswith("nonfinite"):
            assert nonfin > 200
    print("\n| cloud | source | target | tied | straddlers | tail-bound | non-finite | LPP (auto) | cell |")
    print("|---|---|---|---|---|---|---|---|---|")
    for row in rows:
        print("| " + " | ".join(f"{v:.3g}" if isinstance(v, float) else str(v) for v in row) + " |")
