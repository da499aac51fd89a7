"""CPU checks of tests/align_ref.py, the restatement the registration-kernel tests (test_gpu_align_adversarial.py) compare
the GPU with: it agrees with the oracle's NanoGICP::linearize / compute_error, and every cloud generator keeps the property
it was built for, measured on the data."""
import numpy as np
import pytest

import align_ref as A
import knn_ref as R


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    oracle.load(prefer_ref=False)
    return oracle


def test_restatement_matches_oracle_linearize(O):
    """Scan pair at a perturbed pose, thr = 1 m: the same correspondences off ties (and inside the tie set on ties),
    bit-identical distances, M within 1e-12 relative, and H / b / err within the summation bound of the exact sums of
    the per-point terms (plus 16 ulps per term: the oracle forms J^T M J with 4x4 products in another order)."""
    src, tgt = R.scan(O, 1), R.scan(O, 0)
    T = A.perturbed()
    thr = 1.0
    o = O.Gicp(k=10, max_corr_dist=thr, num_threads=1)
    o.set_target(O.Cloud(tgt)); o.set_source(O.Cloud(src))
    o.calc_target_covs(); o.calc_source_covs()
    lo = o.linearize(T, per_point=True)
    nn = A.NN1(O, tgt, A.transform_f32(src, T))
    has = nn.has_corr(thr)
    assert 0.5 < has.mean() < 1.0
    assert np.array_equal(lo["corr"] >= 0, has)
    assert np.array_equal(lo["sqd"][has].view(np.uint32), nn.d[has].view(np.uint32))
    assert nn.in_ties(lo["corr"])[has].all()
    single = has & (nn.nties == 1)
    assert np.array_equal(lo["corr"][single], nn.ties[single, 0])
    # M, restated from the oracle's own correspondences and covariances
    cs, ct = A.sym6(o.get_source_covs()), A.sym6(o.get_target_covs())
    m6 = A.mahal6(cs, ct, T[:3, :3], lo["corr"])
    mo = A.sym6(lo["mahalanobis"])
    rel = np.abs(m6 - mo).max(axis=1)[has] / np.abs(mo).max(axis=1)[has]
    assert rel.max() < 1e-12
    # sums: the oracle's M in the restated terms
    t = A.terms(src, tgt, T, lo["corr"], mo)
    exact, bound = A.exact_sums(t)
    slack = bound + 16 * A.U * np.abs(t).sum(axis=0)
    got = np.concatenate([A.pack_H(lo["H"]), lo["b"], [lo["err"]]])
    assert (np.abs(got - exact) <= slack).all(), np.abs(got - exact) / np.maximum(slack, 1e-300)
    # K5 on the frozen correspondences
    T2 = A.f32_pose(T @ A.perturbed(0.05, (0.01, 0.01, 0.0)))
    e = A.error_terms(src, tgt, T2, lo["corr"], mo)
    ex, bd = A.exact_sums(e)
    assert abs(o.compute_error(T2) - ex[0]) <= bd[0] + 16 * A.U * np.abs(e).sum()


def test_sums_bound_is_order_independent():
    """The bound holds for any summation order and is not loose: shuffled float64 sums of skewed terms stay inside it."""
    rng = np.random.default_rng(0)
    t = rng.normal(size=(20000, 3)) * np.exp(rng.normal(scale=6.0, size=(20000, 1)))
    exact, bound = A.exact_sums(t)
    for s in range(8):
        p = np.random.default_rng(s).permutation(t.shape[0])
        naive = np.zeros(3)
        for row in t[p]:
            naive = naive + row
        assert (np.abs(naive - exact) <= bound).all()
    assert (bound < 1e-9 * np.abs(t).sum(axis=0)).all()


def test_mahal_restatement_is_gicp_math_order():
    """sym3_rcr / sym3_inverse restated: the inverse of C_B + R C_A R^T, to rounding, on random SPD covariances."""
    rng = np.random.default_rng(1)
    n = 500
    X = rng.normal(size=(n, 3, 3))
    ca = X @ X.transpose(0, 2, 1) + 1e-3 * np.eye(3)
    Y = rng.normal(size=(n, 3, 3))
    cb = Y @ Y.transpose(0, 2, 1) + 1e-3 * np.eye(3)
    Rm = np.linalg.qr(rng.normal(size=(3, 3)))[0]
    m6 = A.mahal6(A.sym6(ca), A.sym6(cb), Rm, np.arange(n))
    ref = np.linalg.inv(cb + Rm @ ca @ Rm.T)
    M = A.mat4(m6)[:, :3, :3]
    assert np.allclose(M, ref, rtol=1e-8, atol=1e-8 * np.abs(ref).max())


def test_lattice_half_ties(O):
    src, tgt, T = A.lattice_half()
    nn = A.NN1(O, tgt, A.transform_f32(src, T))
    assert (nn.nties >= 2).all()
    assert (nn.nties == 8).mean() > 0.7
    assert np.isin(nn.nties, (2, 4, 8)).all()


def test_dupes_ties(O):
    tgt = R.dupes(O, 3)
    src = R.scan(O, 1, 1.0)
    nn = A.NN1(O, tgt, A.transform_f32(src, A.perturbed()))
    has = nn.has_corr(1.0)
    assert has.mean() > 0.5 and (nn.nties[has] >= 3).all()
    # the copies sit at the same position
    pos = tgt[nn.ties[has, :3], :3]
    assert (pos == pos[:, :1]).all()


@pytest.mark.parametrize("thr", [0.5, 0.3])
def test_straddlers_hit_the_threshold(O, thr):
    src, tgt, T = A.straddlers(thr)
    nn = A.NN1(O, tgt, A.transform_f32(src, T))
    prev, mid, nxt = A.straddle_values(thr)
    assert all(c >= 96 for c in A.straddle_counts(nn, thr))
    thr2 = thr * thr
    assert float(prev) < thr2 < float(nxt)
    # 0.25 is a float: the middle value equals thr^2 and is rejected by '<'; 0.09 is not: the middle is on one side
    assert (float(mid) == thr2) == (thr == 0.5)
    has = nn.has_corr(thr)
    assert has[nn.d == prev].all() and not has[nn.d == nxt].any()
    assert has[nn.d == mid].all() == (float(mid) < thr2)


def test_tail_bound_clouds(O):
    src, tgt = R.scan(O, 1), R.scan(O, 0)
    nn = A.NN1(O, tgt, A.transform_f32(src, A.perturbed()))
    assert A.tail_bound(nn, 0.05, 1.0).mean() > 0.5
    assert A.tail_bound(nn, 0.1, 1.0).sum() > 256
    fsrc, ftgt = A.far_sources(O)
    fn = A.NN1(O, ftgt, A.transform_f32(fsrc, np.eye(4)))
    n0 = src.shape[0]
    assert (fn.d[n0:].astype(np.float64) > 45.0 ** 2).all() and np.isfinite(fn.d[n0:]).all()


def test_non_finite_and_overflow_rows(O):
    src = R.scan(O, 1)
    bad, fin = R.nan_rows(src)
    ovf, keep = A.overflow_rows(src)
    assert (~fin).sum() > 100 and (~keep).sum() > 100
    T = A.perturbed(20.0)
    # at a rotated pose the 3e38 rows overflow in the float transform; at the identity they stay finite but every
    # squared distance to them is +inf, so they have no nearest point at all
    assert A.transform_overflows(ovf, T)[~keep].mean() > 0.5
    nn = A.NN1(O, R.scan(O, 0), A.transform_f32(ovf, np.eye(4)))
    assert np.isfinite(A.transform_f32(ovf, np.eye(4))[~keep]).all()
    assert np.isinf(nn.d[~keep]).all() and not nn.has_corr(float(np.finfo(np.float32).max))[~keep].any()
