"""CPU checks of the getFitnessScore restatement (tests/fitness_ref.py) the GPU fitness score is compared with: the
kd-tree nearest distances equal an exhaustive float32 search bit for bit, and PCL's filter quirks are kept (the SQUARED
distance compared with max_range, with <=; DBL_MAX when nothing qualifies)."""
import numpy as np
import pytest

import fitness_ref as F


@pytest.fixture(scope="module")
def clouds(orc):
    rng = np.random.default_rng(11)
    tgt = rng.uniform(-10.0, 10.0, size=(3000, 3)).astype(np.float32)
    src = (tgt[:2500] + rng.normal(0.0, 0.3, size=(2500, 3))).astype(np.float32)
    src = np.vstack([src, rng.uniform(-30.0, 30.0, size=(500, 3)).astype(np.float32)])
    c, s = np.cos(0.1), np.sin(0.1)
    T = np.array([[c, -s, 0, 0.2], [s, c, 0, -0.1], [0, 0, 1, 0.05], [0, 0, 0, 1]], dtype=np.float32)
    return src, tgt, T, orc.Cloud(tgt)


def test_restatement_matches_brute_force(clouds):
    src, tgt, T, cloud = clouds
    q = F.transform_f32(src, T)
    d_tree = F.nearest_d2(q, cloud)
    d_brute = F.brute_nearest_d2(q, tgt)
    assert np.array_equal(d_tree.view(np.uint32), d_brute.view(np.uint32))
    for r in (F.DBL_MAX, 1.0, 0.25, 0.01):
        a = F.fitness_score(src, cloud, T, r)
        b = F.score_from_d2(d_brute, r)
        assert a[1] == b[1] and a[0] == b[0]
    assert F.fitness_score(src, cloud, T)[1] == src.shape[0]


def test_transform_operation_order(clouds):
    src, _, T, _ = clouds
    q = F.transform_f32(src, T)
    f = np.float32
    for i in (0, 7, 2999):
        x, y, z = (f(v) for v in src[i])
        for r in range(3):
            ref = f(f(f(T[r, 0] * x) + f(T[r, 1] * y)) + f(f(T[r, 2] * z) + T[r, 3]))
            assert q[i, r].view(np.uint32) == ref.view(np.uint32)


def test_squared_distance_compared_with_le(clouds):
    """max_range equal to one squared distance (promoted to double) counts that point; one double ulp below does not."""
    src, _, T, cloud = clouds
    d2 = F.nearest_d2(F.transform_f32(src, T), cloud)
    pick = float(np.sort(d2)[len(d2) // 2])
    ties = int((d2 == np.float32(pick)).sum())
    s_at, n_at = F.fitness_score(src, cloud, T, pick)
    s_below, n_below = F.fitness_score(src, cloud, T, np.nextafter(pick, -np.inf))
    assert n_at == int((d2.astype(np.float64) <= pick).sum()) and n_at - n_below == ties >= 1
    assert s_at != s_below
    # the comparison is with max_range itself, not max_range^2: 0.5 admits distances up to sqrt(0.5) ~ 0.71 m
    assert F.fitness_score(src, cloud, T, 0.5)[1] == int((d2.astype(np.float64) <= 0.5).sum())
    assert F.fitness_score(src, cloud, T, 0.5)[1] > int((d2.astype(np.float64) <= 0.25).sum())


def test_nothing_qualifies_gives_dbl_max(clouds):
    src, _, T, cloud = clouds
    assert F.fitness_score(src, cloud, T, -1.0) == (F.DBL_MAX, 0)
    assert F.fitness_score(src[:0], cloud, T) == (F.DBL_MAX, 0)
    assert F.fitness_score(src, None, T) == (F.DBL_MAX, 0)
    Tn = T.copy()
    Tn[0, 0] = np.nan
    assert F.fitness_score(src, cloud, Tn) == (F.DBL_MAX, 0)
    # a point at 1e20 overflows its squared distance to inf and is never counted
    far = np.vstack([src[:10], np.array([[1e20, 0, 0]], dtype=np.float32)])
    assert F.fitness_score(far, cloud, np.eye(4, dtype=np.float32))[1] == 10
