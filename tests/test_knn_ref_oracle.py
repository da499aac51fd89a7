"""CPU checks of the kNN / covariance reference and the adversarial clouds (tests/knn_ref.py) the GPU kNN + covariance
kernels are tested against: the covariance restatement equals the oracle's REG_NONE covariances bit for bit, the
kd-tree distances equal brute force, and every generator still has the property it exists for (so that a later change
cannot quietly make the GPU tests easy again)."""
import numpy as np
import pytest

import knn_ref as R
from util import make_small_submap


def boundary_ties(d2, k):
    return d2[:, k - 1] == d2[:, k]


@pytest.fixture(scope="module")
def submap(orc):
    return make_small_submap(orc)[0]


@pytest.mark.parametrize("cloud", ["submap", "line", "lattice"])
def test_raw_cov_restatement_matches_oracle(orc, submap, cloud):
    """raw_cov_from_list on the oracle's own neighbour lists == oracle covariances(k, REG_NONE), bit for bit, wherever
    all k+1 distances are distinct (there the list, and so the summation order, is unique)."""
    xyz = {"submap": submap, "line": R.line(), "lattice": R.lattice()}[cloud]
    c = orc.Cloud(xyz)
    for k in (1, 2, 3, 5, 10, 16, 20, 31, 32):
        covs, idx, _ = c.covariances(k, orc.REG_NONE, with_knn=True)
        assert np.abs(covs[:, 3, :]).max() == 0 and np.abs(covs[:, :, 3]).max() == 0
        d2 = c.knn(np.ascontiguousarray(xyz[:, :3]), k + 1)[1]
        distinct = (d2[:, 1:] != d2[:, :-1]).all(axis=1)
        assert cloud == "lattice" or distinct.mean() > 0.99
        mine = R.raw_cov_from_list(xyz, idx)
        same = (mine.view(np.uint64) == R.cov6(covs).view(np.uint64)).all(axis=1)
        assert same[distinct].all(), (cloud, k, int((~same[distinct]).sum()))
        # summed in the oracle's own list order, ties included, the restatement is the oracle on every point
        assert same.all(), (cloud, k, int((~same).sum()))


def test_raw_cov_missing_neighbours():
    """A -1 entry is a zero column minus the mean."""
    xyz = np.array([[1.0, 2.0, 3.0], [4.0, -1.0, 0.5]], dtype=np.float32)
    got = R.raw_cov_from_list(xyz, np.array([[0, 1, -1]]))
    cols = np.array([[1.0, 2.0, 3.0], [4.0, -1.0, 0.5], [0.0, 0.0, 0.0]])
    d = cols - cols.mean(axis=0)
    ref = (d.T @ d) / 3.0
    assert np.allclose(got[0], ref[[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]], rtol=1e-15, atol=0)


def _generators(orc, submap):
    raw = R.raw_submap(orc)
    return {
        "lattice": R.lattice(), "dupes_2": R.dupes(orc, 2), "dupes_11": R.dupes(orc, 11), "hot_cell": R.hot_cell(orc),
        "flat": R.flat(), "line": R.line(), "sparse": R.sparse(orc, 10), "raw_submap": raw, "far": R.far(submap),
        "nan_rows": R.nan_rows(raw),
    }


@pytest.fixture(scope="module")
def gens(orc, submap):
    return _generators(orc, submap)


def test_kdtree_distances_equal_brute_force(orc, gens):
    """The distances knn_distances takes from the kd-tree above BRUTE_MAX_POINTS equal brute force on every cloud."""
    rng = np.random.default_rng(3)
    for name, c in gens.items():
        if name == "nan_rows":
            c = c[0][c[1]]
        xyz = np.ascontiguousarray(c[:, :3])
        q = xyz[rng.choice(xyz.shape[0], size=min(1500, xyz.shape[0]), replace=False)]
        tree = orc.Cloud(c).knn(q, 33)[1]
        brute = orc.Cloud(c, backend=orc.BACKEND_BRUTE).knn(q, 33)[1]
        assert np.array_equal(tree.view(np.uint32), brute.view(np.uint32)), name
    # and knn_distances itself on a cloud above the brute-force limit
    d = R.knn_distances(orc, gens["raw_submap"][:, :3].copy(), gens["raw_submap"][:4000], 21)
    assert d.shape == (4000, 21) and (np.diff(d, axis=1) >= 0).all()


def test_generators_keep_their_properties(orc, gens):
    g = gens
    xyz = lambda c: np.ascontiguousarray(c[:, :3])          # noqa: E731
    # lattice: boundary ties on most points at the k the tile kernel specialises, and ties inside the lists
    d = R.knn_distances(orc, xyz(g["lattice"]), g["lattice"], 21)
    for k in (10, 20):
        assert boundary_ties(d, k).mean() > 0.5
    assert (d[:, 1:11] == d[:, :10]).any(axis=1).mean() > 0.9
    # dupes_{k+1}: every k-th distance is 0 (k = 10)
    d = R.knn_distances(orc, xyz(g["dupes_11"]), g["dupes_11"], 11)
    assert (d[:, 10] == 0).all()
    d = R.knn_distances(orc, xyz(g["dupes_2"]), g["dupes_2"], 2)
    assert (d[:, 1] == 0).all()
    # hot_cell: HOT_COPIES bit-identical points (they share a cell at any cell edge) and the 2 cm cluster beside them
    hc = g["hot_cell"]
    _, counts = np.unique(hc[:, :3].view(np.dtype((np.void, 12))), return_counts=True)
    assert counts.max() >= R.HOT_COPIES
    hot = hc[(np.abs(hc[:, :3] - np.float32([6.0, -3.0, 0.5])) <= 0.02).all(axis=1)]
    assert hot.shape[0] >= R.HOT_COPIES + R.HOT_CLUSTER
    # flat: exactly coplanar
    assert (g["flat"][:, 2] == 0).all()
    # line: every neighbourhood (near-)collinear — the two smallest eigenvalues of the raw covariance vanish
    covs = orc.Cloud(g["line"]).covariances(10, orc.REG_NONE)[:, :3, :3]
    w = np.linalg.eigvalsh(covs)
    assert np.median(w[:, 1] / w[:, 2]) < 1e-6
    # sparse: isolated points farther than 3 m from everything, and groups whose (k+1)-th neighbour is metres away
    d = R.knn_distances(orc, xyz(g["sparse"]), g["sparse"], 12)
    assert (d[:, 1] > 9.0).sum() >= 60
    assert ((d[:, 10] < 1.0) & (d[:, 11] > 9.0)).sum() >= 32 * 11
    # raw_submap: large enough for AUTO to take the tile path
    assert g["raw_submap"].shape[0] > R.TILE_MIN_POINTS
    # far: more than 20 km from the origin
    assert (np.abs(g["far"][:, 0]) > 19000).all()
    # nan_rows: about 1 % of the rows non-finite, of every kind
    c, fin = g["nan_rows"]
    assert 0.005 < (~fin).mean() < 0.02
    bad = c[~fin][:, :3]
    assert np.isnan(bad).any() and np.isposinf(bad).any() and np.isneginf(bad).any()
