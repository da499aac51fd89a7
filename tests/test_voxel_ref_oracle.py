"""CPU checks of tests/voxel_ref.py: the numpy restatement of the voxel grid equals the CPU oracle bit for bit on every
generator, and every generator has the property it was built for."""
import numpy as np
import pytest

import voxel_ref as V

CASES = V.cases()
IDS = [c.name for c in CASES]
F32 = np.float32


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def by_name(name):
    return next(c for c in CASES if c.name == name)


def grid_of(pts, leaf):
    fin, mn, mx = V.bbox(V.as_xyzi(pts)[:, :3])
    return fin, mn, mx, F32(1.0) / F32(leaf)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_restatement_equals_oracle(orc, case):
    ref, assign, st = V.voxel_filter(case.pts, case.leaf)
    out, oassign, rc = orc.voxel_filter(case.pts, case.leaf, return_assignment=True)
    assert st == rc
    assert ref.shape == out.shape and np.array_equal(bits(ref), bits(out))
    if st == 0:
        assert np.array_equal(assign, oassign)


@pytest.mark.parametrize("name", ["crop_faces", "dirty", "hot_voxel", "faces_0.25", "far_1e+13", "lonely"])
@pytest.mark.parametrize("crop", [1.0, None])
def test_preprocess_and_transform_equal_oracle(orc, name, crop):
    """removeNaN + negative CropBox + voxel grid, and transformPointCloud + voxel grid, against the oracle's steps."""
    from direct_lidar_odometry_b200 import synth
    c = by_name(name)
    ref, _, _ = V.pipeline(c.pts, c.leaf, crop=crop)
    assert np.array_equal(bits(ref), bits(orc.preprocess_points(c.pts, crop, c.leaf)))
    T = synth.trajectory_pose(57).astype(F32)
    ref, _, st = V.pipeline(c.pts, c.leaf, T=T)
    moved = synth.transform_xyzi(c.pts, T)
    if st == 0:
        assert np.array_equal(bits(ref), bits(orc.voxel_filter(moved, c.leaf)))
    else:
        assert np.array_equal(bits(ref), bits(orc.preprocess_points(moved, None, 0.0)))


@pytest.mark.parametrize("kind,height,pad", [("ouster", 1, 0), ("velodyne", 2, 6), ("xyz", 1, 0)])
def test_pointcloud2_decode_then_restatement(orc, kind, height, pad):
    """fromROSMsg (oracle.from_ros_msg) feeds the same records to the restatement as the plain clouds; xyz-only
    messages give intensity 0."""
    from direct_lidar_odometry_b200 import pointcloud2 as pc2
    c = by_name("dirty")
    msg = pc2.make_pointcloud2(c.pts, kind, height=height, row_pad=pad)
    dec = V.from_ros_msg(msg)
    want = c.pts.copy()
    if kind == "xyz":
        want[:, 4] = 0.0
    assert np.array_equal(bits(dec), bits(want))
    ref, _, _ = V.pipeline(dec, c.leaf, crop=1.0)
    assert np.array_equal(bits(ref), bits(orc.preprocess_points(dec, 1.0, c.leaf)))


# ------------------------------------------------------------------------------------------------ properties
def test_faces_land_on_and_next_to_integers():
    for leaf in (0.1, 0.3, 0.25):
        c = by_name(f"faces_{leaf}")
        fin, mn, mx, inv = grid_of(c.pts, leaf)
        q = c.pts[fin, :3] * inv
        r = np.round(q)
        below = q == np.nextafter(r.astype(F32), F32(-np.inf))
        assert below.mean() > 0.05, (leaf, below.mean())
        assert (q == r).mean() > 0.05 and (q < 0).mean() > 0.3
        assert np.signbit(c.pts[:, :3][c.pts[:, :3] == 0]).any()                 # -0.0
        tiny = np.abs(c.pts[:, :3])
        assert ((tiny > 0) & (tiny < np.finfo(F32).tiny)).any()                   # subnormals
        # floor and truncation differ on this cloud
        assert (np.floor(q) != np.trunc(q)).any()


@pytest.mark.parametrize("prod", sorted(V.PASS_EDGES))
def test_pass_edges_have_their_product(prod):
    c = by_name(f"pass_{prod}")
    fin, mn, mx, inv = grid_of(c.pts, 1.0)
    over, minb, div = V.grid_setup(mn, mx, inv)
    assert over == 0 and div[0] * div[1] * div[2] == prod
    assert V.key_bits(c.pts, 1.0) == prod.bit_length()
    keys = V.keys_of(c.pts[fin, :3], inv, minb, div)
    assert keys.max() == prod - 1                                               # the highest key is used
    assert (~fin).any()                                                         # and the invalid key (== prod)


def test_band_keys_cross_2_31(orc):
    c = by_name("band")
    fin, mn, mx, inv = grid_of(c.pts, 1.0)
    over, minb, div = V.grid_setup(mn, mx, inv)
    assert over == 0 and div == [1291, 1291, 1291]
    o_over, dprod, _, _ = V.old_guard(mn, mx, inv)
    assert not o_over and dprod == 1290**3
    prod = div[0] * div[1] * div[2]
    assert 2**31 < prod < 2**32
    keys = V.keys_of(c.pts[fin, :3], inv, minb, div)
    assert (keys >= 2**31).sum() > 100 and (keys < 2**31).sum() > 100
    signed = keys.astype(np.uint32).view(np.int32)
    assert not np.array_equal(np.argsort(signed, kind="stable"), np.argsort(keys, kind="stable"))


def test_slab_wrap_invalid_key_equals_a_finite_key():
    c = by_name("slab_wrap")
    fin, mn, mx, inv = grid_of(c.pts, 1.0)
    o_over, dprod, minb, div = V.old_guard(mn, mx, inv)
    assert not o_over and dprod == 2**30 + 129
    assert div == [2, 2, 2**30 + 129] and div[0] * div[1] * div[2] == 2**32 + 516
    old_invalid = (div[0] * div[1] * div[2]) % 2**32
    keys = V.keys_of(c.pts[fin, :3], inv, minb, div)
    assert old_invalid == 516 and (keys == old_invalid).sum() >= 2 and (~fin).any()
    assert V.grid_setup(mn, mx, inv)[0] == 1


def test_round_up_reaches_the_invalid_key():
    c = by_name("round_up")
    fin, mn, mx, inv = grid_of(c.pts, 1.0)
    o_over, dprod, minb, div = V.old_guard(mn, mx, inv)
    prod = div[0] * div[1] * div[2]
    assert not o_over and minb[0] == -1 and div[0] == 2**24 + 4 and prod < 2**32
    keys = V.keys_of(c.pts[fin, :3], inv, minb, div)
    assert (keys == prod).any()                                                 # a finite point on the invalid key
    assert V.grid_setup(mn, mx, inv)[0] == 1


@pytest.mark.parametrize("name", sorted(V.GUARD_EDGES))
def test_guard_edges_straddle_int32_max(name):
    c = by_name(f"guard_{name}")
    fin, mn, mx, inv = grid_of(c.pts, 1.0)
    _, dprod, _, _ = V.old_guard(mn, mx, inv)
    assert dprod == c.meta["prod"]
    assert (dprod > 2**31 - 1) == (name != "below_2^31-2")
    assert V.grid_setup(mn, mx, inv)[0] == (1 if dprod > 2**31 - 1 else 0)
    assert (dprod == 2**31 - 2) or (dprod >= 2**31)


@pytest.mark.parametrize("name", ["far_1e+13", "far_1e+20", "far_3e+38", "far_offset"])
def test_far_clouds_break_pcl_arithmetic(name):
    c = by_name(name)
    fin, mn, mx, inv = grid_of(c.pts, 0.25)
    o_over, dprod, minb, _ = V.old_guard(mn, mx, inv)
    if name == "far_offset":
        assert not o_over                                                       # PCL's guard lets it through
        assert abs(float(np.floor(mn[0] * inv))) > 2**31 and minb is None       # floor outside int32
    else:
        assert dprod is None or dprod >= 2**63                                  # int64 dx*dy*dz wraps / is undefined
        assert np.abs(c.pts[:, :3]).max() >= 1e13
    assert V.grid_setup(mn, mx, inv)[0] == 1


def test_hot_voxel_spans_many_chunks():
    c = by_name("hot_voxel")
    ref, assign, st = V.voxel_filter(c.pts, c.leaf)
    counts = np.bincount(assign[assign >= 0])
    assert st == 0 and counts.max() >= 20000 and counts.max() > 4 * 4096 // 4   # far more than one block's chunk
    where = np.nonzero(assign == counts.argmax())[0]
    assert where.min() < c.pts.shape[0] // 10 and where.max() > c.pts.shape[0] * 9 // 10


def test_sizes_are_as_named():
    got = sorted(c.pts.shape[0] for c in CASES if c.meta.get("gen") == "size")
    assert got == sorted(V.sizes(148)) and 148 * 4096 in got and 148 * 4096 + 1 in got


def test_dirty_and_lonely():
    c = by_name("dirty")
    xyz, it = c.pts[:, :3], c.pts[:, 4]
    single = (~np.isfinite(xyz)).sum(axis=1) == 1                              # one coordinate at a time
    for a in range(3):
        assert (np.isnan(xyz[:, a]) & single).any() and (np.isinf(xyz[:, a]) & single).any()
    fin = np.isfinite(xyz).all(axis=1)
    assert (np.isnan(it) & fin).any() and (np.isposinf(it) & fin).any() and (np.isneginf(it) & fin).any()
    ref, _, _ = V.voxel_filter(c.pts, c.leaf)
    assert np.isnan(ref[:, 4]).sum() >= 2 and np.isinf(ref[:, 4]).any() and np.isfinite(ref[:, :3]).all()
    lone = by_name("lonely")
    assert np.isfinite(lone.pts[:, :3]).all(axis=1).sum() == 1
    assert V.voxel_filter(lone.pts, lone.leaf)[0].shape[0] == 1


def test_crop_faces_move_min_b_if_counted():
    c = by_name("crop_faces")
    xyz = c.pts[:, :3]
    on_face = (np.abs(xyz) == 1.0).any(axis=1) & (np.abs(xyz) <= 1.0).all(axis=1)
    assert on_face.sum() >= 300
    drop = V.cropped(c.pts, 1.0)
    assert drop[on_face].all()
    just_out = xyz[:, 0] == np.nextafter(F32(1.0), F32(2.0))
    assert just_out.any() and not drop[just_out].any()
    inv = F32(1.0) / F32(c.leaf)
    _, minb_kept, _ = V.grid_setup(xyz[~drop].min(axis=0), xyz[~drop].max(axis=0), inv)
    _, minb_all, _ = V.grid_setup(xyz.min(axis=0), xyz.max(axis=0), inv)
    assert minb_kept[0] != minb_all[0]
    # a strict (<) crop would keep the face points
    strict = ((xyz > -1.0) & (xyz < 1.0)).all(axis=1)
    assert (drop & ~strict).sum() >= 300
