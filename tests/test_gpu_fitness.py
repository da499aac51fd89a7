"""getFitnessScore on the GPU (ngicp_fitness_score / ngicp_fitness_batch, csrc/fitness.cu) against the CPU restatement
of pcl::Registration::getFitnessScore (tests/fitness_ref.py): identical inlier counts and scores within 1e-10 relative
(the nearest distances are the kd-tree's bit for bit; only the fp64 summation order differs) on S2S, S2M and C2 inputs
and on the edge cases; the batch equal to the single calls bit for bit in two launches; the registration state left
alone; a device-assembled target; and the C++ facade."""
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

import fitness_ref as F
from direct_lidar_odometry_b200 import synth, _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "fitness_facade")
DBL_MAX = sys.float_info.max
S2S = dict(k=10, thr=1.0, max_iter=32, trans_eps=0.01)      # cfg/params.yaml:54-58
S2M = dict(k=20, thr=0.5, max_iter=32, trans_eps=0.01)      # cfg/params.yaml:63-67


@pytest.fixture(scope="module")
def G():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from direct_lidar_odometry_b200 import NanoGICP
    return NanoGICP


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    oracle.load(prefer_ref=True)
    return oracle


@pytest.fixture(scope="module")
def scans(O):
    out = []
    for i in (0, 1, 40, 41, 500, 501):
        T = synth.trajectory_pose(i)
        out.append(O.voxel_filter(synth.crop_box_negative(synth.os1_like(i, T)), 0.25))
    return out


def configure(g, cfg):
    g.setCorrespondenceRandomness(cfg["k"]); g.setMaxCorrespondenceDistance(cfg["thr"])
    g.setMaximumIterations(cfg["max_iter"]); g.setTransformationEpsilon(cfg["trans_eps"])


def make(G, src, tgt, cfg=S2S):
    g = G()
    configure(g, cfg)
    g.setInputTarget(tgt)
    g.setInputSource(src)
    return g


def assert_matches(got, ref):
    (s, n), (rs, rn) = got, ref
    assert n == rn, (got, ref)
    if rn == 0:
        assert s == DBL_MAX
    else:
        assert abs(s - rs) <= 1e-10 * abs(rs), (got, ref)


def test_s2s_against_oracle(G, O, scans):
    g = make(G, scans[1], scans[0])
    g.align()
    T = g.getFinalTransformation()
    cloud = O.Cloud(scans[0])
    d2 = F.nearest_d2(F.transform_f32(scans[1], T), cloud)
    pick = float(np.sort(d2)[len(d2) // 3])
    for r in (DBL_MAX, 1.0, 0.25, pick, np.nextafter(pick, -np.inf)):
        assert_matches(g.fitness(T, r), F.score_from_d2(d2, r))
    assert g.fitness(T, pick)[1] - g.fitness(T, np.nextafter(pick, -np.inf))[1] == int((d2 == np.float32(pick)).sum())
    # defaults: the final transformation and an unbounded range, like PCL
    assert g.getFitnessScore() == g.fitness(T)[0] and g.getFitnessScore(0.25) == g.fitness(T, 0.25)[0]
    assert g.fitness(T)[1] == scans[1].shape[0]


def test_s2m_small_submap_against_oracle(G, O):
    from util import make_small_submap
    submap, scan, Tm = make_small_submap(O)
    g = make(G, scan, submap, S2M)
    g.align(synth.perturb_pose(Tm, (0.2, 0.0, 0.0), 1.0).astype(np.float32))
    T = g.getFinalTransformation()
    cloud = O.Cloud(submap)
    for r in (DBL_MAX, 1.0, 0.25):
        assert_matches(g.fitness(T, r), F.fitness_score(scan, cloud, T, r))


def test_c2_workload_against_oracle(G, O):
    sys.path.insert(0, ROOT)
    import bench
    v = G()
    wl = bench.make_workload(lambda p, leaf: v.voxel_filter(p, leaf))
    submap, scan = wl["submap"], wl["scan_0"]
    g = make(G, scan, submap, S2M)
    g.align(wl["guesses"][0])
    T = g.getFinalTransformation()
    cloud = O.Cloud(submap)
    for r in (DBL_MAX, 0.25):
        assert_matches(g.fitness(T, r), F.fitness_score(scan, cloud, T, r))


def test_edge_cases(G, O, scans):
    src, tgt = scans[1], scans[0]
    cloud = O.Cloud(tgt)
    I = np.eye(4, dtype=np.float32)
    # far outside the target, unbounded: the search crosses empty space; bounded: nothing qualifies
    far = src.copy(); far[:, :3] += 500.0
    g = make(G, far, tgt)
    got = g.fitness(I)
    assert got[1] == far.shape[0]
    assert_matches(got, F.fitness_score(far, cloud, I))
    assert g.fitness(I, 1.0) == (DBL_MAX, 0)
    # a point at 1e20: its squared distance overflows to inf and is never counted
    odd = src.copy(); odd[5, 0] = 1e20
    g = G(); g.setInputTarget(tgt); g.registerInputSource(odd)   # the score needs no source index
    got = g.fitness(I)
    assert got[1] == odd.shape[0] - 1
    assert_matches(got, F.fitness_score(odd, cloud, I))
    # a NaN in the transform: no point is finite
    Tn = I.copy(); Tn[1, 2] = np.nan
    assert g.fitness(Tn) == (DBL_MAX, 0)
    # a one-point target
    one = tgt[:1].copy()
    g = make(G, src, one)
    assert_matches(g.fitness(I), F.fitness_score(src, O.Cloud(one), I))
    assert g.fitness(I)[1] == src.shape[0]
    # empty source or target: DBL_MAX, 0, no error (the mirror's setters refuse empty clouds like PCL's; the C ABI takes them)
    g = G(); g.setInputTarget(tgt); g._check(g._L.ngicp_set_source(g._h, None, 0, 32))
    assert g.fitness(I) == (DBL_MAX, 0)
    g = G(); g._check(g._L.ngicp_set_target(g._h, None, 0, 32)); g.setInputSource(src)
    assert g.fitness(I) == (DBL_MAX, 0)


def test_refusals(G, scans):
    from direct_lidar_odometry_b200 import NanoGICPError
    src, tgt = scans[1], scans[0]
    I = np.eye(4, dtype=np.float32)
    g = G(); g.setInputSource(src)
    with pytest.raises(NanoGICPError) as e:
        g.fitness(I)
    assert e.value.code == _lib.E_STATE
    # a target without a search index: a registered (unindexed) source swapped into the target role
    g = G(); g.registerInputSource(tgt); g.swapSourceAndTarget(); g.setInputSource(src)
    with pytest.raises(NanoGICPError) as e:
        g.fitness(I)
    assert e.value.code == _lib.E_STATE
    g = make(G, src, tgt)
    with pytest.raises(NanoGICPError) as e:
        g.fitness(I, float("nan"))
    assert e.value.code == _lib.E_INVALID
    # a sharded handle holds one slab of the submap
    g.set_owner_slab(0, -1.0, 1.0)
    with pytest.raises(NanoGICPError) as e:
        g.fitness(I)
    assert e.value.code == _lib.E_UNSUPPORTED
    g.set_owner_slab(-1)
    assert g.fitness(I)[1] == src.shape[0]


def batch_cases(O, scans):
    from util import make_small_submap
    submap, scan_m, Tm = make_small_submap(O)
    far = scans[0].copy(); far[:, :3] += 500.0
    return [  # (source, target, config, guess): the align_batch parity set, with the two-lanes-per-point S2M pair
        (scans[1], scans[0], S2S, None),
        (scans[3], scans[2], S2S, synth.perturb_pose(np.eye(4), (0.1, 0.05, 0.0), 0.5).astype(np.float32)),
        (scans[5], scans[4], dict(k=20, thr=float(np.finfo(np.float32).max), max_iter=64, trans_eps=5e-4), None),
        (scan_m, submap, S2M, synth.perturb_pose(Tm, (0.2, 0.0, 0.0), 1.0).astype(np.float32)),
        (far, scans[0], S2S, None),
        (scans[0], scans[1], S2S, None),
    ]


def test_batch_bit_identical_to_single_calls(G, O, scans):
    from direct_lidar_odometry_b200 import fitness_batch
    cases = batch_cases(O, scans)
    hs = [make(G, c[0], c[1], c[2]) for c in cases]
    for g, c in zip(hs, cases):
        g.align(c[3])
    for r in (DBL_MAX, 0.25):
        single = [g.fitness(None, r) for g in hs]
        scores, counts = fitness_batch(hs, max_range=r)
        again, counts2 = fitness_batch(hs, max_range=r)
        assert np.array_equal(scores.view(np.uint64), again.view(np.uint64)) and np.array_equal(counts, counts2)
        for (s, n), bs, bn in zip(single, scores, counts):
            assert np.float64(s).view(np.uint64) == bs.view(np.uint64) and n == bn
    assert counts[4] == 0 and counts[0] > 0   # the far pair has nothing within 0.25
    # explicit transforms, with None entries taking the final transformation
    Ts = [np.eye(4, dtype=np.float32), None, None, None, None, np.eye(4, dtype=np.float32)]
    scores, counts = fitness_batch(hs, Ts)
    for g, T, bs, bn in zip(hs, Ts, scores, counts):
        s, n = g.fitness(T)
        assert np.float64(s).view(np.uint64) == bs.view(np.uint64) and n == bn
    from direct_lidar_odometry_b200 import NanoGICPError
    with pytest.raises(NanoGICPError):
        fitness_batch([hs[0], hs[0]])
    with pytest.raises(NanoGICPError):
        fitness_batch([hs[0], G()])


def test_batch_constant_launches(G, scans):
    from direct_lidar_odometry_b200 import fitness_batch
    L = _lib.load()
    hs = [make(G, scans[(i + 1) % 6], scans[i % 6]) for i in range(64)]
    for B in (1, 64):
        fitness_batch(hs[:B])                       # warm: lazy module load, buffers
        c0 = L.ngicp_launch_count()
        scores, counts = fitness_batch(hs[:B])
        assert L.ngicp_launch_count() - c0 <= 2
        assert (counts > 0).all()
    c0 = L.ngicp_launch_count()
    hs[0].fitness()
    assert L.ngicp_launch_count() - c0 <= 2


def test_scoring_leaves_registration_alone(G, scans):
    g1, g2 = make(G, scans[1], scans[0]), make(G, scans[1], scans[0])
    guess = synth.perturb_pose(np.eye(4), (0.05, 0.0, 0.0), 0.2).astype(np.float32)
    g1.align(); g2.align()
    g1.fitness(None, 0.5)
    g1.fitness(np.eye(4, dtype=np.float32))
    g1.align(guess); g2.align(guess)
    assert np.array_equal(g1.final_state().view(np.uint64), g2.final_state().view(np.uint64))
    assert np.array_equal(g1.getFinalHessian().view(np.uint64), g2.getFinalHessian().view(np.uint64))
    T = g1.getFinalTransformation()
    assert g1.compute_error(T.astype(np.float64)) == g2.compute_error(T.astype(np.float64))


def test_kfstore_target_equals_host_target(G, scans):
    from direct_lidar_odometry_b200 import KeyframeStore
    src, a, b = scans[1], scans[0], scans[2]
    store = KeyframeStore(0)
    for part in (a, b):
        k = G(); configure(k, S2S)
        k.setInputSource(part); k.calculateSourceCovariances()
        store.push(k)
    dev = G(); configure(dev, S2S)
    store.set_target(dev, [0, 1])
    dev.setInputSource(src)
    host = make(G, src, np.vstack([a, b]))
    host.align()
    T = host.getFinalTransformation()
    for r in (DBL_MAX, 0.25):
        s1, n1 = dev.fitness(T, r)
        s2, n2 = host.fitness(T, r)
        assert n1 == n2 and np.float64(s1).view(np.uint64) == np.float64(s2).view(np.uint64)


def test_facade_fitness_matches_python_mirror(G, O, scans, tmp_path):
    assert os.path.exists(BIN), "build it with __graft_entry__.build() (make -C tests/cpp)"
    tgt, src, r = scans[0], scans[1], 0.25
    path = tmp_path / "clouds.bin"
    with open(path, "wb") as f:
        for c in (tgt, src):
            f.write(struct.pack("i", c.shape[0]))
            f.write(np.ascontiguousarray(c, dtype=np.float32).tobytes())
        f.write(struct.pack("d", r))
    out = subprocess.run([BIN, str(path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    rows = {d["case"]: d for d in (json.loads(l) for l in out.stdout.splitlines() if l.startswith("{"))}
    assert set(rows) == {"host_target", "kfstore_target", "no_target"}
    assert rows["no_target"]["score"] == DBL_MAX and "getFitnessScore" in out.stderr
    mirror = make(G, src, tgt)
    mirror.align()
    for name in ("host_target", "kfstore_target"):
        T = np.array(rows[name]["T"], dtype=np.float32).reshape(4, 4).T
        assert rows[name]["score"] == mirror.fitness(T)[0]
        assert rows[name]["score_r"] == mirror.fitness(T, r)[0]
    assert np.array_equal(np.array(rows["host_target"]["T"], dtype=np.float32).reshape(4, 4).T, mirror.getFinalTransformation())
    assert_matches(mirror.fitness(None, r), F.fitness_score(src, O.Cloud(tgt), mirror.getFinalTransformation(), r))
