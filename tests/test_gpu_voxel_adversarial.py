"""The voxel grid (K0, csrc/voxel.cu) on clouds built to reach its edges (tests/voxel_ref.py), against the exact
restatement, through every launch path and entry point.

Paths: the fused cooperative kernel (voxel_path 0), the exact multi-kernel pipeline (voxel_path 1 on a fresh handle)
and the speculative multi-kernel pipeline (voxel_path 1 after a call that needed fewer, as many or more key bits).
Entry points: ngicp_voxel_filter, ngicp_preprocess (+-1 m negative crop), ngicp_transform_voxel_filter and
ngicp_preprocess_pointcloud2 (Ouster, Velodyne and xyz-only messages); input strides 12, 16 and 32; host and device
output buffers of capacity m and m - 1.  On every call: records bit-identical to the restatement (a NaN centroid
intensity compared by class: CUDA's canonical NaN and x86's propagated payload differ), the voxel of every input point,
the status, all paths bit-identical to each other, and ngicp_launch_count deltas that show which path ran.
"""
import ctypes as C

import numpy as np
import pytest

import voxel_ref as V

pytestmark = pytest.mark.gpu

CASES = V.cases(with_sizes=False)
IDS = [c.name for c in CASES]
CROP = 1.0
PC2_KINDS = (("ouster", 1, 0), ("velodyne", 2, 6), ("xyz", 1, 0))


@pytest.fixture(scope="module")
def G():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from direct_lidar_odometry_b200 import NanoGICP
    return NanoGICP


@pytest.fixture(scope="module")
def sms(G):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def T():
    from direct_lidar_odometry_b200 import synth
    return synth.trajectory_pose(57).astype(np.float32)


def strided(pts, stride):
    """The cloud as the library reads it at this stride, and the records that reading amounts to."""
    if stride == 32:
        return pts, pts
    if stride == 16:
        src = np.ascontiguousarray(np.c_[pts[:, :3], pts[:, 4]])
        return src, V.as_xyzi(src)
    src = np.ascontiguousarray(pts[:, :3])
    return src, V.as_xyzi(src)


def warm_cloud(b):
    """Two points at leaf 1 whose div_b product is 2^(b-1): the handle's next speculation sorts b key bits."""
    e0 = min(b - 1, 11)
    e1 = min(b - 1 - e0, 11)
    e2 = b - 1 - e0 - e1
    return V.as_xyzi(np.array([[0.5, 0.5, 0.5], [2.0**e0 - 0.5, 2.0**e1 - 0.5, 2.0**e2 - 0.5]], np.float32))


class Entry:
    """One call of an entry point through the C ABI with an explicit output buffer and capacity."""

    def __init__(self, kind, case, T, stride=32, pc2=None):
        from direct_lidar_odometry_b200 import pointcloud2
        self.kind, self.case, self.leaf = kind, case, case.leaf
        if kind == "pc2":
            name, height, pad = pc2
            n = case.pts.shape[0]
            self.msg = pointcloud2.make_pointcloud2(case.pts, name, height=height if n % height == 0 else 1, row_pad=pad)
            self.lay = pointcloud2.xyzi_layout(self.msg)
            self.data = np.frombuffer(self.msg.data, dtype=np.uint8)
            recs = V.from_ros_msg(self.msg)
            self.ref = V.pipeline(recs, self.leaf, crop=CROP)
        else:
            self.src, recs = strided(case.pts, stride)
            self.T = T
            if kind == "voxel":
                self.ref = V.pipeline(recs, self.leaf, compact_on_overflow=False)
            elif kind == "preprocess":
                self.ref = V.pipeline(recs, self.leaf, crop=CROP)
            else:
                self.ref = V.pipeline(recs, self.leaf, T=T)
        self.n = case.pts.shape[0]

    def bits(self):
        if self.kind == "transform":
            return V.key_bits(self.case.pts, self.leaf, T=self.T)
        return V.key_bits(self.case.pts, self.leaf, crop=CROP if self.kind in ("preprocess", "pc2") else None)

    def __call__(self, g, buf, cap):
        from direct_lidar_odometry_b200.nanogicp import _mat_to_abi, _ptr_n_stride
        L, h = g._L, g._h
        m = C.c_size_t(0)
        optr = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
        lo = (C.c_float * 3)(-CROP, -CROP, -CROP)
        hi = (C.c_float * 3)(CROP, CROP, CROP)
        if self.kind == "pc2":
            rc = L.ngicp_preprocess_pointcloud2(h, self.data.ctypes.data, C.byref(self.lay), lo, hi, C.c_float(self.leaf), optr, cap, C.byref(m))
        else:
            p, n, st, _ = _ptr_n_stride(self.src)
            if self.kind == "voxel":
                rc = L.ngicp_voxel_filter(h, p, n, st, C.c_float(self.leaf), optr, cap, C.byref(m))
            elif self.kind == "preprocess":
                rc = L.ngicp_preprocess(h, p, n, st, lo, hi, C.c_float(self.leaf), optr, cap, C.byref(m))
            else:
                Tc = _mat_to_abi(self.T, np.float32)
                rc = L.ngicp_transform_voxel_filter(h, p, n, st, Tc.ctypes.data_as(C.POINTER(C.c_float)), C.c_float(self.leaf), optr, cap, C.byref(m))
        return rc, m.value


def run(g, e, device=False, cap=None):
    """-> (status, records (numpy), launches)"""
    import torch
    cap = max(e.n, 1) if cap is None else cap
    buf = torch.zeros((max(cap, 1), 8), dtype=torch.float32, device="cuda") if device else np.zeros((max(cap, 1), 8), np.float32)
    c0 = g._L.ngicp_launch_count()
    rc, m = e(g, buf, cap)
    launches = g._L.ngicp_launch_count() - c0
    out = buf[:m].cpu().numpy() if device else buf[:m]
    return rc, np.ascontiguousarray(out), launches


def assert_records(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    gn, rn = np.isnan(got), np.isnan(ref)
    assert np.array_equal(gn, rn), what
    gb, rb = got.view(np.uint32).copy(), ref.view(np.uint32).copy()
    gb[gn] = 0
    rb[rn] = 0
    assert np.array_equal(gb, rb), (what, int((gb != rb).any(axis=1).sum()))


def check(g, e, what, device=False):
    rec, assign, st = e.ref
    rc, out, launches = run(g, e, device=device)
    assert rc == st, (what, rc, st)
    assert_records(out, rec, what)
    if assign is not None:
        assert np.array_equal(g.voxel_assignment(e.n), assign), what
    return out, launches


def all_paths(G, e, what, sms):
    """Every path on one entry call; returns the launch counts by path."""
    fused_fits = e.n <= sms * 4096
    outs, launches = {}, {}
    g = G(); g.setVoxelPath(0)
    outs["fused"], launches["fused"] = check(g, e, what + "/fused")
    g = G(); g.setVoxelPath(1)
    outs["exact"], launches["exact"] = check(g, e, what + "/exact")
    bits = e.bits()
    if bits is not None:
        for tag, b in (("fewer", max(1, bits - 9)), ("equal", bits), ("more", min(32, bits + 9))):
            g = G(); g.setVoxelPath(1)
            assert g.voxel_filter(warm_cloud(b), 1.0).shape[0] == (2 if b > 1 else 1)
            outs[tag], launches[tag] = check(g, e, f"{what}/spec_{tag}")
    for k, v in outs.items():
        assert np.array_equal(v.view(np.uint32), outs["exact"].view(np.uint32)), (what, k)
    st = e.ref[2]
    # which path ran: the fused kernel is one launch; the multi-kernel pipeline many.  A speculation with the right
    # width launches what the exact path does; one that was too narrow is redone by the exact path.
    if fused_fits and st == 0:
        assert launches["fused"] == 1, (what, launches)
    else:
        assert launches["fused"] > 1, (what, launches)
    assert launches["exact"] > 1
    if bits is not None:
        assert launches["equal"] == launches["exact"], (what, launches)
        assert launches["more"] >= launches["exact"], (what, launches)
        if bits > 1:
            assert launches["fewer"] > launches["exact"], (what, launches)
    return launches


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_every_path_entry_and_stride(G, T, sms, case):
    for kind in ("voxel", "preprocess", "transform"):
        for stride in (32, 16, 12):
            all_paths(G, Entry(kind, case, T, stride), f"{case.name}/{kind}/{stride}", sms)
    for pc2 in PC2_KINDS:
        all_paths(G, Entry("pc2", case, T, pc2=pc2), f"{case.name}/pc2-{pc2[0]}", sms)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_output_buffers_and_capacity(G, T, case):
    """Host and device output buffers of capacity m (bit-exact) and m - 1 (an error, nothing written past the end, and
    the handle works on), on the fused and the multi-kernel path."""
    for kind in ("voxel", "preprocess"):
        e = Entry(kind, case, T)
        rec, _, st = e.ref
        m = rec.shape[0]
        for path in (0, 1):
            g = G(); g.setVoxelPath(path)
            for device in (False, True):
                rc, out, _ = run(g, e, device=device, cap=max(m, 1))
                assert rc == st
                assert_records(out, rec, (case.name, kind, path, device))
                if m >= 1:
                    import torch
                    guard = 7
                    if device:
                        buf = torch.full((m - 1 + guard, 8), -5.0, dtype=torch.float32, device="cuda")
                    else:
                        buf = np.full((m - 1 + guard, 8), -5.0, np.float32)
                    rc, mm = e(g, buf, m - 1)
                    assert rc < 0, (case.name, kind, path, device, rc)
                    tail = buf[m - 1:].cpu().numpy() if device else buf[m - 1:]
                    assert (tail == -5.0).all()
                    check(g, e, f"{case.name}/{kind}/{path}/{device}/after-error", device=device)


@pytest.mark.parametrize("at", range(len(V.sizes())))
def test_sizes(G, T, sms, at):
    """Warp, block and chunk sizes, sms * 1024 +- 1, the fused kernel's limit sms * 4096 and the fallback past it."""
    n = V.sizes(sms)[at]
    case = V.Case(f"n{n}", V.size_cloud(n), 0.4)
    e = Entry("voxel", case, T)
    launches = all_paths(G, e, case.name, sms)
    if n > sms * 4096:
        assert launches["fused"] > 1
    g = G(); g.setVoxelPath(0)
    check(g, e, case.name + "/device", device=True)
