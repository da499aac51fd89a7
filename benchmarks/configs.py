#!/usr/bin/env python
"""Secondary benchmarks for the other BASELINE.json configs (bench.py is the headline C2 run):

  c1  single OS1-64-like scan pair, S2S align (shipped DLO cfg and library defaults), GPU vs CPU oracle
  c3  odometry replay: the OdomNode S2S + S2M + keyframe/submap sequence over a synthetic trajectory
  c4  independent scan-pair batch throughput (pairs/s), several handles/streams per GPU; under torchrun the pairs
      are partitioned over ranks (direct_lidar_odometry_b200.sharded.partition_pairs)
  c5  dense 128-beam scan (no voxel filter) against a multi-million-point submap sharded over the ranks of one box:
      every rank holds one slab (+ halo) of the target, the LM loop runs as one persistent kernel per GPU and the
      partial H/b/err meet in NVLink peer memory (ngicp_comm_*); run under torchrun, e.g.
      python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 benchmarks/configs.py c5

    python benchmarks/configs.py c1
    python benchmarks/configs.py c3 --scans 300 --cpu-scans 40
    python benchmarks/configs.py c4 --pairs 512 --handles 8

Prints one JSON object per config.  Scan generation (numpy ray casting) is parallelised over host processes.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from direct_lidar_odometry_b200 import synth  # noqa: E402

S2S = dict(k=10, thr=1.0, max_iter=32, trans_eps=0.01)     # cfg/params.yaml:54-58
S2M = dict(k=20, thr=0.5, max_iter=32, trans_eps=0.01)     # cfg/params.yaml:63-67
DEFAULTS = dict(k=20, thr=float(np.finfo(np.float32).max), max_iter=64, trans_eps=5e-4)


def _gen(i):
    T = synth.trajectory_pose(i)
    return i, T, synth.crop_box_negative(synth.os1_like(i, T))


def gen_scans(indices):
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        out = list(ex.map(_gen, indices, chunksize=4))
    return {i: (T, s) for i, T, s in out}


def configure(g, cfg):
    g.setCorrespondenceRandomness(cfg["k"]); g.setMaxCorrespondenceDistance(cfg["thr"])
    g.setMaximumIterations(cfg["max_iter"]); g.setTransformationEpsilon(cfg["trans_eps"])


def pose_err(Ta, Tb):
    dt = float(np.linalg.norm(np.asarray(Ta, float)[:3, 3] - np.asarray(Tb, float)[:3, 3]))
    dR = np.asarray(Ta, float)[:3, :3].T @ np.asarray(Tb, float)[:3, :3]
    sk = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])   # well conditioned near identity
    return dt, float(np.arcsin(min(1.0, float(np.linalg.norm(sk)))))


# ------------------------------------------------------------------------------------------------ C1
def run_c1(args):
    import torch
    from direct_lidar_odometry_b200 import NanoGICP
    from oracle import oracle as O
    scans = gen_scans([0, 1])
    (T0, s0), (T1, s1) = scans[0], scans[1]
    truth = np.linalg.inv(T0) @ T1
    out = {"config": "C1: single OS1-64-like scan pair, voxel 0.25 m, S2S align", "raw_points": [int(s0.shape[0]), int(s1.shape[0])]}
    g = NanoGICP(0)
    threads = os.cpu_count()
    for name, cfg in (("dlo_s2s_cfg", S2S), ("library_defaults", DEFAULTS)):
        configure(g, cfg)

        def gpu_once():
            g.clearSource(); g.clearTarget()
            t0 = time.perf_counter()
            v0 = g.voxel_filter(s0, 0.25); v1 = g.voxel_filter(s1, 0.25)
            t1 = time.perf_counter()
            g.setInputTarget(v0); g.calculateTargetCovariances()
            g.setInputSource(v1); g.calculateSourceCovariances()
            g.sync()
            t2 = time.perf_counter()
            g.align()
            t3 = time.perf_counter()
            return v0, v1, (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3
        for _ in range(5):
            gpu_once()
        reps = [gpu_once() for _ in range(20)]
        v0, v1 = reps[0][0], reps[0][1]
        tm = g.timings()
        gpu = {"voxel_ms": float(np.median([r[2] for r in reps])), "index_and_covs_ms": float(np.median([r[3] for r in reps])),
               "align_ms": float(np.median([r[4] for r in reps])), "align_kernel_ms": tm["align_ms"],
               "iterations": int(g.result.nr_iterations), "trials": int(g.result.n_compute_error)}
        gpu["total_ms"] = gpu["voxel_ms"] + gpu["index_and_covs_ms"] + gpu["align_ms"]

        # the same pair with the voxelised clouds left on the device (out= a CUDA tensor, the additive use of the same calls):
        # no 0.7 MB device-to-host-to-device round trip per cloud between the voxel filter and setInput*
        ob = [torch.zeros((s.shape[0], 8), dtype=torch.float32, device="cuda") for s in (s0, s1)]

        def gpu_dev_once():
            g.clearSource(); g.clearTarget()
            t0 = time.perf_counter()
            d0 = g.voxel_filter(s0, 0.25, out=ob[0]); d1 = g.voxel_filter(s1, 0.25, out=ob[1])
            t1 = time.perf_counter()
            g.setInputTarget(d0); g.calculateTargetCovariances()
            g.setInputSource(d1); g.calculateSourceCovariances()
            g.sync()
            t2 = time.perf_counter()
            g.align()
            t3 = time.perf_counter()
            return (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, g.final_state().copy()
        for _ in range(5):
            gpu_dev_once()
        dreps = [gpu_dev_once() for _ in range(20)]
        gpu_dev = {"voxel_ms": float(np.median([r[0] for r in dreps])), "index_and_covs_ms": float(np.median([r[1] for r in dreps])),
                   "align_ms": float(np.median([r[2] for r in dreps]))}
        gpu_dev["total_ms"] = gpu_dev["voxel_ms"] + gpu_dev["index_and_covs_ms"] + gpu_dev["align_ms"]
        gpu_once()
        gpu_dev["result_bit_identical_to_host_path"] = bool(np.array_equal(dreps[0][3], g.final_state()))

        def cpu_once():
            t0 = time.perf_counter()
            c0 = O.voxel_filter(s0, 0.25); c1 = O.voxel_filter(s1, 0.25)
            t1 = time.perf_counter()
            tgt, src = O.Cloud(c0), O.Cloud(c1)
            o = O.Gicp(k=cfg["k"], max_corr_dist=cfg["thr"], max_iter=cfg["max_iter"], trans_eps=cfg["trans_eps"], num_threads=threads)
            o.set_target(tgt); o.set_source(src)
            o.calc_target_covs(); o.calc_source_covs()
            t2 = time.perf_counter()
            r = o.align()
            t3 = time.perf_counter()
            return r, (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3
        cpu_once()
        creps = [cpu_once() for _ in range(10)]
        r = creps[0][0]
        cpu = {"voxel_ms": float(np.median([c[1] for c in creps])), "index_and_covs_ms": float(np.median([c[2] for c in creps])),
               "align_ms": float(np.median([c[3] for c in creps])), "iterations": int(r.nr_iterations), "trials": int(r.n_compute_error),
               "threads": threads}
        cpu["total_ms"] = cpu["voxel_ms"] + cpu["index_and_covs_ms"] + cpu["align_ms"]
        dt, dr = pose_err(g.final_state(), r.Tx())
        et, er = pose_err(g.final_state(), truth)
        out[name] = {"points": [int(v0.shape[0]), int(v1.shape[0])], "gpu": gpu, "gpu_device_resident": gpu_dev, "cpu": cpu,
                     "speedup_align": cpu["align_ms"] / gpu["align_ms"], "speedup_total": cpu["total_ms"] / gpu["total_ms"],
                     "speedup_total_device_resident": cpu["total_ms"] / gpu_dev["total_ms"],
                     "gpu_vs_cpu_pose": {"dt_m": dt, "dr_rad": dr}, "error_vs_truth": {"dt_m": et, "dr_rad": er}}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ C3
SELECTION = "hull"   # "hull": OdomNode::getSubmapKeyframes (kNN + convex hull + concave hull, N3); "knn": nearest keyframes only


class Replay:
    """OdomNode's per-scan sequence (reference src/dlo/odom.cc:629-697): S2S, submap selection (getSubmapKeyframes,
    :1240-1293, through ngicp_submap_select), S2M, updateKeyframes (:1097-1181; shipped thresholds threshD 5 m,
    threshR 45 deg, adaptive parameters off).  `make()` builds a registration object."""

    def __init__(self, make, voxel, get_T, thresh_d=5.0, knn=10, thresh_r=45.0):
        # the C++ implementation behind the C ABI (csrc/submap_select.cpp); NGICP_SUBMAP_SELECT=qhull takes the
        # scipy/qhull checker instead
        from direct_lidar_odometry_b200 import submap_select as _ss
        SubmapSelector = _ss.SubmapSelector if os.environ.get("NGICP_SUBMAP_SELECT") == "qhull" else _ss.NativeSubmapSelector
        self.s2s, self.s2m = make(S2S), make(S2M)
        self.voxel, self.get_T = voxel, get_T
        self.thresh_d, self.thresh_r, self.knn = thresh_d, thresh_r, knn
        self.selector = SubmapSelector(knn, knn, knn, alpha=thresh_d) if SELECTION == "hull" else None
        self.keyframes = []   # (position, cloud, covs, rotation)
        self.prev_set = None
        self.T = None

    def first(self, scan, T0):
        self.T = T0.astype(np.float32)
        self.T_prev = self.T.copy()
        self.s2s.setInputTarget(scan); self.s2s.calculateTargetCovariances()
        self._add_keyframe(scan)

    def _add_keyframe(self, scan):
        kf = self.voxel(synth.transform_xyzi(scan, self.T), 0.5)
        self.s2s.setInputSource(kf); self.s2s.calculateSourceCovariances()
        self.keyframes.append((self.T[:3, 3].copy(), kf, self.s2s.getSourceCovariances(), self.T[:3, :3].copy()))

    def _new_keyframe_wanted(self):
        """updateKeyframes' decision (odom.cc:1102-1153): farther than threshD from the closest keyframe, or within it but
        rotated by more than threshR with at most one keyframe within 1.5 threshD."""
        p = self.T[:3, 3].astype(np.float32)
        d = np.array([np.float32(np.sqrt(((p - kf[0]).astype(np.float64) ** 2).sum())) for kf in self.keyframes], dtype=np.float32)
        closest = int(np.argmin(d))
        num_nearby = int((d <= np.float32(self.thresh_d * 1.5)).sum())
        dR = self.T[:3, :3].astype(np.float64) @ self.keyframes[closest][3].astype(np.float64).T
        theta = np.degrees(np.arccos(np.clip((np.trace(dR) - 1.0) / 2.0, -1.0, 1.0)))
        dd = d[closest]
        new = dd > self.thresh_d or theta > self.thresh_r
        if dd <= self.thresh_d:
            new = theta > self.thresh_r and num_nearby <= 1
        return bool(new)

    def _set_submap(self, sel):
        self.submap = np.ascontiguousarray(np.vstack([self.keyframes[i][1] for i in sel]))
        self.submap_covs = np.concatenate([self.keyframes[i][2] for i in sel])
        self.s2m.setInputTarget(self.submap); self.s2m.setTargetCovariances(self.submap_covs)
        return self.submap.shape[0]

    def step(self, scan, force_T=None):
        """force_T: adopt this pose after the S2M align (the align's own answer stays in self.T_result) — used to keep
        the GPU replay on the CPU replay's trajectory so that every align is compared on the same inputs."""
        self.events = []
        t_ = time.perf_counter()
        self.s2s.setInputSource(scan)
        self.s2m.registerInputSource(scan)
        self.s2m.source_kdtree_ = self.s2s.source_kdtree_
        self.s2m.source_covs_.clear()
        ta = time.perf_counter()
        self.s2s.align()                      # includes the lazily computed source covariances, as in the reference
        self.align_ms = [(time.perf_counter() - ta) * 1e3, 0.0]
        it_s2s = self.s2s.nr_iterations_
        T_s2s = self.T_prev @ self.s2s.getFinalTransformation()
        self.s2m.source_covs_ = self.s2s.source_covs_
        self.s2s.swapSourceAndTarget()
        if self.selector is not None:
            sel = tuple(self.selector.select([kf[0] for kf in self.keyframes], T_s2s[:3, 3])[0])
        else:
            d = [np.linalg.norm(T_s2s[:3, 3] - kf[0]) for kf in self.keyframes]
            sel = tuple(sorted(np.argsort(d)[: self.knn].tolist()))
        self.events.append(("s2s", (time.perf_counter() - t_) * 1e3)); t_ = time.perf_counter()
        if sel != self.prev_set:
            npts = self._set_submap(sel)
            self.prev_set = sel
            self.events.append(("submap_rebuild_%d" % npts, (time.perf_counter() - t_) * 1e3)); t_ = time.perf_counter()
        ta = time.perf_counter()
        self.s2m.align(T_s2s)
        self.align_ms[1] = (time.perf_counter() - ta) * 1e3
        self.T = self.s2m.getFinalTransformation()
        self.T_result = self.T
        if force_T is not None:
            self.T = np.array(force_T, dtype=np.float32)
        self.T_prev = self.T
        self.events.append(("s2m", (time.perf_counter() - t_) * 1e3)); t_ = time.perf_counter()
        if self._new_keyframe_wanted():
            self._add_keyframe(scan)
            self.events.append(("new_keyframe", (time.perf_counter() - t_) * 1e3))
        return it_s2s, self.s2m.nr_iterations_


class DeviceReplay(Replay):
    """The same sequence with the additive device-resident pieces (SURVEY §8f N1/N2): keyframe clouds are made by the
    fused transform + voxel pass and stay on the GPU, keyframes and their covariances live in a KeyframeStore, and a
    changed submap is assembled device-to-device — no 160 B/point round trip over PCIe."""

    def __init__(self, make, pre, thresh_d=5.0, knn=10):
        import torch
        from direct_lidar_odometry_b200 import KeyframeStore
        super().__init__(make, None, None, thresh_d, knn)
        self.pre = pre
        self.store = KeyframeStore(0)
        self.kf_buf = torch.empty((1 << 17, 8), dtype=torch.float32, device="cuda")

    def _add_keyframe(self, scan):
        kf = self.pre.transform_voxel_filter(scan, self.T, 0.5, out=self.kf_buf)
        self.s2s.setInputSource(kf); self.s2s.calculateSourceCovariances()
        self.store.push(self.s2s)
        self.keyframes.append((self.T[:3, 3].copy(), None, None, self.T[:3, :3].copy()))

    def _set_submap(self, sel):
        self.store.set_target(self.s2m, list(sel))
        return sum(self.store.points(i) for i in sel)


class OracleGicp:
    """Adapter giving the CPU oracle the method names Replay uses."""

    def __init__(self, O, cfg, threads):
        self.O, self.g = O, O.Gicp(k=cfg["k"], max_corr_dist=cfg["thr"], max_iter=cfg["max_iter"], trans_eps=cfg["trans_eps"], num_threads=threads)
        self.nr_iterations_ = 0
        self._src = self._tgt = None

    def setInputTarget(self, c): self._tgt = self.O.Cloud(c); self.g.set_target(self._tgt)
    def setInputSource(self, c): self._src = self.O.Cloud(c); self.g.set_source(self._src)
    def registerInputSource(self, c): self._src = self.O.Cloud(c, build_index=False); self.g.set_source(self._src)
    def calculateTargetCovariances(self): self.g.calc_target_covs()
    def calculateSourceCovariances(self): self.g.calc_source_covs()
    def getSourceCovariances(self): return self.g.get_source_covs()
    def setTargetCovariances(self, c): self.g.set_target_covs(c)
    def swapSourceAndTarget(self): self.g.swap(); self._src, self._tgt = self._tgt, self._src

    class _Covs:
        def __init__(self, outer): self.o = outer
        def clear(self): self.o.g.set_source_covs(np.zeros((0, 4, 4)))

    @property
    def source_covs_(self): return OracleGicp._Covs(self)
    @source_covs_.setter
    def source_covs_(self, v): self.g.set_source_covs(v.o.g.get_source_covs() if isinstance(v, OracleGicp._Covs) else v)
    @property
    def source_kdtree_(self): return None
    @source_kdtree_.setter
    def source_kdtree_(self, v): pass

    def align(self, guess=None):
        self._r = self.g.align(guess)
        self.nr_iterations_ = self._r.nr_iterations
    def getFinalTransformation(self): return self._r.T()


def run_c3(args):
    from direct_lidar_odometry_b200 import NanoGICP
    from oracle import oracle as O
    idx = list(range(args.scans))
    t0 = time.time()
    scans = gen_scans(idx)
    gen_s = time.time() - t0
    vox = NanoGICP(0)

    def make_gpu(cfg):
        g = NanoGICP(0)
        configure(g, cfg)
        return g
    import torch
    if args.device_store:
        rp = DeviceReplay(make_gpu, vox)
        scan_buf = [torch.empty((1 << 17, 8), dtype=torch.float32, device="cuda") for _ in range(2)]
    else:
        rp = Replay(make_gpu, lambda p, l: vox.voxel_filter(p, l), None)
    ms, iters, errs, traj = [], [], [], []
    phase = {}
    raw_in = {}
    if args.pinned:      # raw scans in page-locked host memory (what a driver node that owns its message buffers can do)
        for i in idx:
            raw_in[i] = torch.from_numpy(scans[i][1]).pin_memory()
    # --pipeline 1: the NEXT scan's upload + preprocess (its own handle and stream) runs on a host thread beside the
    # registration of the current one — same arithmetic, same poses; a scan then costs max(preprocess, registration)
    # instead of their sum.  (An odometry node would do this with a two-deep message queue; latency per scan is unchanged.)
    pipe = bool(getattr(args, "pipeline", 0)) and args.device_store
    ex = ThreadPoolExecutor(1) if pipe else None
    nxt = None
    vox_pre = NanoGICP(0) if pipe else vox      # a handle is single-threaded: the prefetch thread gets its own
    if pipe:
        scan_buf.append(torch.empty((1 << 17, 8), dtype=torch.float32, device="cuda"))   # three buffers: i-1 (S2S target), i, i+1

    def pre(j):
        t = time.perf_counter()
        r = raw_in.get(j, scans[j][1])
        s = vox_pre.preprocess(r, 1.0, 0.25, out=scan_buf[j % len(scan_buf)])
        return s, (time.perf_counter() - t) * 1e3
    for i in idx:
        T_true, raw = scans[i]
        raw = raw_in.get(i, raw)
        t1 = time.perf_counter()
        if pipe:
            scan, t_pre = nxt.result() if nxt is not None else pre(i)
            nxt = ex.submit(pre, i + 1) if i + 1 < len(idx) else None
        elif args.device_store:                   # preprocessPoints fused, output stays on the device
            scan = vox.preprocess(raw, 1.0, 0.25, out=scan_buf[i & 1])
        else:
            scan = vox.voxel_filter(raw, 0.25)    # preprocessPoints: vf_scan (crop box applied by the generator)
        if not pipe:
            t_pre = (time.perf_counter() - t1) * 1e3
        if i == 0:
            rp.first(scan, T_true)
            continue
        its = rp.step(scan)
        ms.append((time.perf_counter() - t1) * 1e3)
        for name, v in [("preprocess", t_pre), ("align_s2s_call", rp.align_ms[0]), ("align_s2m_call", rp.align_ms[1])] + \
                [(n.split("_")[0] if n.startswith("submap") else n, v) for n, v in rp.events]:
            phase.setdefault(name, []).append(v)
        if ms[-1] > 5.0:
            print(f"slow scan {i}: {ms[-1]:.1f} ms voxel+{[(n, round(v, 2)) for n, v in rp.events]} "
                  f"s2s kernels {({k: round(v, 3) for k, v in rp.s2s.timings().items()})} grid {rp.s2s.grid_info(1)}", file=sys.stderr)
        iters.append(its)
        errs.append(pose_err(rp.T, T_true))
        traj.append(np.array(rp.T, dtype=np.float32).copy())
    ms = np.array(ms)
    sel_txt = (f"submap = {rp.knn} nearest + {rp.knn} convex-hull + {rp.knn} concave-hull keyframes as OdomNode::getSubmapKeyframes" if SELECTION == "hull"
               else f"knn-{rp.knn} submap")
    out = {"config": f"C3: odometry replay, {args.scans} synthetic OS1-64 scans (S2S + S2M + keyframes by OdomNode::updateKeyframes' rule, threshD 5 m / threshR 45 deg; {sel_txt})"
                     + (", device-resident keyframes + fused preprocess (N1/N2)" if args.device_store else ", host keyframes as in OdomNode")
                     + (", raw scans in pinned host memory" if args.pinned else ", raw scans in pageable host memory")
                     + (", next scan's preprocess pipelined beside the registration" if pipe else ""),
           "gpu": {"ms_per_scan_mean": float(ms.mean()), "ms_per_scan_p50": float(np.percentile(ms, 50)), "ms_per_scan_p99": float(np.percentile(ms, 99)),
                   "keyframes": len(rp.keyframes), "final_translation_error_m": errs[-1][0], "max_translation_error_m": float(max(e[0] for e in errs)),
                   "max_rotation_error_rad": float(max(e[1] for e in errs)), "mean_iterations_s2s": float(np.mean([i[0] for i in iters])),
                   "mean_iterations_s2m": float(np.mean([i[1] for i in iters]))},
           "scan_generation_s": gen_s}
    # host wall time per phase, summed over the run and divided by the number of scans (rebuilds / keyframes are rare)
    out["gpu"]["phase_ms_per_scan"] = {k: float(np.sum(v) / len(ms)) for k, v in phase.items()}
    out["gpu"]["phase_counts"] = {k: len(v) for k, v in phase.items()}
    if args.device_store:
        # the additive path must reproduce the OdomNode-style host path bit for bit
        rh = Replay(make_gpu, lambda p, l: vox.voxel_filter(p, l), None)
        same = 0
        for i in idx:
            T_true, raw = scans[i]
            scan = vox.voxel_filter(raw, 0.25)
            if i == 0:
                rh.first(scan, T_true)
                continue
            rh.step(scan)
            same += int(np.array_equal(np.array(rh.T, dtype=np.float32), traj[i - 1]))
        out["gpu"]["poses_bit_identical_to_host_keyframe_path"] = f"{same}/{len(traj)}"
    # CPU oracle over the first --cpu-scans scans with the same sequence: timing + iteration-count / pose parity
    n_cpu = min(args.cpu_scans, args.scans)
    if n_cpu > 1:
        threads = os.cpu_count()
        rc = Replay(lambda cfg: OracleGicp(O, cfg, threads), lambda p, l: O.voxel_filter(p, l), None)
        cms, same_iters, dpose, mism, cal = [], 0, [], [], []
        rg = Replay(make_gpu, lambda p, l: vox.voxel_filter(p, l), None)
        for i in range(n_cpu):
            T_true, raw = scans[i]
            t1 = time.perf_counter()
            scan = O.voxel_filter(raw, 0.25)
            if i == 0:
                rc.first(scan, T_true); rg.first(vox.voxel_filter(raw, 0.25), T_true)
                continue
            ic = rc.step(scan)
            cms.append((time.perf_counter() - t1) * 1e3)
            cal.append(list(rc.align_ms))
            # teacher forcing: the GPU replay continues from the CPU replay's pose, so both see the same scan, the same
            # guess and keyframes placed by the same poses at every step (chained replays drift apart by rounding and
            # are then no longer "identical inputs")
            ig = rg.step(vox.voxel_filter(raw, 0.25), force_T=rc.T)
            same_iters += int(tuple(ic) == tuple(ig))
            if tuple(ic) != tuple(ig):
                mism.append({"scan": i, "cpu": [int(v) for v in ic], "gpu": [int(v) for v in ig], "dt_m": pose_err(rc.T, rg.T_result)[0]})
            dpose.append(pose_err(rc.T, rg.T_result))
        out["cpu"] = {"scans": n_cpu, "threads": threads, "ms_per_scan_mean": float(np.mean(cms)),
                      "align_s2s_call_ms": float(np.mean([c[0] for c in cal])), "align_s2m_call_ms": float(np.mean([c[1] for c in cal])),
                      "identical_iteration_counts": f"{same_iters}/{n_cpu - 1}", "iteration_mismatches": mism[:20],
                      "comparison": "per scan on identical inputs (GPU replay teacher-forced onto the CPU trajectory)", "max_gpu_vs_cpu_dt_m": float(max(d[0] for d in dpose)),
                      "max_gpu_vs_cpu_dr_rad": float(max(d[1] for d in dpose))}
        out["speedup_ms_per_scan"] = out["cpu"]["ms_per_scan_mean"] / float(ms[: n_cpu - 1].mean())
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ C4
def c4_pair_indices(n_pairs, rank, world):
    """Pair i registers scan i+1 against scan i of the 10 001-pose trajectory (SURVEY section 8d); ranks take contiguous
    blocks of pairs (direct_lidar_odometry_b200.sharded.partition_pairs)."""
    from direct_lidar_odometry_b200 import sharded
    return list(sharded.partition_pairs(n_pairs, rank, world))


def c4_make_scans(vox, first, count, device, batch=16):
    """Voxelised (0.25 m) scans first .. first+count-1 as device tensors, generated on the GPU by the torch ray-caster
    (synth.os1_like_batch_torch: same scene, same per-scan RNG streams as the numpy generator)."""
    import torch
    out = []
    buf = torch.empty((1 << 17, 8), dtype=torch.float32, device=device)
    for b0 in range(first, first + count, batch):
        idx = list(range(b0, min(b0 + batch, first + count)))
        raws = synth.os1_like_batch_torch(idx, [synth.trajectory_pose(i) for i in idx], device)
        for raw in raws:
            v = vox.voxel_filter(raw, 0.25, out=buf)
            out.append(v.clone())
    return out


C4_SPLIT = [0.0, 0.0]   # seconds the main thread waited for wave preparation / spent in ngicp_align_batch


def c4_run(handle_sets, scans, pair_offsets, wave, threads=8):
    """Register pairs (scans[o+1] -> scans[o]) for o in pair_offsets in waves of `wave` pairs.  A wave's clouds are
    indexed and their covariances computed from `threads` host threads, each pair on its own handle / stream; the wave's
    LM loops then run as ONE ngicp_align_batch launch.  Two sets of handles alternate, so the host threads prepare wave
    w+1 while wave w's batch kernel runs.  Returns per pair (nr_iterations, n_compute_error, final_x)."""
    from direct_lidar_odometry_b200 import align_batch
    results = []

    def prep(args):
        h, o = args
        h.clearSource(); h.clearTarget()
        h.setInputTarget(scans[o]); h.calculateTargetCovariances()
        h.setInputSource(scans[o + 1]); h.calculateSourceCovariances()
    waves = [pair_offsets[w0:w0 + wave] for w0 in range(0, len(pair_offsets), wave)]
    with ThreadPoolExecutor(threads) as ex:
        def submit(w):
            hs = handle_sets[w & 1][:len(waves[w])]
            return hs, [ex.submit(prep, a) for a in zip(hs, waves[w])]
        nxt = submit(0) if waves else None
        for w in range(len(waves)):
            hs, futs = nxt
            t0 = time.perf_counter()
            for f in futs:
                f.result()
            t1 = time.perf_counter()
            nxt = submit(w + 1) if w + 1 < len(waves) else None
            align_batch(hs)
            t2 = time.perf_counter()
            C4_SPLIT[0] += t1 - t0; C4_SPLIT[1] += t2 - t1
            for h in hs:
                results.append((int(h.result.nr_iterations), int(h.result.n_compute_error), np.array(h.result.final_x)))
    return results


def c4_bench(local, rank, world, pairs=10000, wave=64, threads=8, sample_check=0):
    """C4 on this rank's GPU (torch.distributed already initialised when world > 1).  Returns the result dict on rank 0,
    None elsewhere.  Timing: barrier, wall clock around this rank's waves (each wave ends with the host reading the
    results of its ngicp_align_batch launch), max over ranks."""
    import torch
    import torch.distributed as dist
    from direct_lidar_odometry_b200 import NanoGICP
    dev = torch.device("cuda", local)
    mine = c4_pair_indices(pairs, rank, world)
    vox = NanoGICP(local)
    t0 = time.perf_counter()
    scans = c4_make_scans(vox, mine[0], len(mine) + 1, dev)          # this rank's pairs are contiguous: n+1 scans
    gen_s = time.perf_counter() - t0
    from direct_lidar_odometry_b200 import _lib
    handles = [[NanoGICP(local) for _ in range(wave)] for _ in range(2)]
    for hs in handles:
        for h in hs:
            configure(h, S2S)
            # Many handles share the GPU here, so what counts is launches per pair and how well the streams interleave, not
            # the latency of one call.  Measured on one B200 (2000 pairs, 8 host threads, pairs/s): multi-kernel index +
            # warp kNN 7436, fused index + warp kNN 6304, multi-kernel index + tile kNN 5462, fused + tile 2855 — a
            # cooperative launch (the fused index) has to wait until all its blocks fit at once and holds up the other
            # streams meanwhile, and the tile path needs ten small launches per cloud.  NGICP_C4_KNN / NGICP_C4_INDEX: A/B.
            h.setKnnPath(_lib.KNN_TILE if os.environ.get("NGICP_C4_KNN") == "tile" else _lib.KNN_WARP)
            h.setIndexPath({"fused": 0, "multi": 1, "cluster": 3}[os.environ.get("NGICP_C4_INDEX", "cluster")])
    offs = list(range(len(mine)))
    c4_run(handles, scans, offs[:2 * wave], wave, threads)      # warm-up (both handle sets)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    C4_SPLIT[0] = C4_SPLIT[1] = 0.0
    t0 = time.perf_counter()
    res = c4_run(handles, scans, offs, wave, threads)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    t = torch.tensor([el], dtype=torch.float64, device=dev)
    cnt = torch.tensor([len(res)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(cnt)
    out = None
    if rank == 0:
        out = {"config": f"C4: {pairs} DISTINCT independent S2S scan pairs (pair i = scans i+1 -> i of the 10 001-pose trajectory, "
                         f"~{int(np.mean([s.shape[0] for s in scans[:64]]))} pts each; index + k=10 covariances for both clouds + align per pair), "
                         f"partitioned over {world} GPU(s); waves of {wave} pairs, one ngicp_align_batch launch per wave",
               "n_gpus": world, "pairs": int(cnt.item()), "wave": wave, "host_threads_per_gpu": threads, "seconds": float(t.item()),
               "pairs_per_s": float(cnt.item() / t.item()), "ms_per_pair_per_gpu": float(t.item() * 1e3 * world / cnt.item()),
               "mean_iterations": float(np.mean([r[0] for r in res])), "scan_generation_s_rank0": gen_s,
               "main_thread_split_s": {"waiting_for_index_and_covariances": C4_SPLIT[0], "in_align_batch": C4_SPLIT[1]}}
        if sample_check > 0:
            # a seeded sample of this rank's pairs against the CPU oracle (identical inputs: the device scans copied back)
            from oracle import oracle as O
            rng = np.random.default_rng(2026)
            pick = np.sort(rng.choice(len(offs), size=min(sample_check, len(offs)), replace=False))
            same, worst = 0, (0.0, 0.0)
            for o in pick.tolist():
                a, b = scans[o].cpu().numpy(), scans[o + 1].cpu().numpy()
                og = O.Gicp(k=S2S["k"], max_corr_dist=S2S["thr"], max_iter=S2S["max_iter"], trans_eps=S2S["trans_eps"], num_threads=os.cpu_count())
                og.set_target(O.Cloud(a)); og.set_source(O.Cloud(b))
                r = og.align()
                it, ne, fx = res[o]
                dt, dr = pose_err(fx.reshape(4, 4).T, r.Tx())
                same += int((it, ne) == (int(r.nr_iterations), int(r.n_compute_error)))
                worst = (max(worst[0], dt), max(worst[1], dr))
            out["oracle_sample"] = {"pairs_checked": int(len(pick)), "identical_counts": same, "max_dt_m": worst[0], "max_dr_rad": worst[1]}
    del handles, scans
    return out


def run_c4(args):
    import torch
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out = c4_bench(local, rank, world, args.pairs, args.wave, args.handles, args.check_pairs)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ C5
def _gen_dense(i):
    T = synth.trajectory_pose(i)
    s = synth.crop_box_negative(synth.os1_like(i, T, beams=128, cols=2048))
    return i, T, s


def c5_workload(n_target, log):
    # outside the checkout, which may be read-only; per user, so nobody else's file is read
    cache = os.path.join(tempfile.gettempdir(), f"ngicp_bench_cache_{os.getuid()}", f"c5_v2_{n_target}.npz")
    if os.path.exists(cache):
        z = np.load(cache)
        return {k: z[k] for k in z.files}
    t0 = time.time()
    stride = 33                                            # keyframes 5 m apart
    n_key = max(2, int(np.ceil(n_target / 200_000.0)) + 1)
    src_i = (n_key // 2) * stride + 10                     # the scan sits in the middle of its submap, as in DLO
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        out = list(ex.map(_gen_dense, [j * stride for j in range(n_key)] + [src_i]))
    keys = [synth.transform_xyzi(s, T.astype(np.float32)) for _, T, s in out[:-1]]
    target = np.ascontiguousarray(np.vstack(keys)[:n_target])
    _, Ts, src = out[-1]
    wl = dict(target=target, source=np.ascontiguousarray(src), truth=Ts,
              guess=synth.perturb_pose(Ts, (0.2, 0.0, 0.0), 1.0).astype(np.float32))
    log(f"C5 workload: {n_key} dense keyframes -> {target.shape[0]} target pts, source {src.shape[0]} pts, {time.time() - t0:.1f}s")
    try:
        os.makedirs(os.path.dirname(cache), exist_ok=True)
        tmp = cache + f".{os.getpid()}.npz"
        np.savez(tmp, **wl)
        os.replace(tmp, cache)
    except OSError:
        pass
    return wl


def _sha1(a):
    import hashlib
    return hashlib.sha1(np.ascontiguousarray(a).view(np.uint8)).hexdigest()


def c5_bench(local, rank, world, target_points=5_000_000, steps=10, cov_halo=2.0, balance=0.0, shard_source_covs=0, check=1):
    """C5 on `world` GPUs (torch.distributed already initialised when world > 1): every rank holds one slab (+ halo) of the
    target, the scan's index + covariances and the fused LM kernel with the in-kernel NVLink exchange run per step.
    Returns the result dict on rank 0.  Compared with the CPU oracle through tests/golden/c5_oracle_<n>.json."""
    import torch
    import torch.distributed as dist
    from direct_lidar_odometry_b200 import NanoGICP, sharded
    dev = torch.device("cuda", local)
    log = (lambda *a: print(*a, file=sys.stderr)) if rank == 0 else (lambda *a: None)
    if rank == 0:
        wl = c5_workload(target_points, log)
    if world > 1:
        dist.barrier()
    if rank != 0:
        wl = c5_workload(target_points, log)
    target, source, guess, truth = wl["target"], wl["source"], wl["guess"], wl["truth"]
    be = sharded.CudaShardBackend(local, k=S2M["k"], max_corr_dist=S2M["thr"])
    be.set_align_params(S2M["max_iter"], S2M["trans_eps"])
    g = be.g
    stream = torch.cuda.ExternalStream(g._L.ngicp_get_stream(g._h), device=dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- target: this rank's slab, index + k=20 covariances on this GPU, halo grown until exact ----
    sync_all()
    t0 = time.perf_counter()
    expected = synth.transform_xyzi(source, np.asarray(guess, dtype=np.float64))[:, :3] if balance > 0 else None
    info = be.build_target_shard(target, rank, world, halo=S2M["thr"] + 0.01, k=S2M["k"], cov_halo=cov_halo,
                                 queries=expected, query_weight=balance)
    sync_all()
    t_build = time.perf_counter() - t0
    tm = g.timings()
    build_gpu_ms = tm["set_target_ms"] + tm["target_covs_ms"]          # last round of the halo loop
    if world > 1:
        be.connect_fused(rank, world)
    src_d = torch.from_numpy(source).to(dev)

    def step():
        if shard_source_covs and world > 1:
            be.set_source_sharded(src_d, rank, world)   # index replicated, k=20 covariances split over the ranks + all-reduce
        else:
            be.set_source(src_d)         # index + k=20 covariances of the dense scan (replicated on every rank)
        return be.align_fused(guess)     # persistent LM kernel, exchange in peer memory

    for _ in range(3):
        res = step()
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    al = []
    for a, b in ev:
        sync_all()
        a.record(stream)
        res = step()
        b.record(stream)
        b.synchronize()
        al.append(g.timings()["align_ms"])
    ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / steps, float(np.mean(al)), build_gpu_ms],
                      dtype=torch.float64, device=dev)
    npts = torch.tensor([info["shard_points"]], dtype=torch.int64, device=dev)
    fx = torch.from_numpy(res["final_x"]).to(dev)
    fx_all = [torch.zeros_like(fx) for _ in range(world)]
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_gather(fx_all, fx)
        shard_pts = [torch.zeros_like(npts) for _ in range(world)]
        dist.all_gather(shard_pts, npts)
    else:
        fx_all, shard_pts = [fx], [npts]
    identical = all(bool(torch.equal(fx_all[0], f)) for f in fx_all)
    line = None
    if rank == 0:
        dt, dr = pose_err(res["final_x"], truth)
        line = {"config": f"C5: dense 128-beam scan ({source.shape[0]} pts, no voxel filter) vs {target.shape[0]}-pt submap sharded over "
                          f"{world} GPU(s): slabs + halo, k=20 covariances per slab, fused LM with the H/b/err exchange in NVLink peer memory",
                "n_gpus": world, "steps": steps, "ms_per_scan": float(ms[0].item()), "align_ms": float(ms[1].item()),
                "target_build_gpu_ms": float(ms[2].item()), "target_build_wall_s": t_build, "cov_halo_m": info["cov_halo"],
                "halo_rounds": info["rounds"], "shard_points": [int(x.item()) for x in shard_pts], "slab_query_weight": balance,
                "source_covs": "split over the ranks + NCCL all-reduce" if (shard_source_covs and world > 1) else "replicated on every rank",
                "iterations": res["nr_iterations"], "n_linearize": res["n_linearize"], "n_compute_error": res["n_compute_error"],
                "converged": res["converged"], "ranks_bit_identical": identical, "pose_error_m": dt, "pose_error_rad": dr,
                "rank0_kernel_ms": {k: round(v, 4) for k, v in g.timings().items()}}
        gold_path = os.path.join(ROOT, "tests", "golden", f"c5_oracle_{target.shape[0]}.json")
        if os.path.exists(gold_path):
            gold = json.load(open(gold_path))
            gdt, gdr = pose_err(res["final_x"], np.array(gold["final_x"]).reshape(4, 4))
            line["vs_oracle"] = {"fixture": os.path.relpath(gold_path, ROOT),
                                 "inputs_identical_to_fixture": bool(_sha1(target) == gold["target_sha1"] and _sha1(source) == gold["source_sha1"]),
                                 "dT_vs_oracle_m": gdt, "dR_vs_oracle_rad": gdr,
                                 "counts_equal": bool((res["nr_iterations"], res["n_linearize"], res["n_compute_error"]) ==
                                                      (gold["nr_iterations"], gold["n_linearize"], gold["n_compute_error"])),
                                 "oracle_counts": [gold["nr_iterations"], gold["n_linearize"], gold["n_compute_error"]]}
        if check and world > 1:
            # the same registration unsharded on this GPU: iteration counts and pose must agree
            u = NanoGICP(local)
            configure(u, S2M)
            u.setInputTarget(target); u.calculateTargetCovariances()
            u.setInputSource(src_d); u.calculateSourceCovariances()
            u.align(guess)
            line["unsharded_align_ms"] = u.timings()["align_ms"]
            line["unsharded_iterations"] = int(u.result.nr_iterations)
            line["max_abs_dT_vs_unsharded"] = float(np.abs(u.final_state() - res["final_x"]).max())
            del u
    if world > 1:
        dist.barrier()
        be.g.comm_close()
    return line


def run_c5(args):
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    line = c5_bench(local, rank, world, args.target_points, args.steps, args.cov_halo, args.balance, args.shard_source_covs, args.check)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("which", choices=["c1", "c3", "c4", "c5"])
    ap.add_argument("--device-store", type=int, default=0, help="c3: device-resident keyframes + fused preprocess (N1/N2)")
    ap.add_argument("--target-points", type=int, default=5_000_000)
    ap.add_argument("--cov-halo", type=float, default=2.0)
    ap.add_argument("--shard-source-covs", type=int, default=0, help="c5: split the scan's covariances over the ranks (all-reduce) instead of replicating them")
    ap.add_argument("--balance", type=float, default=0.0, help="c5: weight of the scan's point distribution when placing the slab cuts (0 = equal target counts)")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--check", type=int, default=1)
    ap.add_argument("--scans", type=int, default=300)
    ap.add_argument("--selection", choices=["hull", "knn"], default="hull", help="c3: submap keyframe selection")
    ap.add_argument("--cpu-scans", type=int, default=40)
    ap.add_argument("--pinned", type=int, default=0, help="c3: keep the raw scans in pinned host memory")
    ap.add_argument("--pipeline", type=int, default=0, help="c3: preprocess scan i+1 on a host thread while scan i is registered")
    ap.add_argument("--pairs", type=int, default=10000)
    ap.add_argument("--wave", type=int, default=64, help="c4: pairs per ngicp_align_batch launch")
    ap.add_argument("--check-pairs", type=int, default=0, help="c4: oracle-check a seeded sample of this many of rank 0's pairs")
    ap.add_argument("--handles", type=int, default=8)
    a = ap.parse_args()
    SELECTION = a.selection
    {"c1": run_c1, "c3": run_c3, "c4": run_c4, "c5": run_c5}[a.which](a)
