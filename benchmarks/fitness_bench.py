#!/usr/bin/env python
"""getFitnessScore timings: the fused GPU call (ngicp_fitness_score), the batched call (ngicp_fitness_batch) and the
composition a caller could build before it existed — ngicp_transform_source (points to the host), ngicp_knn(k=1) (back
to the device and the distances back to the host), and PCL's filter and serial sum on the host.

  C2  bench.make_workload: the ~22k-point scan against the 500k-point submap at the pose align() found
  C4  one wave of 64 voxelised S2S pairs of benchmarks/configs.py's generator, after one align_batch

Every path ends in a host synchronisation, so a call's wall clock is its full cost to the caller; the CUDA events
bracket the same calls on the one stream all handles are switched to for the measurement.  Repeated calls read the
target from a warm L2 (the C2 submap's points are 8 MB).  A separate torch.profiler pass gives per-kernel device
time.  Every path must find the same inlier counts.

    python benchmarks/fitness_bench.py [--reps 100] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

DBL_MAX = sys.float_info.max


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    parts = [p.strip() for p in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return dict(zip(("name", "power_limit", "sm_max_clock"), parts)) if len(parts) == 3 else {"nvidia_smi": q.stderr.strip()}


def composed(g, n, max_range):
    """transform on the device -> host -> kNN(k=1) on the device -> host -> PCL's filter and serial sum."""
    import ctypes as C
    from direct_lidar_odometry_b200 import _lib
    q = np.empty((n, 4), dtype=np.float32)
    Tf = np.ascontiguousarray(g.getFinalTransformation().T).reshape(16)
    g._check(g._L.ngicp_transform_source(g._h, Tf.ctypes.data_as(C.POINTER(C.c_float)), q.ctypes.data, n))
    ok = np.isfinite(q[:, :3]).all(axis=1)
    _, d2 = g.knn(_lib.TARGET, q[ok], 1)
    d = d2[:, 0].astype(np.float64)
    d = d[d <= max_range]
    return (float(np.add.accumulate(d)[-1]) / d.size if d.size else DBL_MAX), int(d.size)


def timed(fn, reps, warm, stream):
    import torch
    for _ in range(warm):
        fn()
    wall, dev = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        e0.record(stream)
        t0 = time.perf_counter()
        fn()
        t1 = time.perf_counter()
        e1.record(stream)
        e1.synchronize()
        wall.append((t1 - t0) * 1e6)
        dev.append(e0.elapsed_time(e1) * 1e3)
    return {"wall_us_median": float(np.median(wall)), "wall_us_p10": float(np.percentile(wall, 10)),
            "wall_us_p90": float(np.percentile(wall, 90)), "events_us_median": float(np.median(dev)), "reps": reps}


def kernel_times(fn, calls):
    """device time per call of each kernel the calls launch (torch.profiler, a run of its own)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.count > 0:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            out[ev.key[:80]] = {"us_per_call": float(t) / calls, "launches_per_call": ev.count / calls}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--wave", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.reps >= 50
    import torch
    assert torch.cuda.is_available(), "fitness_bench measures the GPU: no CUDA device"
    import bench
    import configs
    from direct_lidar_odometry_b200 import NanoGICP, align_batch, fitness_batch
    stream = torch.cuda.Stream()
    res = {"gpu": card_info(), "torch_device": torch.cuda.get_device_name(0), "reps": args.reps, "warmup": args.warmup}

    # ---- C2
    vox = NanoGICP(0)
    wl = bench.make_workload(lambda p, leaf: vox.voxel_filter(p, leaf))
    g = NanoGICP(0)
    configs.configure(g, configs.S2M)
    g.setInputTarget(wl["submap"]); g.setInputSource(wl["scan_0"])
    g.align(wl["guesses"][0])
    g.set_stream(stream.cuda_stream)
    ns = wl["scan_0"].shape[0]
    c2 = {"n_source": ns, "n_target": int(wl["submap"].shape[0])}
    for r in (DBL_MAX, 0.25):
        key = "unbounded" if r == DBL_MAX else f"max_range_{r}"
        f_score, f_n = g.fitness(None, r)
        c_score, c_n = composed(g, ns, r)
        assert f_n == c_n, (f_n, c_n)
        c2[key] = {"inliers": f_n, "score": f_score, "score_composed": c_score,
                   "fused": timed(lambda: g.fitness(None, r), args.reps, args.warmup, stream),
                   "composed": timed(lambda: composed(g, ns, r), args.reps, args.warmup, stream)}
    c2["kernels_fused"] = kernel_times(lambda: g.fitness(), 20)
    c2["kernels_composed"] = kernel_times(lambda: composed(g, ns, DBL_MAX), 20)
    res["c2"] = c2

    # ---- C4 wave
    W = args.wave
    scans = configs.c4_make_scans(vox, 0, W + 1, torch.device("cuda", 0))
    hs = []
    for o in range(W):
        h = NanoGICP(0)
        configs.configure(h, configs.S2S)
        h.setInputTarget(scans[o]); h.setInputSource(scans[o + 1])
        hs.append(h)
    align_batch(hs)
    torch.cuda.synchronize()
    for h in hs:
        h.set_stream(stream.cuda_stream)
    sizes = [int(s.shape[0]) for s in scans[1:]]
    c4 = {"pairs": W, "mean_source_points": float(np.mean(sizes))}
    for r in (DBL_MAX, 0.25):
        key = "unbounded" if r == DBL_MAX else f"max_range_{r}"
        b_scores, b_n = fitness_batch(hs, max_range=r)
        singles = [h.fitness(None, r) for h in hs]
        comp = [composed(h, n, r) for h, n in zip(hs, sizes)]
        assert [s[1] for s in singles] == [int(x) for x in b_n] == [c[1] for c in comp]
        assert all(np.float64(s[0]).view(np.uint64) == b.view(np.uint64) for s, b in zip(singles, b_scores))
        c4[key] = {"inliers_total": int(np.sum(b_n)),
                   "batch": timed(lambda: fitness_batch(hs, max_range=r), args.reps, args.warmup, stream),
                   "fused_single_calls": timed(lambda: [h.fitness(None, r) for h in hs], args.reps, args.warmup, stream),
                   "composed": timed(lambda: [composed(h, n, r) for h, n in zip(hs, sizes)], args.reps, args.warmup, stream)}
    c4["kernels_batch"] = kernel_times(lambda: fitness_batch(hs), 20)
    res["c4_wave"] = c4
    for h in hs + [g]:
        h.set_stream(None)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
