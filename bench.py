#!/usr/bin/env python
"""bench.py — headline benchmark of the NanoGICP hot path (BASELINE.json configs[1], "C2"):

    one step = register a ~20k-point voxelised OS1-64-like scan against a 500 000-point keyframe submap:
               target index build + target covariances (k=20) + source index + source covariances +
               LM align (DLO's S2M parameters: k=20, max-corr 0.5 m, 32 iterations, eps 0.01)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`value`  : scan pairs per second, inputs already resident in HBM (device pointers into the C ABI)
`e2e`    : same through the public API with pinned HOST buffers (H2D of both clouds and D2H of the result inside the
           timed region)
`roofline`: dominant kernel group (exact kNN + covariance over the 500k submap) — algorithmic 64 B/point / its CUDA-event time
`cpu_baseline`: the CPU oracle (reference's vendored nanoflann + restated GICP math, OpenMP) on this host's cores
--impl reference: that CPU path alone, same workload/metric.
--dump-outputs DIR: after the timed steps, what the last one computed goes to DIR/<name>.npy (see dump_outputs), so that
two builds can be compared output for output on the same seeded inputs.
N>1: one process per GPU (torchrun), every rank registers its own scans against the submap (weak scaling), no collective
on the data path; barrier + max-over-ranks timing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from direct_lidar_odometry_b200 import synth  # noqa: E402

S2M = dict(k=20, thr=0.5, max_iter=32, trans_eps=0.01)     # reference cfg/params.yaml:63-67
SUBMAP_POINTS = 500_000
KEYFRAME_STRIDE = 33                                         # 5 m at 0.15 m per scan (threshD, cfg/params.yaml:40)
SRC_INDEX = 12 * KEYFRAME_STRIDE + 10
SRC_LEAF = 0.27
# generated inputs are cached outside the checkout, which may be read-only; per user, so nobody else's file is read
CACHE = os.environ.get("NGICP_BENCH_CACHE",
                       os.path.join(tempfile.gettempdir(), f"ngicp_bench_cache_{os.getuid()}", "c2_v2.npz"))
DUMP_TARGET_COV_ROWS = 1 << 16     # --dump-outputs: seeded sample of the 500k target covariances (8 MiB instead of 64)


def make_workload(voxel_filter, log=lambda *a: None):
    """Synthetic C2 inputs (SURVEY.md §8d): world-frame submap of exactly 500k points and scans to register."""
    if os.path.exists(CACHE):
        z = np.load(CACHE)
        return {k: z[k] for k in z.files}
    t0 = time.time()
    keys, total, j = [], 0, 0
    while total < SUBMAP_POINTS:
        i = j * KEYFRAME_STRIDE
        T = synth.trajectory_pose(i)
        s = synth.crop_box_negative(synth.os1_like(i, T, beams=128, cols=1024))
        w = synth.transform_xyzi(s, T.astype(np.float32))         # transformPointCloud, reference odom.cc:484
        v = voxel_filter(w, 0.5)                                    # vf_submap, odom.cc:487-490
        keys.append(v)
        total += v.shape[0]
        j += 1
    submap = np.ascontiguousarray(np.vstack(keys)[:SUBMAP_POINTS])
    scans, truths, guesses = [], [], []
    for r in range(8):                                              # one source scan per possible rank
        i = SRC_INDEX + 7 * r
        T = synth.trajectory_pose(i)
        s = synth.crop_box_negative(synth.os1_like(i, T))
        v = voxel_filter(s, SRC_LEAF)                               # vf_scan
        scans.append(v)
        truths.append(T)
        guesses.append(synth.perturb_pose(T, (0.2, 0.0, 0.0), 1.0).astype(np.float32))
    wl = dict(submap=submap, truths=np.stack(truths), guesses=np.stack(guesses), n_keyframes=np.int64(j))
    for r, sc in enumerate(scans):
        wl[f"scan_{r}"] = np.ascontiguousarray(sc)
    log(f"workload: {j} keyframes -> {submap.shape[0]} pts, scans {[s.shape[0] for s in scans]} pts, generated in {time.time() - t0:.1f}s")
    try:
        os.makedirs(os.path.dirname(CACHE), exist_ok=True)
        tmp = CACHE + f".{os.getpid()}.npz"
        np.savez(tmp, **wl)
        os.replace(tmp, CACHE)
    except OSError:
        pass
    return wl


# ----------------------------------------------------------------------------------------------- CPU (oracle) arm
def cpu_step(orc, submap, scan, guess, threads):
    """The same step on the CPU path: serial kd-tree builds + OpenMP covariances/align (reference structure)."""
    t = {}
    t0 = time.perf_counter()
    tgt = orc.Cloud(submap)
    t["target_index_ms"] = (time.perf_counter() - t0) * 1e3
    g = orc.Gicp(k=S2M["k"], max_corr_dist=S2M["thr"], max_iter=S2M["max_iter"], trans_eps=S2M["trans_eps"], num_threads=threads)
    g.set_target(tgt)
    t1 = time.perf_counter()
    g.calc_target_covs()
    t["target_covs_ms"] = (time.perf_counter() - t1) * 1e3
    t1 = time.perf_counter()
    src = orc.Cloud(scan)
    g.set_source(src)
    g.calc_source_covs()
    t["source_ms"] = (time.perf_counter() - t1) * 1e3
    t1 = time.perf_counter()
    r = g.align(guess)
    t["align_ms"] = (time.perf_counter() - t1) * 1e3
    t["total_ms"] = (time.perf_counter() - t0) * 1e3
    return r, t


def run_cpu(wl, steps, warmup, rank_scan=0):
    from oracle import oracle as orc
    L = orc.load(prefer_ref=True)
    threads = os.cpu_count() or L.orc_max_threads()   # all host cores (torchrun pins OMP_NUM_THREADS=1 in the environment)
    submap, scan, guess = wl["submap"], wl[f"scan_{rank_scan}"], wl["guesses"][rank_scan]
    for _ in range(warmup):
        cpu_step(orc, submap, scan, guess, threads)
    times, phases, r = [], [], None
    for _ in range(steps):
        r, t = cpu_step(orc, submap, scan, guess, threads)
        times.append(t["total_ms"])
        phases.append(t)
    ms = float(np.mean(times))
    ph = {k: float(np.mean([p[k] for p in phases])) for k in phases[0]}
    kind = "port"
    desc = ("oracle/_ref: reference's own nanoflann kd-tree + restated NanoGICP math" if L.orc_has_ref_nanoflann()
            else "oracle: restated kd-tree + restated NanoGICP math")
    return dict(ms=ms, phases=ph, threads=threads, kind=kind, desc=desc, result=r)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80,
                 "sw_power_cap": 0x4, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------------------------- GPU arm
def gpu_step(g, submap, scan, guess):
    g.clearTarget()                      # defeat the pointer-identity cache: every step rebuilds everything
    g.clearSource()
    g.setInputTarget(submap)             # K1: 500k-point grid index
    g.calculateTargetCovariances()       # K2+K3: kNN(20) + plane covariances over the submap
    g.setInputSource(scan)               # K1 on the scan
    g.calculateSourceCovariances()
    g.align(guess)                       # K4/K5 + LM, one persistent kernel; returns after the 496-byte result is on the host
    return g.result


def dump_outputs(out_dir, g):
    """What a caller of gpu_step receives from its last call, as .npy files: the registration result (float32 transform,
    float64 state / Hessian / LM values, counts as float64) and the covariances of both clouds, the target's as a fixed
    seeded sample of rows."""
    r = g.result
    tc = g.getTargetCovariances()
    rows = np.sort(np.random.default_rng(0).choice(tc.shape[0], min(DUMP_TARGET_COV_ROWS, tc.shape[0]), replace=False))
    arrays = {"final_transformation": g.getFinalTransformation(), "final_state": g.final_state(),
              "final_hessian": g.getFinalHessian(), "lm_lambda_last_error": np.array([r.lm_lambda, r.last_error]),
              "counts": np.array([r.nr_iterations, r.converged, r.n_linearize, r.n_compute_error, r.lm_failed], np.float64),
              "source_covariances": g.getSourceCovariances(),
              "target_covariances_sample": tc[rows], "target_covariances_sample_rows": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=3, help="bounded CPU-baseline sample (full C2 steps)")
    ap.add_argument("--cell", type=float, default=0.0)
    ap.add_argument("--table", type=int, default=0, help="grid table capacity in cells (0 = library default)")
    ap.add_argument("--extras", type=int, default=1, help="also run the partitioned configs C4 (10k distinct pairs) and C5 "
                    "(5M-point submap sharded over the ranks, fused NVLink exchange) and report them as sub-objects")
    ap.add_argument("--c4-pairs", type=int, default=10000)
    ap.add_argument("--c5-target", type=int, default=5_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what rank 0's last timed GPU step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    config = {"workload": "C2: S2M register 1 voxelised OS1-64-like scan vs 500k-pt keyframe submap "
                          "(target index + k=20 covariances + source index/covariances + LM align), synthetic",
              "submap_points": SUBMAP_POINTS, "k": S2M["k"], "max_corr_dist": S2M["thr"], "max_iter": S2M["max_iter"],
              "trans_eps": S2M["trans_eps"], "l2": "flushed between timed steps (256 MiB write)",
              "parallelism": f"{world} independent streams (one process per GPU, no data-path collective)"}

    # ------------------------------------------------------------------ reference arm: CPU only, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import oracle as orc
        wl = make_workload(lambda p, leaf: orc.voxel_filter(p, leaf), log=lambda *a: print(*a, file=sys.stderr))
        config["source_points"] = int(wl["scan_0"].shape[0])
        c = run_cpu(wl, args.steps, args.warmup)
        val = 1e3 / c["ms"]
        line = {"impl": "reference", "metric": "scan_pairs_per_s", "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": c["ms"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 kNN / f64 GICP", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": c["threads"], "kind": c["kind"],
                                 "sample": f"{args.steps} full C2 steps; {c['desc']}", "phases_ms": c["phases"]},
                "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "iterations": int(c["result"].nr_iterations)}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    from direct_lidar_odometry_b200 import NanoGICP, _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    g = NanoGICP(local_rank)
    g.setCorrespondenceRandomness(S2M["k"]); g.setMaxCorrespondenceDistance(S2M["thr"])
    if os.environ.get("NGICP_TILE_MIN"):       # experiments: cloud size from which the tile kNN path is taken
        g.setKnnPath(0, int(os.environ["NGICP_TILE_MIN"]))
    g.setMaximumIterations(S2M["max_iter"]); g.setTransformationEpsilon(S2M["trans_eps"])
    if args.cell > 0:
        g.setGridCellSize(args.cell)
    if args.table > 0:
        g.setGridTableCells(args.table)
    if local_rank == 0:
        wl = make_workload(lambda p, leaf: g.voxel_filter(p, leaf), log=lambda *a: print(*a, file=sys.stderr))
    if world > 1:
        dist.barrier()
    if local_rank != 0:
        wl = make_workload(lambda p, leaf: g.voxel_filter(p, leaf))
    scan_np, guess = wl[f"scan_{rank % 8}"], wl["guesses"][rank % 8]
    submap_np = wl["submap"]
    config["source_points"] = int(scan_np.shape[0])
    dev = torch.device("cuda", local_rank)
    submap_d = torch.from_numpy(submap_np).to(dev)
    scan_d = torch.from_numpy(scan_np).to(dev)
    submap_h = torch.from_numpy(submap_np).pin_memory()
    scan_h = torch.from_numpy(scan_np).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(g._L.ngicp_get_stream(g._h), device=dev)
    L = _lib.load()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(submap, scan, steps):
        """steps timed steps, each bracketed by CUDA events on the launching stream; L2 flushed in between."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        phases = []
        res = None
        for a, b in ev:
            flush.zero_()
            torch.cuda.synchronize()
            a.record(stream)
            res = gpu_step(g, submap, scan, guess)
            b.record(stream)
            b.synchronize()
            phases.append(g.timings())
        ms = [a.elapsed_time(b) for a, b in ev]
        return ms, phases, res

    for _ in range(warmup):
        gpu_step(g, submap_d, scan_d, guess)
    barrier()
    launches0 = L.ngicp_launch_count()
    with ClockSampler(local_rank) as clk:
        t_wall0 = time.perf_counter()
        ms_dev, phases, res = timed(submap_d, scan_d, args.steps)
        barrier()
        t_wall = time.perf_counter() - t_wall0
    launches = (L.ngicp_launch_count() - launches0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, g)      # before the end-to-end steps below overwrite the handle's results
    grids = {"target": g.grid_info(1), "source": g.grid_info(0)}
    # end to end: pinned host buffers in, result struct out, every step
    for _ in range(2):
        gpu_step(g, submap_h, scan_h, guess)
    barrier()
    ms_e2e, _, res_e2e = timed(submap_h, scan_h, args.steps)
    barrier()

    tot = torch.tensor([sum(ms_dev), sum(ms_e2e)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    tot_dev_ms, tot_e2e_ms = tot.tolist()
    value = world * args.steps / (tot_dev_ms * 1e-3)
    e2e_value = world * args.steps / (tot_e2e_ms * 1e-3)

    if rank == 0:
        ph = {k: float(np.mean([p[k] for p in phases])) for k in phases[0]}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        kcov_ms = ph["target_covs_ms"]
        alg_bytes = 64.0 * SUBMAP_POINTS                  # 16 B point read + 48 B covariance written, per point
        achieved = alg_bytes / (kcov_ms * 1e-3) / 1e9
        # DRAM traffic and warp-instruction count of the group come from the ncu capture committed under profiles/
        # (profiles/extract_knn_cov.py writes the JSON together with the SHA-1 of the kernel source it was measured on):
        # a capture of another kernel version is reported as stale instead of being passed off as current.
        traffic, issue_frac, ncu_note = None, None, "no ncu extraction under profiles/"
        try:
            import hashlib
            meta = json.load(open(os.path.join(ROOT, "profiles", "knn_cov_ncu_r2.json")))
            src_sha = hashlib.sha1(open(os.path.join(ROOT, "direct_lidar_odometry_b200", "csrc", "knn_cov.cu"), "rb").read()).hexdigest()
            if meta.get("knn_cov_cu_sha1") == src_sha:
                traffic = meta["dram_bytes_per_launch"]
                ncu_note = f"profiles/knn_cov_ncu_r2.json ({meta.get('report', '?')}), same kernel source"
                sm_mhz = clk.summary().get("sm_mhz") or 1965.0
                # issue-slot utilisation: warp instructions of the group / (SMs x 4 schedulers x cycles of the live-measured time)
                issue_frac = meta["warp_instructions_per_launch"] / (148 * 4 * sm_mhz * 1e6 * kcov_ms * 1e-3)
            else:
                ncu_note = "profiles/knn_cov_ncu_r2.json was measured on another version of knn_cov.cu: traffic withheld (stale)"
        except Exception:
            pass
        line = {"metric": "scan_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": tot_dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 kNN / f64 GICP", "data": "synthetic", "config": config,
                "phases_ms": ph, "iterations": int(res.nr_iterations), "n_linearize": int(res.n_linearize),
                "n_compute_error": int(res.n_compute_error), "converged": int(res.converged),
                "pose_error_m": float(np.linalg.norm(np.array(res.final_x).reshape(4, 4).T[:3, 3] - wl["truths"][rank % 8][:3, 3])),
                "wall_s_timed_region": t_wall,
                "roofline": {"kernel": "K2+K3 over the 500k-pt submap: knn_plan_kernel + knn_lists_tile_kernel + knn_lists_rest_kernel (exact kNN, k=20) + cov_from_lists_kernel (plane covariances)", "bound": "hbm",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                             "issue_frac": issue_frac, "ncu_source": ncu_note,
                             "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kcov_ms, "peak_source": peak_src,
                             "share_of_step": kcov_ms / (tot_dev_ms / args.steps),
                             "limiter": "instruction issue, not bandwidth (see issue_frac and profiles/): exact kNN is a select over ~170 staged "
                                        "candidates per query; the fraction of the HBM roofline is small by construction"},
                "e2e": {"value": e2e_value, "unit": "pairs/s", "ms_per_step": tot_e2e_ms / args.steps,
                        "h2d_bytes_per_step": int(submap_np.nbytes + scan_np.nbytes), "d2h_bytes_per_step": 496},
                "gpu_launches": int(launches), "grids": grids, "clocks": clk.summary()}
        if world == 1:
            c = run_cpu(wl, args.cpu_steps, 0)
            line["cpu_baseline"] = {"value": 1e3 / c["ms"], "unit": "pairs/s", "cores": c["threads"], "kind": c["kind"],
                                    "sample": f"{args.cpu_steps} full C2 steps on the host CPU; {c['desc']}",
                                    "ms_per_step": c["ms"], "phases_ms": c["phases"],
                                    "iterations": int(c["result"].nr_iterations)}
            # parity of THIS run: the GPU step's result against the CPU arm's on the same inputs (north-star tolerances)
            ro = c["result"]
            Tg, Tc = np.array(res.final_x).reshape(4, 4).T, ro.Tx()
            dR = Tg[:3, :3].T @ Tc[:3, :3]
            sk = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
            dt, dr = float(np.linalg.norm(Tg[:3, 3] - Tc[:3, 3])), float(np.arcsin(min(1.0, float(np.linalg.norm(sk)))))
            counts_g = [int(res.nr_iterations), int(res.n_linearize), int(res.n_compute_error), int(res.converged)]
            counts_c = [int(ro.nr_iterations), int(ro.n_linearize), int(ro.n_compute_error), int(ro.converged)]
            Te = np.array(res_e2e.final_x).reshape(4, 4).T
            line["parity"] = {"against": "cpu_baseline arm (oracle) on the same submap, scan and guess",
                              "pose_dt_m": dt, "pose_dr_rad": dr, "tolerance": {"dt_m": 1e-4, "dr_rad": 1e-5},
                              "counts_gpu": counts_g, "counts_cpu": counts_c, "counts_equal": counts_g == counts_c,
                              "e2e_result_bit_identical_to_device_resident": bool(np.array_equal(Te, Tg)),
                              "ok": bool(dt < 1e-4 and dr < 1e-5 and counts_g == counts_c)}
    # ------------------------------------------------------------------ the partitioned configs, same launch, same clock
    if args.extras:
        del submap_d, scan_d, submap_h, scan_h, flush
        g.clearSource(); g.clearTarget()
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
        import configs as bc
        c4 = c5 = None
        try:
            # host threads that enqueue the per-pair index + covariance work: what the box's cores allow per rank, at most 8
            # (8 ranks x 8 threads on 32 cores: 41.7k pairs/s; x 3 threads: 57.2k — the ranks were fighting for cores)
            c4_threads = max(2, min(8, (os.cpu_count() or 8) // world - 1))
            c4 = bc.c4_bench(local_rank, rank, world, pairs=args.c4_pairs, wave=64, threads=c4_threads, sample_check=24 if world == 1 else 0)
        except Exception as e:  # keep the headline line even if an extra fails
            c4 = {"error": repr(e)}
        barrier()
        try:
            # the scan's k=20 covariances are split over the ranks + one all-reduce when there is more than one
            # (2 GPUs: 3.72 -> 3.63 ms/scan; the replicated covariances are the largest non-align item at 8)
            c5 = bc.c5_bench(local_rank, rank, world, target_points=args.c5_target, steps=args.steps, check=1,
                             shard_source_covs=1 if world > 1 else 0)
        except Exception as e:
            c5 = {"error": repr(e)}
        barrier()
        if rank == 0:
            line["c4"] = c4
            line["c5"] = c5
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
