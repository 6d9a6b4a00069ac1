#!/usr/bin/env python
"""bench.py -- BA windows/s of the B200 window solver on BASELINE.json's headline configuration, plus one sub-record per
other BASELINE configuration.

Headline: one "step" = one complete trimmed bundle-adjustment solve (all LM iterations + trimming round, Ceres-equivalent
termination) of a BATCH of independent synthetic windows of config 2 (30 keyframes / 3000 landmarks / 40000 observations,
mono + lidar depth, FP64).  `value` is whole-job windows/s with the batch resident in HBM; `e2e` is the same metric
through the host-buffer C-ABI path (pack + H2D + solve + D2H every step).

`sub_records` (rank 0, same timing discipline: >= 3 warm-ups, CUDA events on the solver's stream, working sets larger
than L2 or stated otherwise; each with the CPU oracle beside it):
  config2_batch   config 2 at batch 1 / 64 / 1024 (latency and throughput, BASELINE.md section 3 row 2)
  config3         + ground-plane prior + plane chain, FP64 and FP32 linearisation (row 3)
  config4_lidar   lidar depth extraction, 120k-point cloud, 2000 features (row 4)
  config5         100 KF / 20k LM / 300k obs window: one GPU, and -- when launched on N > 1 ranks -- the landmark-sharded
                  solve with the NCCL all-reduce of the reduced system, checked against the one-GPU solve (row 5)

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--no-sub] [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "BA windows/s (30 KF, 3k LM, 40k obs)"
# Algorithmic bytes per observation of the residual/Jacobian kernel, mono + depth FP64 (SURVEY.md 8(d)): reads u, v, d (12) +
# keyframe index (4) + landmark data (~3); writes residual 3x8 + J_pose 3x6x8 [+ J_landmark 3x3x8].  Since round 2 the
# small-window path does not materialise J_landmark (its consumers re-form it as J_pose[:, 3:6] R): 259 - 72 = 187 B.
FUSED = os.environ.get("KBA_FUSED", "1") != "0"
# One-kernel linearisation (kba_linearize.cuh, default): the Jacobian is never materialised; the kernel reads the measurements
# and writes V_i = (J_p^T J_l) L^-T (144 B per observation) plus the landmark blocks.  SURVEY.md 8(d) gives the algorithmic
# bytes of such a fused kernel: reads 16 + 2.7, writes E_ij 144 per observation + (C_j 48 + g_j 24) per landmark = 5.4 -> 168 B.
LIN1 = FUSED and os.environ.get("KBA_LINEARIZE", "1") != "0"
B_OBS_ALGORITHMIC = 168.0 if LIN1 else (187.0 if FUSED else 259.0)
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of that kernel / its observations, from the ncu --set full
# capture summarised in profiles/ (re-measured whenever the kernel changes)
B_OBS_DRAM_MEASURED = 184.6 if LIN1 else (199.0 if FUSED else 277.0)
TRAFFIC_SOURCE = ("ncu --set full, profiles/r02_ncu_summary.md (k_linearize)" if LIN1 else
                  "ncu --set full, profiles/r02_ncu_summary.md (k_eval_obs<true>, J_landmark not materialised)" if FUSED else
                  "ncu --set full, profiles/r01_v11_ncu_summary.md: (0.200 GB read + 1.293 GB written) / 5.39 M observations")
KERNEL_NAME = ("k_linearize (residual/Jacobian + landmark blocks + V rows, one kernel)" if LIN1 else "k_eval_obs<true> (residual/Jacobian)")
ALG_NOTE = ("SURVEY 8(d), fused Hessian kernel: 18.7 B read + 144 B (E_ij) written per observation + 72 B per landmark; the Jacobian "
            "stays in registers.  The kernel is bound by instruction latency at 16 warps per SM (issue slots 31 % used, FP64 pipe 24 % busy), not by HBM: see profiles/r02_ncu_summary.md" if LIN1 else
            "19 B read + 168 B written (residual 24 + J_pose 144); J_landmark (72 B) is not materialised" if FUSED else "SURVEY 8(d): 259 B/obs")
CONFIG2 = "config 2: 30 KF / 3000 LM / 40000 obs, mono + lidar depth, FP64"


def usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def make_windows(n_distinct, rank, config=2):
    from limo_b200 import parallel
    return parallel.windows_for_rank(n_distinct, rank, config)


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 60 * 10**6  # array data of --dump-outputs: with the .npy headers, below 64 MB
SOLVE_FIELDS = ("initial_cost", "final_cost", "num_iterations", "num_successful_steps", "termination", "num_landmarks",
                "num_residual_blocks")


def dump_outputs(out_dir, results, windows):
    """Writes what a caller of the resident batch solve receives, one DIR/<name>.npy per array (float64; the rejection flags
    as float32), windows stacked along the first axis in batch order, so that two builds can be compared output for output.
    solve_<field> holds the summary of every inner solve, zero past num_solves.  When the whole batch would exceed
    DUMP_LIMIT_BYTES, a fixed, seeded sample of whole windows is written; window_index names the windows kept."""
    from limo_b200.capi_types import KBA_MAX_SOLVES
    arrays = {
        "kf_pose": np.stack([r.kf_pose for r in results]),
        "kf_plane": np.stack([r.kf_plane for r in results]),
        "lm_pos": np.stack([r.lm_pos[:w.n_lm] for r, w in zip(results, windows)]),
        "lm_rejected": np.stack([r.lm_rejected[:w.n_lm] for r, w in zip(results, windows)]).astype(np.float32),
        "status": np.array([r.c.status for r in results], dtype=np.float64),
        "num_solves": np.array([r.c.num_solves for r in results], dtype=np.float64),
        "initial_cost": np.array([r.c.initial_cost for r in results]),
        "final_cost": np.array([r.c.final_cost for r in results]),
        "window_index": np.arange(len(results), dtype=np.float64),
    }
    for f in SOLVE_FIELDS:
        a = np.zeros((len(results), KBA_MAX_SOLVES))
        for i, r in enumerate(results):
            a[i, :r.c.num_solves] = [getattr(s, f) for s in r.solves]
        arrays["solve_" + f] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES * len(results) // total
        idx = np.sort(np.random.default_rng(0).choice(len(results), keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs: the oracle (restatement of the reference's Ceres path; Ceres itself is not installable offline, DESIGN.md)
# ---------------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def oracle():
    """the CPU oracle, compiled -O3 -march=native for THIS host (BASELINE.md section 2)"""
    if not _ORACLE:
        os.environ.setdefault("OMP_WAIT_POLICY", "passive")
        from oracle import oracle as orc
        _ORACLE["build"] = orc.use_native_build()
        orc.lib()
        _ORACLE["mod"] = orc
    return _ORACLE["mod"]


def cpu_threads_all():
    return min(usable_cores(), 128)


def thread_candidates(cores):
    """OpenMP thread counts probed for the CPU legs.  The oracle parallelises over observations and is memory-bound: on the
    128-core, two-socket GPU hosts 128 threads measured 25x SLOWER than 32 (profiles/r02_bench.md), so the probe stays
    within one socket's worth of threads and picks the fastest."""
    return sorted({t for t in (16, 32, 64) if t <= cores} or {cores})


def cpu_time_windows(windows, n_sample, threads, warm=True):
    """n_sample full window solves, cycling through `windows`; returns (windows/s, seconds)"""
    orc = oracle()
    if warm:
        orc.solve_window(windows[0], num_threads=threads)  # page-in, thread pool
    t = time.perf_counter()
    for i in range(n_sample):
        orc.solve_window(windows[i % len(windows)], num_threads=threads)
    dt = time.perf_counter() - t
    return n_sample / dt, dt


def cpu_baseline_record(windows, n_all, n_three, label):
    """the reference's algorithm on this host's cores: with every core OpenMP can use, with the best of {32, all} threads
    (memory-bound beyond a socket), and with the reference's own setting of 3 threads (robust_solving.hpp:98)"""
    cores = cpu_threads_all()
    cand = thread_candidates(cores)
    probe = {}
    for t in cand:  # one solve each to pick the faster thread count (the warm-up of the measurement)
        _, dt = cpu_time_windows(windows, 1, t, warm=(t == cand[0]))
        probe[t] = dt
    best = min(probe, key=probe.get)
    val, dt = cpu_time_windows(windows, n_all, best, warm=False)
    rec = {"value": val, "unit": "windows/s", "cores": best, "kind": "port", "build": _ORACLE["build"],
           "sample": "%d full window solves of %s, %.1f s (oracle/, OpenMP; one-solve probe: %s)"
                     % (n_all, label, dt, ", ".join("%d threads %.2f s" % (t, probe[t]) for t in cand))}
    if n_three > 0:
        v3, d3 = cpu_time_windows(windows, n_three, 3, warm=False)
        rec["reference_setting_3_threads"] = {"value": v3, "unit": "windows/s", "cores": 3,
                                              "sample": "%d solves, %.1f s (num_threads = 3 as robust_solving.hpp:98)" % (n_three, d3)}
    return rec


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (its restatement in oracle/, since Ceres is not installable
    offline -- see DESIGN.md) on the host cores, same metric, configuration and WINDOWS as the b200 arm."""
    if rank != 0:
        return
    n_distinct = max(1, min(args.distinct, args.batch))
    wins = make_windows(n_distinct, 0)
    cores = cpu_threads_all()
    cand = thread_candidates(cores)
    probe = {t: cpu_time_windows(wins, 1, t, warm=True)[1] for t in cand}
    threads = min(probe, key=probe.get)
    for i in range(max(args.warmup - 1, 0)):
        oracle().solve_window(wins[i % len(wins)], num_threads=threads)
    per_step = 1  # a bounded sample of the step's batch: one window per step, cycling through the same windows
    t = time.perf_counter()
    for s in range(args.steps):
        oracle().solve_window(wins[s % len(wins)], num_threads=threads)
    dt = time.perf_counter() - t
    val = args.steps * per_step / dt
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "windows/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": CONFIG2, "batch_windows_per_gpu": args.batch, "distinct_windows_per_gpu": n_distinct,
                      "sample": "one window solve per step, cycling through the b200 arm's %d distinct windows" % n_distinct},
           "cpu_baseline": {"value": val, "unit": "windows/s", "cores": threads, "kind": "port", "build": _ORACLE["build"],
                            "sample": "%d full window solves (oracle/, OpenMP %d threads; probe %s)"
                                      % (args.steps, threads, ", ".join("%d: %.2f s" % (t_, probe[t_]) for t_ in cand))},
           "e2e": {"value": val, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def timed_resident(torch, batch, opt, stream, steps, warmup, barrier=None):
    """K solves of a resident batch between CUDA events on the solver's stream; returns ms for the K steps"""
    for _ in range(warmup):
        batch.solve(opt)
    if barrier:
        barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        batch.solve(opt)
    ev1.record(stream)
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def sub_config2_batches(torch, capi, h, stream, base, opt, cpu_ws):
    """config 2 at batch 1 / 64 / 1024: latency of one solve and throughput (resident and end to end)"""
    out = []
    for b, steps in ((1, 10), (64, 5), (1024, 3)):
        wins = [base[i % len(base)] for i in range(b)]
        batch = h.batch(wins)
        ms = timed_resident(torch, batch, opt, stream, steps, 3)
        res = None
        t = time.perf_counter()
        for _ in range(steps):
            batch.upload(); batch.solve(opt); res = batch.download(results=res)
        ms_e2e = 1e3 * (time.perf_counter() - t)
        out.append({"batch": b, "steps": steps, "windows_per_s": b * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                    "e2e_windows_per_s": b * steps / (ms_e2e * 1e-3), "converged": all(r.c.status == 0 for r in res),
                    "l2_policy": "working set %.2f GB%s" % (b * wins[0].n_obs * 168 / 1e9, " (fits L2: latency case)" if b == 1 else "")})
        batch.close()
    one = out[0]
    one["speedup_vs_cpu_one_window"] = (1.0 / cpu_ws) / (one["ms_per_step"] * 1e-3)
    return out


def sub_config3(torch, capi, h, stream, rank):
    """config 3: + ground-plane residuals, plane blocks and the regularisation chain; FP64 and FP32 linearisation"""
    wins = make_windows(8, rank, config=3)
    batch_n = 148
    tiled = [wins[i % len(wins)] for i in range(batch_n)]
    rec = {"workload": "config 3: 30 KF / 3000 LM / 40000 obs + ground-plane prior + plane chain, trimmed", "batch": batch_n}
    results = {}
    for name, prec in (("fp64", 0), ("fp32", 1)):
        opt = capi.default_options()
        opt.precision = prec
        batch = h.batch(tiled)
        ms = timed_resident(torch, batch, opt, stream, 3, 3)
        res = batch.download()
        results[name] = res
        rec[name] = {"windows_per_s": batch_n * 3 / (ms * 1e-3), "ms_per_step": ms / 3,
                     "converged": all(r.c.status == 0 for r in res),
                     "lm_iterations_mean": float(np.mean([sum(s.num_iterations for s in r.solves) for r in res]))}
        batch.close()
    a, b = results["fp64"][:len(wins)], results["fp32"][:len(wins)]  # the distinct windows
    dt = [float(np.linalg.norm(x.kf_pose[:, 4:] - y.kf_pose[:, 4:], axis=1).max()) for x, y in zip(a, b)]
    dc = [float(abs(x.c.final_cost - y.c.final_cost) / x.c.final_cost) for x, y in zip(a, b)]
    drej = [int((x.lm_rejected != y.lm_rejected).sum()) for x, y in zip(a, b)]
    same = [i for i, d in enumerate(drej) if d == 0]
    rec["fp32_vs_fp64"] = {"windows_compared": len(a), "max_translation_diff_m": max(dt), "max_rel_cost_diff": max(dc),
                           "landmarks_rejected_differently_max": max(drej), "windows_with_identical_rejections": len(same),
                           "max_translation_diff_m_identical_rejections": max([dt[i] for i in same], default=None),
                           "max_rel_cost_diff_identical_rejections": max([dc[i] for i in same], default=None),
                           "stated_tolerance": "BASELINE.md section 3: FP32 linearisation -- translation <= 1e-2 m; cost relative <= 1e-5 when the "
                                               "trimming rejects the same landmarks, else the costs are those of different problems"}
    rec["cpu_baseline"] = cpu_baseline_record(wins, 3, 0, "config 3")
    return rec


def sub_config4(torch, capi, h):
    """lidar depth extraction: 120k-point cloud -> 1242x375, 2000 features"""
    from limo_b200 import synth
    cloud, T, K, feats = synth.make_lidar_scene()
    for _ in range(3):
        depth, ms = h.lidar_depth(cloud, T, K, feats)
    n = 50
    t = time.perf_counter()
    dev = []
    for _ in range(n):
        depth, ms = h.lidar_depth(cloud, T, K, feats)
        dev.append(ms)
    wall = time.perf_counter() - t
    dev_ms = float(np.median(dev))
    peak, _ = measured_peak()
    orc = oracle()
    orc.lidar_depth(cloud, T, K, feats)
    t = time.perf_counter()
    for _ in range(5):
        d_cpu = orc.lidar_depth(cloud, T, K, feats)
    cpu_s = (time.perf_counter() - t) / 5
    alg = 16.0 * len(cloud) * 2 + 24.0 * len(cloud)  # two projection passes over x,y,z,i + the cell-sorted point records
    return {"workload": "config 4: %d-point cloud -> 1242x375, %d features" % (len(cloud), len(feats)),
            "clouds_per_s_device": 1e3 / dev_ms, "device_ms_per_cloud": dev_ms,
            "clouds_per_s_e2e": n / wall, "e2e_note": "kba_lidar_depth with host buffers: H2D of the cloud (%.2f MB) + kernels + D2H, per call" % (cloud.nbytes / 1e6),
            "features_with_depth": int((depth > 0).sum()), "bit_exact_vs_oracle": bool(np.array_equal(depth, d_cpu)),
            "roofline": {"bound": "hbm", "achieved": alg / (dev_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (dev_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_cloud": alg,
                         "note": "2 MB per cloud: launch-latency bound (4 kernels), not bandwidth bound -- batch clouds to use the GPU"},
            "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "clouds/s", "cores": 1, "kind": "port", "build": _ORACLE["build"],
                             "sample": "5 clouds, single thread (oracle/lidar_oracle.c; parity unpinned: no reference code exists)"}}


def sub_config5(torch, capi, h, stream, rank, local_rank, world):
    """one 100-keyframe window: on one GPU, and sharded by landmark blocks over all ranks (NCCL all-reduce of [S | rhs])"""
    from limo_b200 import parallel, synth
    import torch.distributed as dist
    win = synth.make_window(5)
    opt = capi.default_options()
    rec = {"workload": "config 5: %d KF / %d LM / %d obs, mono + lidar depth, FP64" % (win.n_kf, win.n_lm, win.n_obs)}
    ref = None
    if rank == 0:
        batch = h.batch([win])
        ms = timed_resident(torch, batch, opt, stream, 3, 3)
        ref = batch.download(iterations_capacity=1)[0]
        batch.close()
        rec["one_gpu"] = {"ms_per_solve": ms / 3, "windows_per_s": 3 / (ms * 1e-3),
                          "lm_iterations": [s.num_iterations for s in ref.solves], "converged": ref.c.status == 0}
    if world > 1:
        sub, j0, j1 = parallel.shard_window(win, rank, world)
        idt = torch.zeros(capi.SHARD_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(capi.shard_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        comm = capi.ShardComm(h, rank, world, bytes(idt.cpu().numpy().tobytes()))
        batch = h.batch([sub])
        batch.set_shard(comm, j0, win.n_lm)
        ms = timed_resident(torch, batch, opt, stream, 3, 3, barrier=lambda: parallel.barrier(cuda=True))
        ms, = parallel.max_over_ranks([ms], device="cuda")
        r = batch.download()[0]
        # all-reduce of one [S | rhs] buffer, timed alone on the same ranks (the solve issues one per linearisation)
        nr_cap = ((6 * win.n_kf + 1 + 63) // 64) * 64
        buf = torch.zeros(nr_cap * nr_cap, dtype=torch.float64, device="cuda")
        for _ in range(5):
            dist.all_reduce(buf)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(20):
            dist.all_reduce(buf)
        e1.record(); torch.cuda.synchronize()
        ar_us, = parallel.max_over_ranks([1e3 * e0.elapsed_time(e1) / 20], device="cuda")
        lm_full = torch.zeros(win.n_lm * 3, dtype=torch.float64, device="cuda")
        lm_full[3 * j0:3 * j1] = torch.from_numpy(np.ascontiguousarray(r.lm_pos[:sub.n_lm]).reshape(-1)).cuda()
        dist.all_reduce(lm_full)
        if rank == 0:
            dl = np.linalg.norm(lm_full.cpu().numpy().reshape(-1, 3) - ref.lm_pos[:win.n_lm], axis=1)
            rec["sharded"] = {
                "n_gpus": world, "ms_per_solve": ms / 3, "speedup_vs_one_gpu": rec["one_gpu"]["ms_per_solve"] / (ms / 3),
                "allreduce_us": ar_us, "allreduce_bytes": int(buf.numel() * 8),
                "allreduce_note": "one [S | rhs] all-reduce of the reduced pose system, timed alone (20 calls); the solve issues one per linearisation",
                "lm_iterations": [s.num_iterations for s in r.solves],
                "same_iterations_as_one_gpu": [s.num_iterations for s in r.solves] == [s.num_iterations for s in ref.solves],
                "max_translation_diff_vs_one_gpu_m": float(np.linalg.norm(r.kf_pose[:, 4:] - ref.kf_pose[:, 4:], axis=1).max()),
                "rel_cost_diff_vs_one_gpu": float(abs(r.solves[-1].final_cost - ref.solves[-1].final_cost) / ref.solves[-1].final_cost),
                "p95_landmark_diff_vs_one_gpu_m": float(np.percentile(dl, 95)),
                "parity_ok": bool(np.linalg.norm(r.kf_pose[:, 4:] - ref.kf_pose[:, 4:], axis=1).max() <= 1e-6)}
        batch.close()
        comm.close()
    if rank == 0 and world == 1:
        _, dt = cpu_time_windows([win], 1, min(32, cpu_threads_all()), warm=False)
        rec["cpu_baseline"] = {"value": 1.0 / dt, "unit": "windows/s", "cores": min(32, cpu_threads_all()), "kind": "port",
                               "build": _ORACLE["build"], "sample": "1 full solve of the config-5 window, %.1f s" % dt}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=296, help="windows per GPU per step (two per SM: the windows of a batch\n"
                    "advance in lock-step passes, a larger batch amortises the passes in which only the slowest windows are left)")
    ap.add_argument("--distinct", type=int, default=16, help="distinct synthetic windows per GPU (tiled to --batch)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=6, help="window solves timed for cpu_baseline (~0.5 s each); 0 = skip the CPU legs")
    ap.add_argument("--in-flight", type=int, default=4, help="steps in flight of the end-to-end measurement (handles / streams)")
    ap.add_argument("--no-sub", action="store_true", help="headline only: skip the sub-records of configs 3, 4, 5 and the batch sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (rank 0's windows) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")

    from limo_b200 import parallel
    rank, local_rank, world = parallel.rank_info()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the kba_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    parallel.init("nccl", torch.device("cuda", local_rank))
    from limo_b200 import capi
    # host threads that pack a step's windows: share the box's cores between the ranks and the steps in flight
    os.environ.setdefault("KBA_HOST_THREADS", str(max(2, min(16, usable_cores() // (max(1, min(args.in_flight, usable_cores() // (4 * world))) * world)))))

    n_distinct = max(1, min(args.distinct, args.batch))
    base = make_windows(n_distinct, rank)
    windows = [base[i % n_distinct] for i in range(args.batch)]
    n_obs_win = windows[0].n_obs

    # a stream of its own, not the legacy default stream: the library issues a solve as one CUDA graph (the passes are the body
    # of a conditional WHILE node), and the legacy stream cannot be captured -- there it falls back to kernel-by-kernel launches
    torch.cuda.set_stream(torch.cuda.Stream())
    stream = torch.cuda.current_stream()
    h = capi.Handle(local_rank, stream=stream.cuda_stream)
    opt = capi.default_options()
    batch = h.batch(windows)

    def barrier():
        parallel.barrier(cuda=True)

    # ---- warm-up ----
    for _ in range(args.warmup):
        batch.solve(opt)
    barrier()
    h.counters(reset=True)
    h.enable_kernel_timing(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed region: K steps, inputs resident in HBM ----
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        batch.solve(opt)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    cnt = h.counters(reset=True)
    h.enable_kernel_timing(False)
    results = batch.download()
    if args.dump_outputs and rank == 0:  # before the end-to-end steps below reuse these result buffers
        dump_outputs(args.dump_outputs, results, windows)
    done = all(r.c.status == 0 for r in results)
    converged = all(r.solves[r.c.num_solves - 1].termination == 0 for r in results)  # KBA_TERM_CONVERGENCE of the final solve
    iters = [sum(s.num_iterations for s in r.solves) for r in results]

    # ---- end-to-end: host buffers -> pack -> H2D -> solve -> D2H, every step ----
    for _ in range(1):
        batch.upload(); batch.solve(opt); batch.download(results=results)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e0.record(stream)
    t_up = t_dn = 0.0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        batch.upload()       # host pack (threads) + async H2D
        t1 = time.perf_counter()
        batch.solve(opt)     # returns when every window is done
        t2 = time.perf_counter()
        batch.download(results=results)
        t_up += t1 - t0; t_dn += time.perf_counter() - t2
    e1.record(stream)
    barrier()
    ms_e2e_seq = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t_wall))

    # ---- end-to-end, several steps in flight: further handles (own stream, own device buffers) let the host pack and copy
    #      step i+1 while the GPU solves step i.  Every step still does its own pack + H2D + solve + D2H inside the
    #      timed region; ctypes releases the GIL during the C calls, so two Python threads are enough. ----
    # a lane needs a host thread for the launches plus a few packing threads: fewer lanes when the ranks share few cores
    n_lanes = max(1, min(args.in_flight, usable_cores() // (4 * world)))
    extra = []
    lanes = [(batch, results)]
    if n_lanes * world > 1:  # the additional handles sleep while they wait for the GPU (see kba_api.cu wait_stream)
        os.environ["KBA_BLOCKING_SYNC"] = "1"
    for _ in range(n_lanes - 1):
        st_ = torch.cuda.Stream()
        h_ = capi.Handle(local_rank, stream=st_.cuda_stream)
        b_ = h_.batch(windows)
        extra.append((st_, h_, b_))
        lanes.append((b_, b_.download()))
    for b_, r_ in lanes:  # warm-up of both lanes
        b_.upload(); b_.solve(opt); b_.download(results=r_)
    barrier()

    todo = {"left": args.steps}
    todo_lock = threading.Lock()

    def lane(idx):
        torch.cuda.set_device(local_rank)
        b_, r_ = lanes[idx]
        while True:
            with todo_lock:  # the lanes pull steps from one counter: balanced for any K
                if todo["left"] <= 0:
                    return
                todo["left"] -= 1
            b_.upload(); b_.solve(opt); b_.download(results=r_)

    threads = [threading.Thread(target=lane, args=(i,)) for i in range(min(n_lanes, args.steps))]
    t_wall = time.perf_counter()
    for t_ in threads:
        t_.start()
    for t_ in threads:
        t_.join()
    torch.cuda.synchronize()
    ms_e2e = 1e3 * (time.perf_counter() - t_wall)
    barrier()
    done = done and all(r.c.status == 0 for _, rs in lanes[1:] for r in rs)
    clocks = sampler.stop()  # sampled over all timed regions
    h2d, d2h = batch.transfer_bytes()
    # the materialising residual/Jacobian kernel alone (k_eval_obs<true>: what large windows, the FP32 mode and kba_eval run, and
    # what k_linearize replaced on this path): every window active, 20 back-to-back launches between CUDA events, best of 3
    jac_alone_ms = None
    if rank == 0:
        batch.jacobian_pass(opt, 5)
        jac_alone_ms = min(batch.jacobian_pass(opt, 20) for _ in range(3)) / 20.0
    for _, h_, b_ in extra:
        b_.close()
        h_.close()
    batch.close()

    ms, ms_e2e, ms_e2e_seq = parallel.max_over_ranks([ms, ms_e2e, ms_e2e_seq], device="cuda")  # slowest rank

    # ---- sub-records: the other BASELINE configurations (rank 0; the sharded config-5 solve on all ranks) ----
    sub = {}
    do_cpu = args.cpu_sample > 0
    cpu_rec = None
    if rank == 0 and do_cpu:
        cpu_rec = cpu_baseline_record(base, args.cpu_sample, 2, "the same workload")
    if not args.no_sub:
        if world == 1 and do_cpu:
            sub["config2_batch"] = sub_config2_batches(torch, capi, h, stream, base, opt, cpu_rec["value"])
            sub["config3"] = sub_config3(torch, capi, h, stream, rank)
            sub["config4_lidar"] = sub_config4(torch, capi, h)
        if do_cpu or world > 1:
            sub["config5"] = sub_config5(torch, capi, h, stream, rank, local_rank, world)
        if world > 1:
            sub["note"] = "N > 1: only the sharded config-5 record is measured next to the headline; configs 3 / 4 and the batch sweep are in the N = 1 line"

    if rank == 0:
        total_windows = world * args.batch * args.steps
        value = total_windows / (ms * 1e-3)
        peak, peak_src = measured_peak()
        jac_gbs = (cnt.jacobian_obs * B_OBS_ALGORITHMIC / (cnt.ms_jacobian * 1e-3) / 1e9) if cnt.ms_jacobian > 0 else None
        out = {
            "metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": CONFIG2,
                       "batch_windows_per_gpu": args.batch, "distinct_windows_per_gpu": n_distinct,
                       "parallelism": "independent windows per GPU (no data-path collective)" if world > 1 else "1 GPU",
                       "lm_iterations_per_window_mean": float(np.mean(iters)),
                       "lm_iterations_per_window_max": int(np.max(iters)),
                       "l2_policy": "inputs larger than L2 (%.1f GB of V blocks written and re-read per pass)"
                                    % (args.batch * n_obs_win * 144.0 / 1e9),
                       "all_windows_finished": bool(done), "all_final_solves_converged": bool(converged)},
            "e2e": {"value": total_windows / (ms_e2e * 1e-3), "unit": "windows/s",
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps_in_flight": n_lanes, "sequential_value": total_windows / (ms_e2e_seq * 1e-3),
                    "host_pack_upload_ms_per_step": 1e3 * t_up / args.steps,
                    "download_ms_per_step": 1e3 * t_dn / args.steps},
            "gpu_launches": int(cnt.launches_total),
            "roofline": {"kernel": KERNEL_NAME, "bound": "hbm", "achieved": jac_gbs,
                         "peak": peak, "unit": "GB/s", "frac": (jac_gbs / peak) if jac_gbs else None,
                         "peak_source": peak_src,
                         "traffic": B_OBS_DRAM_MEASURED * cnt.jacobian_obs / max(cnt.launches_jacobian, 1),
                         "traffic_unit": "bytes per launch", "traffic_source": TRAFFIC_SOURCE,
                         "algorithmic_bytes_per_obs": B_OBS_ALGORITHMIC,
                         "algorithmic_note": ALG_NOTE,
                         "launch_ms_mean": cnt.ms_jacobian / max(cnt.launches_jacobian, 1),
                         "launches": int(cnt.launches_jacobian), "share_of_timed_region": cnt.ms_jacobian / ms,
                         "obs_per_launch_mean": cnt.jacobian_obs / max(cnt.launches_jacobian, 1)},
            "roofline_jacobian_kernel": {
                "kernel": "k_eval_obs<true> alone (materialising residual/Jacobian kernel; not on the timed path of this workload)",
                "bound": "hbm", "achieved": args.batch * n_obs_win * 187.0 / (jac_alone_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": args.batch * n_obs_win * 187.0 / (jac_alone_ms * 1e-3) / 1e9 / peak, "launch_ms": jac_alone_ms,
                "algorithmic_bytes_per_obs": 187.0,
                "note": "19 B read + 168 B written (residual 24 + J_pose 144; J_landmark = translation columns of J_pose x R is not stored)"},
            "host_cores": usable_cores(),
            "cpu_baseline": cpu_rec if cpu_rec else {"value": None, "unit": "windows/s", "cores": 0, "kind": "port", "sample": "skipped (--cpu-sample 0)"},
            "sub_records": sub,
            "clocks": clocks,
        }
        print(json.dumps(out))
    h.close()
    parallel.finalize()


if __name__ == "__main__":
    main()
