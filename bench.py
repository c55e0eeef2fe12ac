#!/usr/bin/env python
"""bench.py — headline benchmark of the COVINS hot path on B200 (contract: see DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--gba-config C3] [--dump-outputs DIR]

Metric (BASELINE.json): global-BA iterations/s & descriptor-match Gpairs/s on the 5-agent EuRoC-sized synthetic map
(config C3: 2000 KF / 100k LM / ~800k obs; 1000 ORB features per KF).  One "step" is one pass of the hot path: one outer
trust-region iteration of the visual-inertial global BA (linearise → Schur → Cholesky → dogleg → candidate cost) and one
query keyframe matched against every keyframe of the rank's map shard (2 Gpairs, fused k-NN + ratio filter).  The legs
are timed separately; the JSON line carries the GBA rate as `value` and the matching rate under `match` (each with its
own e2e / roofline / cpu_baseline); `pgo` carries the pose-graph optimisation rate on the same map, `match.sift_l2` /
`match.landmark_descriptor` the SIFT and ComputeDescriptor kernels.  Scalars of the nested legs are repeated at the top
level (`match_gpairs_per_sec`, `pgo_iterations_per_sec`, …) so that per-N scaling records carry them.

`--impl reference`: the CPU arm — the compiled CPU port of the optimisation path (oracle/ba_port.cpp: analytic Jacobians,
Schur complement, tile-sparse BLAS-3 Cholesky, Ceres dogleg; OpenMP on all host cores) on the SAME config and the SAME
number of trust-region iterations, and OpenCV's own BFMatcher.knnMatch (cv2, the library call the reference makes) for the
matching leg.  The reference binary itself (Ceres/CHOLMOD/robopt/ROS) cannot be built offline (DESIGN.md §1).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_KF, N_FEAT = 2000, 1000          # C3: 5 agents x 400 KF, 1000 ORB features per KF
THR, RATIO = 40.0, 0.8             # config/config_backend.yaml:38-39
N_COPIES = 4                       # 4 x 64 MB map copies rotated per step → inputs (256 MB) > L2 (126 MB)

WORKLOAD = ("C3 5-agent EuRoC-sized synthetic map (2000 KF / 100k LM / ~800k obs, 1000 ORB features per KF): "
            "visual-inertial global-BA trust-region iterations + ORB k-NN(k=2)+ratio-filter of one query KF vs every KF")


def _measured():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def _peaks():
    d = _measured()
    return (d["hbm_gbs"], "MEASURED_PEAKS.json") if "hbm_gbs" in d else (6650.0, "fallback (B200_PROFILING.md)")


def _traffic(key):
    """dram bytes per launch of a dominant kernel, from the committed ncu --set full captures (profiles/r02_traffic.json,
    written by tools/r02_traffic.py out of the .ncu-rep files); None when no capture is committed for `key`."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(key)
    return (d["dram_bytes"], d.get("source")) if d else (None, None)


class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU during the timed region (pynvml)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self._stop = index, [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        # NVML queries are slow (milliseconds) and serialise with the CUDA driver of this process: at N > 1 the host is in the
        # loop of every iteration (the all-reduce callback), and a 50 ms polling period doubled the measured step time (2 GPUs:
        # 44.9 ms per step against 20.5 ms of device phases).  So: few samples — the first 50 ms into the region, then one per second.
        nv = self.nv
        names = {getattr(nv, n): n for n in dir(nv) if n.startswith("nvmlClocksEventReason") or n.startswith("nvmlClocksThrottleReason")}
        if self._stop.wait(0.05):
            return
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in (names.items() if r else ()):
                    if isinstance(bit, int) and bit and (r & bit) and bit != getattr(nv, "nvmlClocksThrottleReasonGpuIdle", 1):
                        short = name.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", "")
                        if short not in ("All", "None", "ApplicationsClocksSetting", "GpuIdle"):
                            self.reasons.add(short)
            except Exception:
                pass
            if self._stop.wait(1.0):
                break

    def __enter__(self):
        if self.nv:
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=1.0)
            if not self.samples:     # region shorter than 50 ms: one sample right after it (the GPU is still clocked up)
                try:
                    self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                except Exception:
                    pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def dist_info():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Writes each array (numpy or torch) as d/<name>.npy so that two builds can be compared output for output:
    float64 stays float64, every other type becomes float32 (integers up to 2^24 exactly, larger ones float64)."""
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        if a.dtype != np.float64:
            exact32 = a.dtype.kind == "f" or a.size == 0 or np.abs(a).max() < 2 ** 24
            a = a.astype(np.float32 if exact32 else np.float64)
        out[name] = a
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"outputs take {total} bytes, more than the {DUMP_LIMIT_BYTES} a dump may hold")
    os.makedirs(d, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)


def _cores():
    """usable host cores: affinity mask capped by the cgroup CPU quota (the GPU boxes expose 128 CPUs with a 16-core quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


# ==================================================================================================
# CPU legs (oracle/ is the checker and the timed CPU port, never the product)
# ==================================================================================================
def cpu_gba(config, iters, warmup=0):
    """The compiled CPU port of the optimisation path on `config`: `iters` trust-region iterations of the visual-inertial
    GBA solve (the same solve the GPU arm times), all host cores.  Returns (cpu_baseline dict, e2e value)."""
    from covins_b200 import synth_map
    from oracle import ba_port as bp
    cores = _cores()
    p = synth_map.make_config(config)
    if warmup > 0:
        bp.solve(p, warmup, visual_only=False, threads=cores)
    done, t_solve, t_total, ph = 0, 0.0, 0.0, None
    while done < iters:                     # a solve that converges early is repeated from the initial state
        t0 = time.perf_counter()
        r = bp.solve(p, iters - done, visual_only=False, threads=cores)
        dt = time.perf_counter() - t0
        n = max(int(r["iterations"]), 1)
        done += n; t_total += dt; t_solve += dt - r["phase_s"]["setup"]; ph = r["phase_s"]
    base = {"value": done / t_solve, "unit": "iterations/s", "cores": cores, "kind": "port", "iterations": done,
            "sample": f"oracle/ba_port.cpp (C++17/OpenMP x{cores}: analytic Jacobians, Schur complement, tile-sparse Cholesky on "
                      f"scipy's OpenBLAS dgemm/dsyrk/dtrsm/dpotrf {'(in use)' if bp.lib().blas else '(NOT found: plain loops)'}, Ceres dogleg): "
                      f"{done} trust-region iterations of the visual-inertial GBA on synthetic config {config} "
                      f"({p['K']} KF / {p['L']} LM / {len(p['obs_kf'])} obs) in {t_solve:.1f} s (+ {t_total - t_solve:.1f} s problem set-up); "
                      f"restated CPU path, not the Ceres/CHOLMOD binary (unavailable offline)",
            "phase_s_last_call": {k: round(v, 3) for k, v in ph.items()},
            "factor_gflops": round(r["factor_flops"] * max(int(r["iterations"]), 1) / max(ph["factor"], 1e-9) / 1e9, 1)}
    return base, done / t_total


def cpu_pgo(p, edges, iters):
    from oracle import ba_port as bp
    cores = _cores()
    pp = dict(K=p["K"], L=0, pose=p["pose"], pose_const=p["pose_const"], extr=p["extr"], cam_of_kf=p.get("cam_of_kf"))
    t0 = time.perf_counter()
    r = bp.solve(pp, iters, visual_only=True, cauchy_reproj=0.0, cauchy_edge=0.5, edges=edges, threads=cores)
    dt = time.perf_counter() - t0 - r["phase_s"]["setup"]
    n = max(int(r["iterations"]), 1)
    return {"value": n / dt, "unit": "iterations/s", "cores": cores, "kind": "port", "iterations": n,
            "sample": f"oracle/ba_port.cpp (OpenMP x{cores}) on the same pose graph: {n} iterations in {dt:.2f} s"}


def cpu_match_cv2(steps, warmup, n_cand=48):
    """cv2.BFMatcher(NORM_HAMMING).knnMatch — the OpenCV call of placerec_gen_be.cpp:99 — per candidate keyframe"""
    from covins_b200 import synth
    cores = _cores()
    desc, _ = synth.orb_keyframes(seed=3, n_kf=n_cand + 1, n_feat=N_FEAT)
    q, cands = desc[0], desc[1:]
    kind = "reference"
    try:
        import cv2
        cv2.setNumThreads(cores)
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)

        def step():
            for c in cands:  # the per-candidate loop of placerec_gen_be.cpp:72-125; only the C++ call is timed —
                bf.knnMatch(q, c, k=2)   # unpacking DMatch objects in Python would charge the CPU arm for the binding
        sample = (f"cv2 {cv2.__version__} BFMatcher(NORM_HAMMING).knnMatch(k=2), 1000-feature query KF vs {n_cand} candidate "
                  f"KFs per step (the OpenCV call of placerec_gen_be.cpp:99, OpenCV-internal threads; the ratio filter is "
                  f"negligible and not timed)")
    except Exception:
        from oracle import knn as ora
        kind = "port"
        t = cands.reshape(-1, 32); seg = synth.seg_ptr_uniform(n_cand, N_FEAT)

        def step():
            i, d = ora.knn_hamming_batch(q, t, seg, 2, threads=cores)
            return int(ora.ratio_filter(i, d.astype(np.float32), THR, RATIO)[2].sum())
        sample = f"oracle/knn_oracle.c (OpenMP, {cores} threads), 1000-feature query KF vs {n_cand} candidate KFs per step"
    for _ in range(max(1, min(warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    gp = n_cand * N_FEAT * N_FEAT * steps / dt / 1e9
    return {"value": gp, "unit": "Gpairs/s", "cores": cores, "kind": kind, "sample": sample}, dt / steps * 1e3


def cpu_match_port(budget_s=8.0):
    """oracle port (OpenMP, all cores) on a bounded sample of the same workload."""
    from covins_b200 import synth
    from oracle import knn as ora
    cores = _cores()
    n_cand = 64
    desc, _ = synth.orb_keyframes(seed=3, n_kf=n_cand + 1, n_feat=N_FEAT)
    q, t, seg = desc[0], desc[1:].reshape(-1, 32), synth.seg_ptr_uniform(n_cand, N_FEAT)
    ora.knn_hamming_batch(q, t, seg, 2, threads=cores)
    t0 = time.perf_counter(); reps = 0
    while time.perf_counter() - t0 < budget_s and reps < 400:
        i, d = ora.knn_hamming_batch(q, t, seg, 2, threads=cores)
        ora.ratio_filter(i, d.astype(np.float32), THR, RATIO)
        reps += 1
    dt = time.perf_counter() - t0
    return {"value": n_cand * N_FEAT * N_FEAT * reps / dt / 1e9, "unit": "Gpairs/s", "cores": cores, "kind": "port",
            "sample": f"oracle/knn_oracle.c OpenMP x{cores}: 1000-feature query KF vs {n_cand} candidate KFs, "
                      f"{reps} repetitions in {dt:.1f} s"}


def cpu_sift_port(budget_s=6.0):
    from covins_b200 import synth
    from oracle import knn as ora
    cores = _cores()
    n_cand, nf = 64, 300
    desc, _ = synth.sift_keyframes(seed=5, n_kf=n_cand + 1, n_feat=nf)
    q, t, seg = desc[0], desc[1:].reshape(-1, 128), synth.seg_ptr_uniform(n_cand, nf)
    ora.knn_l2_batch(q, t, seg, 2, threads=cores)
    t0 = time.perf_counter(); reps = 0
    while time.perf_counter() - t0 < budget_s and reps < 400:
        ora.knn_l2_batch(q, t, seg, 2, threads=cores); reps += 1
    dt = time.perf_counter() - t0
    return {"value": n_cand * nf * nf * reps / dt / 1e9, "unit": "Gpairs/s", "cores": cores, "kind": "port",
            "sample": f"oracle/knn_oracle.c (exact brute-force L2, OpenMP x{cores}): 300 SIFT queries vs {n_cand} candidate KFs x 300 rows, {reps} repetitions in {dt:.1f} s"}


# ==================================================================================================
# reference arm
# ==================================================================================================
def run_reference(args):
    rank, world, _ = dist_info()
    if rank != 0:
        return
    gba, e2e = cpu_gba(args.gba_config, args.steps, warmup=min(args.warmup, 1))
    match_base, ms_match = cpu_match_cv2(args.steps, args.warmup)
    match = {"metric": "match_gpairs_per_sec", "value": match_base["value"], "unit": "Gpairs/s", "ms_per_step": ms_match,
             "cpu_baseline": match_base}
    line = {
        "impl": "reference", "metric": "gba_iterations_per_sec", "value": gba["value"], "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": gba["iterations"], "warmup": min(args.warmup, 1), "ms_per_step": 1e3 / gba["value"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "gba_config": args.gba_config,
                   "note": "same map, same solve and the same number of trust-region iterations as the GPU arm; the matching "
                           "leg is a bounded sample (48 candidate keyframes per step), see match.cpu_baseline.sample"},
        "cpu_baseline": gba,
        "e2e": {"value": e2e, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "match": match, "match_gpairs_per_sec": match["value"],
    }
    print(json.dumps(line))


# ==================================================================================================
# our arm
# ==================================================================================================
def fp64_gemm_peak(dev):
    """FP64 GEMM throughput of this GPU (cuBLAS DGEMM 6144^3 via torch) — the denominator for the DMMA Cholesky,
    which MEASURED_PEAKS.json does not hold."""
    import torch
    n = 6144
    a = torch.randn(n, n, device=dev, dtype=torch.float64); b = torch.randn(n, n, device=dev, dtype=torch.float64)
    torch.matmul(a, b); torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def int8_gemm_peak(dev):
    """int8 x int8 -> int32 tensor throughput of this GPU (cuBLASLt IGEMM 8192^3 via torch._int_mm): the measured
    denominator of the kind::i8 matcher (MEASURED_PEAKS.json holds no int8 figure)."""
    import torch
    try:
        n = 8192
        a = torch.randint(-8, 8, (n, n), device=dev, dtype=torch.int8); b = torch.randint(-8, 8, (n, n), device=dev, dtype=torch.int8)
        torch._int_mm(a, b); torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12, "cuBLASLt IGEMM 8192^3 (torch._int_mm) measured in this run"
    except Exception as ex:  # noqa: BLE001
        bf = _measured().get("bf16_tflops", 1590.0)
        return 2.0 * bf, f"2 x bf16_tflops of MEASURED_PEAKS.json (torch._int_mm unavailable: {type(ex).__name__})"


def run_ours(args):
    import torch
    import torch.distributed as dist
    import covins_b200
    from covins_b200 import matching as M, optimization as O, synth, synth_map

    rank, world, local = dist_info()
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        # a rank that dies must end the run (watchdog abort) instead of parking the others for NCCL's default 10 minutes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(seconds=int(os.environ.get("COVINS_NCCL_TIMEOUT", "240"))))
    ctx = covins_b200.Context(local)
    dev = torch.device("cuda", local)
    hbm_peak, peak_src = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    # =============================================================================================
    # leg 1: global BA (strong scaling: the same C3 map; landmark blocks sharded over ranks, the reduced camera system
    # reduce-scattered onto tile-column owners over NVLink, factorisation distributed by tile columns)
    # =============================================================================================
    t_gen = time.perf_counter()
    prob = synth_map.make_config(args.gba_config)
    t_gen = time.perf_counter() - t_gen
    n_obs = len(prob["obs_kf"])
    solver = O.BaSolver(ctx, prob, visual_only=False, rank=rank, world=world, allreduce=O.torch_allreduce() if world > 1 else None)
    p2p = bool(solver.p2p)

    def run_iters(n):
        done = 0
        while done < n:
            k = solver.iterate(n - done)
            done += k
            if done < n:            # converged / terminated early: back to the initial state (cvb_ba_restart), solve again
                solver.restart()
        return done

    run_iters(args.warmup)
    solver.restart()                # the timed region starts from the initial state: its first iterations are real work
    solver.timing(reset=True)
    ctx.sync(); barrier()
    l0 = ctx.launch_count()
    with ClockSampler(local) as clk:
        t0 = time.perf_counter()
        run_iters(args.steps)
        ctx.sync()
        dt_gba = time.perf_counter() - t0
    barrier()
    gba_launches = ctx.launch_count() - l0
    dt_gba = max_over_ranks(dt_gba)
    tm = solver.timing(reset=True)
    gba_rate = args.steps / dt_gba
    res = solver.result()
    solver.close()
    dev_ms = sum(tm[k] for k in ("linearize_ms", "build_schur_ms", "factor_ms", "solve_ms", "step_ms"))

    # e2e GBA: the host-buffer C-ABI call a user makes (flatten → H2D → symbolic → iterations → D2H)
    e2e_iters = args.steps
    e2e_runs = []
    for rep in range(4):   # the whole call (create → iterate → read back) is repeated: one untimed warm-up call (first-use costs
        barrier()          # of the allocator / IPC mappings), then three timed ones of which the median is reported
        t0 = time.perf_counter()
        s2 = O.BaSolver(ctx, prob, visual_only=False, rank=rank, world=world, allreduce=O.torch_allreduce() if world > 1 else None)
        t1 = time.perf_counter()
        done = s2.iterate(e2e_iters)
        t2 = time.perf_counter()
        r2 = s2.result()   # noqa: F841  (the D2H read-back is part of the call)
        ctx.sync()
        dt_call = max_over_ranks(time.perf_counter() - t0)
        if rep > 0:
            e2e_runs.append((dt_call, done))
        if os.environ.get("COVINS_BENCH_VERBOSE") and rank == 0:
            print(f"[e2e] create {1e3*(t1-t0):.1f} ms, iterate {1e3*(t2-t1):.1f} ms, result {1e3*(time.perf_counter()-t2):.1f} ms", file=sys.stderr)
        s2.close()
    dt_e2e, done = sorted(e2e_runs)[1]
    h2d_gba = sum(np.asarray(v).nbytes for k, v in prob.items() if isinstance(v, np.ndarray) and not k.startswith("gt_"))
    d2h_gba = (7 + 9) * 8 * prob["K"] + 24 * prob["L"]

    # PGO leg (SURVEY §8d: "same for PGO"): Optimization::PoseGraphOptimization on the same map — poses only, loop +
    # successor + 5-predecessor between-factors built by the host logic of optimization_be.cpp:886-1021, Cauchy(0.5) on
    # the loop edges; replicas only (12k dofs, DESIGN §6).  Iterations counted as for the GBA.
    pgo = None
    if rank == 0:
        edges = O.pgo_edges(prob, prob["pose"])
        pp = dict(K=prob["K"], L=0, pose=prob["pose"], pose_const=prob["pose_const"], extr=prob["extr"], cam_of_kf=prob.get("cam_of_kf"))
        ps = O.BaSolver(ctx, pp, visual_only=True, cauchy_reproj=0.0, cauchy_edge=0.5, edges=edges)

        def pgo_iters(n):
            done_ = 0
            while done_ < n:
                k_ = ps.iterate(n - done_)
                done_ += k_
                if done_ < n:
                    ps.restart()
            return done_
        pgo_steps = args.steps
        pgo_iters(args.warmup); ps.restart()
        ctx.sync(); lp = ctx.launch_count(); t0 = time.perf_counter()
        pgo_iters(pgo_steps)
        ctx.sync(); dt_pgo = time.perf_counter() - t0
        rp = ps.result(); ps.close()
        n_e = int(len(edges["i"]))
        pgo_bytes = (2 * 56 + 48 * 8) * n_e + 288 * (prob["K"] + n_e)          # SURVEY §8d: per-iteration algorithmic bytes
        pgo = {"metric": "pgo_iterations_per_sec", "value": pgo_steps / dt_pgo, "unit": "iterations/s", "ms_per_step": dt_pgo / pgo_steps * 1e3,
               "steps": pgo_steps, "gpu_launches": int(ctx.launch_count() - lp), "dtype": "f64",
               "config": {"workload": "PoseGraphOptimization on the same map: poses only (6K dofs), loop + successor + predecessor between-factors",
                          "K": int(prob["K"]), "n_edges": n_e, "n_loop": int(edges["robust"].sum())},
               "initial_cost": rp["initial_cost"], "final_cost": rp["final_cost"],
               "roofline": {"bound": "hbm", "achieved": pgo_bytes / (dt_pgo / pgo_steps) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": pgo_bytes / (dt_pgo / pgo_steps) / 1e9 / hbm_peak, "traffic": None,
                            "note": "latency-bound: a 12k-dof block-banded system factored as dependent tile columns; the roofline "
                                    "says how far from bandwidth-bound this leg is"}}
        if world == 1 and not os.environ.get("COVINS_SKIP_CPU_BASELINE"):
            pgo["cpu_baseline"] = cpu_pgo(prob, edges, 10)
    # roofline of the dominant GBA kernel: syrk_kernel (FP64 DMMA trailing update of the tile-sparse Cholesky)
    dgemm_peak = fp64_gemm_peak(dev) if rank == 0 else 0.0
    # factor_flops = tile-GEMM flops THIS rank executed; world > 1: the work is split by tile columns
    chol_tflops = tm["factor_flops"] / (tm["factor_ms"] * 1e-3) / 1e12 if tm["factor_ms"] > 0 else 0.0

    # =============================================================================================
    # leg 2: matching (weak scaling: every rank holds a C3-sized shard of keyframes; no data-path collective)
    # =============================================================================================
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    # ORB-like keyframes with shared landmarks (synth.orb_keyframes: matched Hamming ~16, unmatched ~128), so the ratio test
    # accepts real matches and the compaction / D2H of accepted matches is exercised; copy c = the map with its keyframes rotated
    base_desc, _ = synth.orb_keyframes(seed=3 + rank, n_kf=N_KF, n_feat=N_FEAT)
    h_base = np.ascontiguousarray(base_desc.reshape(N_KF * N_FEAT, 32))
    d_base = torch.from_numpy(h_base).to(dev)
    maps = [d_base] + [torch.roll(d_base.view(N_KF, N_FEAT, 32), 97 * c, 0).reshape(-1, 32).contiguous() for c in range(1, N_COPIES)]
    q = maps[0][123 * N_FEAT:124 * N_FEAT].clone()
    h_seg = synth.seg_ptr_uniform(N_KF, N_FEAT)
    d_seg = torch.from_numpy(h_seg).to(dev)
    pairs = N_KF * N_FEAT * N_FEAT

    # the map databases: keyframes appended once (outside every timed region, as in the server's life cycle: a keyframe's
    # descriptors never change), which also writes their tensor-core operand tiles; requests read only resident data
    h_maps_np = [m.cpu().pin_memory().numpy() for m in maps[:2]]
    dbs = []
    for c in range(N_COPIES):
        db = M.DescriptorDatabase(ctx, reserve_rows=N_KF * N_FEAT)
        db.append(h_maps_np[c] if c < 2 else maps[c].cpu().numpy(), np.full(N_KF, N_FEAT, np.int32))
        dbs.append(db)

    def step_match(i):          # device request against the resident map (cvb_db_match_hamming_dev)
        return dbs[i % N_COPIES].match_hamming_dev(q, THR, RATIO)

    def step_match_raw(i):      # raw-pointer API: packed rows only, the operand tiles are expanded inside every call
        return M.match_candidates_hamming(ctx, q, maps[i % N_COPIES], (d_seg, h_seg), THR, RATIO)

    m_steps = args.steps
    for i in range(args.warmup):
        step_match(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count()
    e0.record()
    for i in range(m_steps):
        out_m = step_match(i)
    e1.record()
    barrier()
    ms_match = max_over_ranks(e0.elapsed_time(e1))
    match_launches = ctx.launch_count() - l0
    n_accepted = int(out_m[2].sum().item())
    gp = pairs * world * m_steps / (ms_match * 1e-3) / 1e9

    for i in range(3):
        step_match_raw(i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(10):
        step_match_raw(i)
    e1.record(); torch.cuda.synchronize()
    ms_raw = e0.elapsed_time(e1) / 10

    h_q = q.cpu().pin_memory().numpy()
    e2e_steps = args.steps
    for i in range(2):
        M.match_candidates_hamming(ctx, h_q, h_maps_np[i % 2], h_seg, THR, RATIO)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        M.match_candidates_hamming(ctx, h_q, h_maps_np[i % 2], h_seg, THR, RATIO)
    barrier()
    dt = max_over_ranks(time.perf_counter() - t0)
    e2e_gp = pairs * world * e2e_steps / dt / 1e9
    # e2e through the resident-map API (cvb_db_*): keyframes uploaded once when they join the map (outside the timed
    # region, as in the server's life cycle), per request the query keyframe goes up and the accepted matches come down.
    h_queries = [np.ascontiguousarray(h_maps_np[0][k * N_FEAT:(k + 1) * N_FEAT]) for k in (123, 777, 1500, 42)]
    db_steps = args.steps
    d2h_db = 0
    for i in range(3):
        dbs[i % N_COPIES].match_hamming(h_queries[i % 4], THR, RATIO)
    barrier()
    step_s = []
    t0 = time.perf_counter()
    for i in range(db_steps):
        ts = time.perf_counter()
        out = dbs[i % N_COPIES].match_hamming(h_queries[i % 4], THR, RATIO)   # returns after the D2H of the matches
        step_s.append(time.perf_counter() - ts)
        d2h_db += out[0].nbytes + 4 + sum(o.nbytes for o in out[1:])
    barrier()
    dt_db_mean = max_over_ranks(time.perf_counter() - t0) / db_steps
    dt_db = max_over_ranks(float(np.median(step_s)))      # per-request median: robust against host scheduling noise
    e2e_db_gp = pairs * world / dt_db / 1e9
    for db in dbs:
        db.close()
    alg_bytes = 32 * N_KF * N_FEAT + 32 * N_FEAT + 8 * N_KF * N_FEAT + 4 * N_KF   # SURVEY §8d: 32 Nt + 32 Nq + outputs
    ms_step = ms_match / m_steps
    hbm_gbs = alg_bytes / (ms_step * 1e-3) / 1e9
    # dominant kernel: cvb_tc::xt::tc_xt_kernel<2> — u8 x s8 -> s32 tcgen05 GEMM over the resident operand tiles (K = 256 bit
    # bytes + a 32-byte key slice that makes the accumulator the sort key) + fused top-2 / ratio filter.  Algorithmic ops:
    # 2 x 256 per pair (SURVEY 8d); the key slice's 12.5 % extra MMA work is not counted.
    tops = 2.0 * 256 * pairs / (ms_step * 1e-3) / 1e12
    tile_bytes_per_launch = ((N_FEAT + 127) // 128) * N_KF * 128 * 288
    i8_peak, i8_src = int8_gemm_peak(dev) if rank == 0 else (1.0, "")
    # the scalar POPC kernel (previous formulation, still used for small / DenseMatcher shapes) for comparison
    os.environ["COVINS_B200_MATCH_KERNEL"] = "popc"
    for i in range(2):
        step_match_raw(i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(5):
        step_match_raw(i)
    e1.record(); torch.cuda.synchronize()
    ms_popc = e0.elapsed_time(e1) / 5
    os.environ.pop("COVINS_B200_MATCH_KERNEL", None)
    popc_peak = M.microbench_popc(ctx, 20000) if rank == 0 else 0.0
    # SIFT / L2 leg (C5 shard: 300-feature query vs 10000 KF x 300 x 128-d u8), extra information
    sift = None
    if rank == 0:
        n_kf5, nf5 = 10000, 300
        ts = torch.randint(0, 256, (n_kf5 * nf5, 128), dtype=torch.uint8, device=dev, generator=g)
        qs = ts[:nf5].clone(); hs = synth.seg_ptr_uniform(n_kf5, nf5); ds = torch.from_numpy(hs).to(dev)
        for _ in range(3):
            M.knn_match_l2(ctx, qs, ts, (ds, hs), 2)
        torch.cuda.synchronize(); e0.record()
        for _ in range(5):
            M.knn_match_l2(ctx, qs, ts, (ds, hs), 2)
        e1.record(); torch.cuda.synchronize()
        ms_l2 = e0.elapsed_time(e1) / 5
        l2_tops = 2.0 * 128 * n_kf5 * nf5 * nf5 / (ms_l2 * 1e-3) / 1e12
        sift = {"metric": "match_l2_gpairs_per_sec", "value": n_kf5 * nf5 * nf5 / (ms_l2 * 1e-3) / 1e9, "unit": "Gpairs/s",
                "ms_per_step": ms_l2, "config": "C5 shard: 300 SIFT queries vs 10000 KF x 300 rows x 128-d u8 (384 MB), k=2, exact brute force",
                "roofline": {"bound": "tensor", "achieved": l2_tops, "peak": i8_peak, "unit": "TOP/s", "frac": l2_tops / i8_peak, "traffic": None,
                             "peak_source": i8_src}}
        if world == 1 and not os.environ.get("COVINS_SKIP_CPU_BASELINE"):
            sift["cpu_baseline"] = cpu_sift_port()
        del ts
    # Landmark::ComputeDescriptor batched over the C3 map's landmarks (SURVEY §8a M7): 100k landmarks x 8 observers
    lmdesc = None
    if rank == 0:
        n_lm7, per7 = 100_000, 8
        c7 = torch.randint(0, 256, (n_lm7 * per7, 32), dtype=torch.uint8, device=dev, generator=g)
        p7 = torch.arange(0, n_lm7 * per7 + 1, per7, dtype=torch.int32, device=dev)
        for _ in range(3):
            M.landmark_descriptors(ctx, c7, p7)
        torch.cuda.synchronize(); e0.record()
        for _ in range(10):
            M.landmark_descriptors(ctx, c7, p7)
        e1.record(); torch.cuda.synchronize()
        ms7 = e0.elapsed_time(e1) / 10
        b7 = n_lm7 * per7 * 32 + n_lm7 * 36 + (n_lm7 + 1) * 4
        lmdesc = {"metric": "landmark_descriptors_per_sec", "value": n_lm7 / (ms7 * 1e-3), "unit": "landmarks/s", "ms_per_step": ms7,
                  "config": "Landmark::ComputeDescriptor for 100000 landmarks x 8 observers (25.6 MB of descriptors), one launch",
                  "roofline": {"bound": "hbm", "achieved": b7 / (ms7 * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                               "frac": b7 / (ms7 * 1e-3) / 1e9 / hbm_peak, "traffic": None, "algorithmic_bytes_per_launch": b7,
                               "note": "32 B per observation read once + 36 B per landmark written; includes the clone of the old descriptors"}}
        del c7
    tr_match, tr_match_src = _traffic("tc_xt_kernel")
    match = {
        "metric": "match_gpairs_per_sec", "value": gp, "unit": "Gpairs/s", "ms_per_step": ms_step, "steps": m_steps,
        "scaling": "weak", "dtype": "u8",
        "config": {"workload": "fused k-NN(k=2)+ratio filter of one 1000-feature ORB query KF against the 2000 KFs x 1000 "
                               "features of the rank's map shard, resident in HBM as packed rows + tensor-core operand tiles "
                               "(cvb_db_match_hamming_dev: device query in, dense device results out)",
                   "data": "synth.orb_keyframes: keyframes share landmarks (matched Hamming ~16, unmatched ~128)",
                   "accepted_matches_per_step": n_accepted,
                   "pairs_per_step_per_gpu": pairs,
                   "l2_policy": f"{N_COPIES} map copies (256 MB > 126 MB L2) rotated per step",
                   "parallelism": f"map sharded by keyframe x{world}, no data-path collective"},
        "e2e": {"value": e2e_db_gp, "unit": "Gpairs/s", "h2d_bytes_per_step": int(h_queries[0].nbytes),
                "d2h_bytes_per_step": int(d2h_db // db_steps), "steps": db_steps, "ms_per_step": dt_db * 1e3,
                "mean_ms_per_step": dt_db_mean * 1e3, "timing": "median over the requests of the wall time of one complete call (each call returns after its D2H)",
                "api": "cvb_db_match_hamming: host query in, per-keyframe match counts + compacted accepted matches out; the "
                       "map's descriptors were appended once with cvb_db_append (outside the timed region) and stay in HBM; "
                       f"{N_COPIES} databases (256 MB > L2) rotated per step",
                "upload_every_call": {"value": e2e_gp, "unit": "Gpairs/s",
                                      "h2d_bytes_per_step": int(h_q.nbytes + h_maps_np[0].nbytes + h_seg.nbytes),
                                      "d2h_bytes_per_step": N_KF * N_FEAT * 8 + N_KF * 4, "steps": e2e_steps,
                                      "api": "cvb_match_hamming_batch: the whole 64 MB map re-uploaded from host memory on "
                                             "every call and the dense [n_kf][nq] result matrices downloaded (PCIe-bound)"}},
        "gpu_launches": int(match_launches),
        "roofline": {"bound": "tensor", "achieved": tops, "peak": i8_peak, "unit": "TOP/s", "frac": tops / i8_peak, "traffic": tr_match,
                     "traffic_source": tr_match_src, "peak_source": i8_src,
                     "kernel": "cvb_tc::xt::tc_xt_kernel<2> (tcgen05.mma kind::i8 u8 x s8, query block in TMEM, operand tiles by cp.async.bulk, "
                               "accumulator = packed sort key, fused top-2 + ratio filter)",
                     "hw_peak": {"tops": 2 * 8192 * 148 * 1.965e9 / 1e12, "frac": tops / (2 * 8192 * 148 * 1.965e9 / 1e12),
                                 "source": "8192 MAC/clk/SM measured with tools/micro/umma_rate.cu (profiles/r02_umma_rate.txt) x 148 SMs x 1965 MHz"},
                     "operand_tile_bytes_per_launch": tile_bytes_per_launch,
                     "raw_pointer_api": {"ms_per_step": ms_raw, "gpairs_per_s": pairs / (ms_raw * 1e-3) / 1e9,
                                         "note": "cvb_match_hamming_batch_dev on packed rows only: the 590 MB of operand tiles are expanded inside "
                                                 "every call (HBM-bound pre-pass) before the same kernel runs"},
                     "hbm": {"achieved_gbs": hbm_gbs, "peak_gbs": hbm_peak, "frac": hbm_gbs / hbm_peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes},
                     "scalar_popc_kernel": {"ms_per_step": ms_popc, "gpairs_per_s": pairs / (ms_popc * 1e-3) / 1e9,
                                            "int_pipe_frac": (8 * pairs / (ms_popc * 1e-3) / 1e9) / popc_peak if popc_peak else None,
                                            "peak_gpopc_s": popc_peak}},
        "sift_l2": sift,
        "landmark_descriptor": lmdesc,
    }

    tr_gba, tr_gba_src = _traffic("syrk_kernel")
    line = {
        "metric": "gba_iterations_per_sec", "value": gba_rate, "unit": "iterations/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt_gba / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "gba_config": args.gba_config, "K": int(prob["K"]), "L": int(prob["L"]), "n_obs": int(n_obs),
                   "n_imu": int(len(prob["imu_i"])), "n_loop": int(len(prob["loop_i"])), "reduced_system_dim": int(15 * prob["K"]),
                   "l2_policy": "working set (0.8 GB of packed tiles of the reduced camera system + 0.5 GB of observation records at C3) >> 126 MB L2",
                   "parallelism": (f"landmark blocks sharded x{world}; reduced camera system reduce-scattered by peer pull (CUDA IPC over NVLink) onto "
                                   f"tile-column owners; Cholesky distributed by tile columns, panels handed over through peer memory; small vectors all-reduced (NCCL)"
                                   if p2p else f"landmark blocks sharded x{world}; all-reduce of the reduced normal equations; solve replicated") if world > 1 else "single GPU",
                   "peer_path": p2p,
                   "iteration_counting": "trust-region iterations as Ceres counts them (accepted + rejected); the timed region starts at the "
                                         "initial state; a solve that converges inside it is restarted from the initial state (cvb_ba_restart)",
                   "map_generation_s": round(t_gen, 1)},
        "e2e": {"value": done / dt_e2e, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d_gba // max(done, 1)),
                "d2h_bytes_per_step": int(d2h_gba // max(done, 1)), "steps": int(done),
                "runs_s": [round(r[0], 4) for r in e2e_runs],
                "note": "cvb_ba_create + iterate + result_get on host buffers: flatten/H2D/symbolic setup and the D2H read are inside; median of 3 complete calls after one warm-up call"},
        "gpu_launches": int(gba_launches),
        "clocks": clk.summary(),
        "phase_ms_per_step": {k: round(v / args.steps, 3) for k, v in tm.items() if k.endswith("_ms")},
        "device_ms_per_step": dev_ms / args.steps,
        "final_cost": res["final_cost"], "initial_cost": res["initial_cost"],
        "roofline": {"bound": "tensor", "achieved": chol_tflops, "peak": dgemm_peak, "unit": "TFLOP/s",
                     "frac": chol_tflops / dgemm_peak if dgemm_peak else None, "traffic": tr_gba, "traffic_source": tr_gba_src,
                     "peak_source": "cuBLAS DGEMM 6144^3 measured in this run (FP64; MEASURED_PEAKS.json holds no FP64 figure)",
                     "kernel": "cvb_chol::syrk_kernel (FP64 DMMA m8n8k4, 64x64x128 per CTA, 3 CTAs/SM) inside the tile-sparse Cholesky of the reduced camera system; "
                               "achieved = tile-GEMM flops executed by rank 0 / factorisation time (includes the latency-bound diagonal-tile chain)",
                     "flops_per_factorisation_dense_equivalent": (15.0 * prob["K"]) ** 3 / 3.0},
        "match": match,
        "pgo": pgo,
        # scalars of the nested legs at the top level (per-N scaling records keep them)
        "match_gpairs_per_sec": gp, "match_e2e_gpairs_per_sec": e2e_db_gp,
        "pgo_iterations_per_sec": pgo["value"] if pgo else None,
        "sift_l2_gpairs_per_sec": sift["value"] if sift else None,
        "gba_e2e_iterations_per_sec": done / dt_e2e,
    }
    if rank == 0:
        if world == 1 and not os.environ.get("COVINS_SKIP_CPU_BASELINE"):
            # bounded sample of the same workload on the host cores (the full same-steps run is `--impl reference`)
            line["cpu_baseline"], _ = cpu_gba(args.gba_config, 4)
            line["match"]["cpu_baseline"] = cpu_match_port()
        if args.dump_outputs:
            # the result of the last timed step of each leg, as its caller receives it
            dump_outputs(args.dump_outputs, {
                "gba_pose": res["pose"], "gba_speedbias": res["speedbias"], "gba_landmarks": res["lm"],
                "gba_landmark_owner": res["lm_owner"], "gba_cost_history": res["cost"],
                "pgo_pose": rp["pose"], "pgo_cost_history": rp["cost"],
                "match_train": out_m[0], "match_dist": out_m[1], "match_count": out_m[2]})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gba-config", default=os.environ.get("COVINS_GBA_CONFIG", "C3"))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step of each leg computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
