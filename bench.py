#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched ENLSIP engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA engine)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm (compiled port of the oracle)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + outputs of the last timed step, as DIR/*.npy

Workload (config.workload): BASELINE.json config 3 -- batched bound + equality constrained
Gaussian-peak curve fits, n=6, m=128, 1 equality + 12 bounds, forward-difference Jacobians,
B problems per GPU (4M at the named size), synthetic data of SURVEY.md section 8d (seed 128).
A "step" is one complete solve of the whole batch.  `value` times the solve with inputs already
resident in HBM; `e2e` times the C-ABI call with pinned HOST buffers (H2D of y, S, x0 and D2H of
x, f, exit codes, iteration counts inside the timed region).  Multi-GPU: the batch is sharded, one
process per GPU, no collective on the solve path (weak scaling: B problems per GPU).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "batched CNLS solves/s (n=6,m=128)"      # first half of BASELINE.json's metric; the second half (GN iters/s,
                                                  # m=4M, n=256) is the "large" object of the same JSON line
UNIT = "solves/s"
ALG_BYTES_PER_SOLVE = 128 * 8 + 48 + 8 + 48 + 8 + 12   # SURVEY.md 8d: y, x0, S in; x, f, (exit, iters, t) out = 1148 B
NCU_DRAM_BYTES_PER_SOLVE = (33.66e6 + 901.2e6) / 30000  # dram__bytes_read + dram__bytes_write of one ncu --set full capture
ALG_FLOP_PER_SOLVE = 2.0e5 * 6.12                       # SURVEY.md 8d estimate per iteration x mean iterations of the stream


def fp64_fma_peak():
    p = os.path.join(ROOT, "profiles", "r1_fp64_peaks.json")
    if os.path.exists(p):
        return float(json.load(open(p))["fp64_dfma_tflops"])
    return 40.0


def sample_rows(B, k, seed=0):
    """--dump-outputs: a fixed, seeded sample of k of the B problems of a batch (all of them when B <= k), sorted."""
    if B <= k:
        return np.arange(B)
    return np.sort(np.random.default_rng(seed).choice(B, k, replace=False))


def write_outputs(dirname, prefix, arrays, rows=None):
    """--dump-outputs: the arrays a caller of a timed path receives after its last step, as DIR/<prefix><name>.npy in
    float64 (the integer outputs are exact in it), so that two builds can be compared output for output.  `rows` keeps
    those problems of a batched output and is written as <prefix>index.npy."""
    os.makedirs(dirname, exist_ok=True)
    if rows is not None:
        np.save(os.path.join(dirname, prefix + "index.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        if rows is not None:
            a = a[rows]
        np.save(os.path.join(dirname, prefix + name + ".npy"), a.astype(np.float64))


def large_outputs(mod):
    """What solve() hands the caller of one large-regime problem."""
    return {"x": mod.sol[0], "f": mod.obj_value, "exit_code": mod.exit_code, "status": mod.status_code,
            "iters": mod.iterations, "nact": mod.nb_active, "active": mod.active[0]}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            p = [s.strip() for s in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_port(B, nthreads, seed_start=0):
    """Compiled scalar port of the solver core (oracle/hostport) on the host cores: solves/s."""
    import ctypes
    import math
    import __graft_entry__ as ge
    import enlsip_jl_b200 as E
    lib = ctypes.CDLL(ge.build_hostport())
    # every `qr(., ColumnNorm())` of the solve runs in OpenBLAS' dgeqp3 (the routine Julia calls), not in the engine's
    # restatement of it (oracle/hostport/hostport.cpp: hostport_use_lapack)
    lib.hostport_use_lapack.argtypes = [ctypes.c_char_p]
    blas = ge.openblas_path()
    cpu_port.lapack = bool(blas) and lib.hostport_use_lapack(blas.encode()) == 0

    class Opt(ctypes.Structure):
        _fields_ = [("max_iter", ctypes.c_int), ("scaling", ctypes.c_int), ("jac_mode", ctypes.c_int),
                    ("second_derivatives", ctypes.c_int), ("time_limit", ctypes.c_double), ("eps_abs", ctypes.c_double),
                    ("eps_rel", ctypes.c_double), ("eps_x", ctypes.c_double), ("eps_c", ctypes.c_double),
                    ("eps_rank", ctypes.c_double)]

    se = math.sqrt(np.finfo(float).eps)
    opt = Opt(100, 0, 1, 1, 1e3, 1e-10, se, se, se, se)
    y, S, x0, _ = E.synth.gen_gauss_peaks_batch(B, start=seed_start)
    n, lmax = 6, 13
    x = np.zeros((B, n)); f = np.zeros(B)
    ints = [np.zeros(B, np.int32) for _ in range(4)]
    act = np.zeros((B, lmax), np.int32); cnt = np.zeros((B, 2), np.int32)
    vp = ctypes.c_void_p
    lib.hostport_solve.argtypes = [ctypes.c_int, ctypes.c_longlong] + [vp] * 5 + [ctypes.POINTER(Opt)] + [vp] * 9 + \
                                  [ctypes.c_int, ctypes.c_int]
    p = lambda a: a.ctypes.data_as(vp)
    lo, up = np.ascontiguousarray(E.synth.GP_LOW), np.ascontiguousarray(E.synth.GP_UPP)
    y = np.ascontiguousarray(y)

    def run():
        t0 = time.perf_counter()
        lib.hostport_solve(1, B, p(x0), p(y), p(S), p(lo), p(up), ctypes.byref(opt), p(x), p(f), p(ints[0]), p(ints[1]),
                           p(ints[2]), p(ints[3]), p(act), p(cnt), None, 0, nthreads)
        return time.perf_counter() - t0

    return run, ints[2]


# =================================================================================================
# large-Jacobian regime (BASELINE.json config 4): GN iterations/s at m = 4M, n = 256, 64 equalities
# =================================================================================================
LARGE_METRIC = "GN iters/s (m=4M,n=256)"
NCU_TRAIL_DRAM_BYTES_PER_ROW_COL = (2.248e9 + 1.829e9) / (1048576 * 224.0)   # profiles/r1_c4_trail_staged_v0_ncu.txt
LARGE_N, LARGE_NB = 256, 64


def fp64_tensor_peak():
    """Measured FP64 DMMA peak of this pool's B200s (tools/fp64_peaks.cu; MEASURED_PEAKS.json has no FP64 entry)."""
    p = os.path.join(ROOT, "profiles", "r1_fp64_peaks.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["fp64_dmma_m8n8k4_tflops"]), "measured mma.sync.m8n8k4.f64 peak (tools/fp64_peaks.cu, profiles/r1_fp64_peaks.json)"
    return 40.0, "fallback: B200 FP64 tensor datasheet figure"


def gen_large_shard(torch, dev, m_global, row0, rows, n=LARGE_N, nb=LARGE_NB):
    """Rows [row0, row0 + rows) of the C4 problem of SURVEY.md 8d: synth.gen_single_index(m, 256, 64, seed=4), the very
    data of tests/golden/c4_2p22_oracle.npz (row chunks own their generator seed, so every world size sees the same
    global W and y).  Generated on the host, then moved to the device."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(m_global, n, nb, seed=4, start=row0, rows=rows)
    W = torch.from_numpy(d["W"]).to(dev)
    y = torch.from_numpy(d["y"]).to(dev)
    return W, y, d["x0"], d["rho"]


def c5_flops(n, m, t):
    """Dense FP64 flops of one Gauss-Newton iteration of the reference's own math (SURVEY.md 8d, C5 row):
    qr(A_act') 2nt^2 - 2/3 t^3, J*Q1 4mnt, qr(J2) 2mk^2 - 2/3 k^3 with k = n - t."""
    k = n - t
    return 2.0 * n * t * t - 2.0 / 3.0 * t ** 3 + 4.0 * m * n * t + 2.0 * m * k * k - 2.0 / 3.0 * k ** 3


def large_cpu_reference(n, m_rows, nb, seed, ineq, bounds, cores):
    """One Gauss-Newton iteration of the reference's dense algorithm on the host cores (oracle/hostport/largeport.cpp
    largeport_ref_iteration): new_point!, dgeqp3 of A_act', dormqr J*Q1 on the full m x n Jacobian, dgeqp3 of J2,
    triangular solves -- the LAPACK routines Julia calls, from the SciPy wheel's OpenBLAS, all threads.
    Returns (seconds, t, phase seconds) or None when the library cannot be bound."""
    import ctypes
    import __graft_entry__ as ge
    import enlsip_jl_b200 as E
    blas = ge.openblas_path()
    if not blas:
        return None
    lib = ctypes.CDLL(ge.build_largeport())
    vp = ctypes.c_void_p
    lib.largeport_ref_iteration.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                            vp, vp, vp, vp, vp, vp, ctypes.c_int, vp, vp, vp]
    d = E.synth.gen_single_index(m_rows, n, nb, seed=seed, ineq=ineq)
    lo = None if bounds is None else np.full(n, float(bounds[0]))
    up = None if bounds is None else np.full(n, float(bounds[1]))
    secs = np.zeros(5); pdir = np.zeros(n); t = ctypes.c_int(0)
    pp = lambda a: None if a is None else a.ctypes.data_as(vp)
    rc = lib.largeport_ref_iteration(blas.encode(), n, m_rows, nb, 1 if ineq else 0, pp(lo), pp(up), pp(d["W"]), pp(d["y"]),
                                     pp(d["rho"]), pp(d["x0"]), cores, pp(secs), pp(pdir), ctypes.byref(t))
    if rc != 0:
        return None
    return float(secs[0]), int(t.value), [float(v) for v in secs]


def large_cpu_baseline(sample_rows, m_global, passes_per_iteration=4.0 / 3.0):
    """C4 on the host cores: the reference's algorithm with OpenBLAS LAPACK on `sample_rows` of the m_global rows (the
    whole problem when sample_rows == m_global).  Every dense step of an iteration is linear in m, so
    seconds(m_global) = seconds(sample) * m_global / sample_rows.  `passes_per_iteration`: a solve that reports k
    iterations executes k + 1 passes of the loop (EF:2776-2878; the last one terminates) -- 4 passes for the 3 reported
    iterations of this problem, the same accounting as the GPU arm."""
    cores = os.cpu_count() or 1
    got = large_cpu_reference(LARGE_N, sample_rows, LARGE_NB, 4, False, None, cores)
    if got is None:
        return {"value": None, "unit": "iters/s", "cores": cores, "kind": "reference-algorithm", "sample": "OpenBLAS could not be bound"}
    secs, t, ph = got
    per_pass = secs * m_global / sample_rows
    v = 1.0 / (per_pass * passes_per_iteration)
    return {"value": v, "unit": "iters/s", "cores": cores, "kind": "port",
            "sample": "%d of the %d rows (n=256, 64 equalities): one pass of the reference's dense iteration "
                      "(new_point! %.2f s, dgeqp3(A') + dormqr J*Q1 %.2f s, dgeqp3(J2) %.2f s, solves %.2f s) with OpenBLAS "
                      "LAPACK on all cores, scaled linearly to %d rows, %.3g passes per reported iteration; C++ restatement "
                      "(oracle/hostport/largeport.cpp) -- Julia itself is absent from this image"
                      % (sample_rows, m_global, ph[1], ph[2], ph[3], ph[4], m_global, passes_per_iteration)}


C5_N, C5_M, C5_NB = 4096, 16384, 1024
C5_METRIC = "GN iters/s (n=4096,m=16384)"


def c5_cpu_baseline(scale=2, passes_per_iteration=8.0 / 7.0, t_full=511):
    """C5 on the host cores: the same reference-algorithm pass on the problem shrunk by `scale` in every dimension
    (one problem cannot be row-sampled without changing its shape), scaled by the algorithmic flop ratio."""
    cores = os.cpu_count() or 1
    n, m, nb = C5_N // scale, C5_M // scale, C5_NB // scale
    got = large_cpu_reference(n, m, nb, 5, True, (-2.0, 2.0), cores)
    if got is None:
        return {"value": None, "unit": "iters/s", "cores": cores, "kind": "reference-algorithm", "sample": "OpenBLAS could not be bound"}
    secs, t, ph = got
    ratio = c5_flops(C5_N, C5_M, t_full) / c5_flops(n, m, t)
    per_pass = secs * ratio
    return {"value": 1.0 / (per_pass * passes_per_iteration), "unit": "iters/s", "cores": cores, "kind": "port",
            "sample": "the C5 family at n=%d, m=%d, %d inequalities + bounds (t = %d active): one pass of the reference's dense "
                      "iteration with OpenBLAS LAPACK on all cores in %.2f s (new_point! %.2f, dgeqp3(A') + dormqr J*Q1 %.2f, "
                      "dgeqp3(J2) %.2f, solves %.2f), scaled by the flop ratio %.1f to the named size (t = %d), %.3g passes "
                      "per reported iteration" % (n, m, nb, t, secs, ph[1], ph[2], ph[3], ph[4], ratio, t_full, passes_per_iteration)}


def c2_arm(args, torch, dist, E, rank, world, local, dev):
    """BASELINE.json config 2: B instances of Hock-Schittkowski 65 (n = 3, m = 3, 1 inequality + 6 bounds, analytic
    Jacobians; test/problems/HS65.jl with perturbed starts) per GPU, one thread per problem.  Same timing rules as the
    headline: warm-up, barrier + CUDA events, max over ranks."""
    B = args.c2_problems
    x0 = torch.from_numpy(np.ascontiguousarray(E.synth.gen_hs65_batch(B, start=rank * B))).to(dev)
    mod = E.CnlsModel("hs65", x0, x_low=E.synth.HS65_LOW, x_upp=E.synth.HS65_UPP, device=local)
    out = {"x": torch.empty(B, 3, dtype=torch.float64, device=dev), "f": torch.empty(B, dtype=torch.float64, device=dev)}
    for k in ("exit_code", "status", "iters", "nact"):
        out[k] = torch.empty(B, dtype=torch.int32, device=dev)
    steps = max(3, args.steps // 4)
    for _ in range(3):
        E.solve(mod, want_active=False, want_counters=False, out=out)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = mod.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        E.solve(mod, want_active=False, want_counters=False, out=out)
    ev1.record()
    torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, "hs65_", out, sample_rows(B, 1 << 16))
    st = out["status"].cpu().numpy()
    ec = out["exit_code"].cpu().numpy()
    res = {"metric": "batched CNLS solves/s (HS65: n=3, m=3)", "value": world * B / (ms * 1e-3), "unit": "solves/s", "n_gpus": world,
           "steps": steps, "warmup": 3, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "dtype": "f64",
           "config": {"workload": "C2 HS65 n=3 m=3, 1 inequality + 6 bounds, analytic Jacobians (BASELINE.json config 2)",
                      "problems_per_gpu": B, "seed": 65, "l2": "inputs 24 B per problem: the state lives on chip, not an HBM workload"},
           "gpu_launches": int(mod.launch_count() - l0),
           "quality": {"converged_fraction": float(np.mean(st == 1)), "mean_iterations": float(out["iters"].float().mean().item()),
                       "reference_would_hang_fraction": float(np.mean(ec == -98))}}
    del mod
    return res


def c5_arm(args, torch, E, dev, local):
    """BASELINE.json config 5 (n = 4096, m = 16384, 1024 inequalities + 8192 bounds) on ONE GPU ("replicas only",
    SURVEY.md 8e): one step = one complete solve from x0."""
    d = E.synth.gen_single_index(C5_M, C5_N, C5_NB, seed=5, ineq=True)
    lo, up = np.full(C5_N, -2.0), np.full(C5_N, 2.0)
    W = torch.from_numpy(d["W"]).to(dev)
    y = torch.from_numpy(d["y"]).to(dev)
    mod = E.LargeCnlsModel("single_index", d["x0"], {"W": W, "y": y, "rho": d["rho"]}, ineq=True, x_low=lo, x_upp=up, device=local)
    for _ in range(max(1, args.large_warmup)):
        E.solve(mod, trace_cap=40)
    ts = [int(v) for v in mod.trace[0][: int(mod.iterations[0]) + 1, 1]]
    st0 = mod.stats()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    its = 0
    for _ in range(args.c5_steps):
        E.solve(mod)
        its += int(mod.iterations[0])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, "large5_", large_outputs(mod))
    st1 = mod.stats()
    dst = {k: st1[k] - st0[k] for k in st1 if k != "rows_pad"}
    nfac = max(dst["factorisations"], 1.0)
    flops_it = [c5_flops(C5_N, C5_M, t) for t in ts if t > 0]
    flops_mean = float(np.mean(flops_it)) if flops_it else c5_flops(C5_N, C5_M, 511)
    peak, peak_src = fp64_tensor_peak()
    per_pass_s = dt / max(dst["points"] - args.c5_steps, 1.0)          # passes of the loop = points evaluated - 1 per solve
    achieved = flops_mean / per_pass_s / 1e12
    res = {"metric": C5_METRIC, "value": its / dt, "unit": "iters/s", "n_gpus": 1, "steps": args.c5_steps,
           "warmup": max(1, args.large_warmup), "scaling": "replicas only (SURVEY.md 8e)", "higher_is_better": True, "dtype": "f64",
           "ms_per_iteration": dt * 1e3 / max(its, 1), "iterations_reported_by_solver_per_solve": its / args.c5_steps,
           "passes_of_the_loop_per_solve": (dst["points"] - args.c5_steps) / args.c5_steps,
           "working_set_sizes": ts, "exit_code": int(mod.exit_code[0]), "objective": float(mod.obj_value[0]),
           "config": {"workload": "C5 single-index n=4096 m=16384, 1024 inequalities + 8192 bounds (BASELINE.json config 5)",
                      "l2": "W is 0.54 GB, [J | r] 0.54 GB, the compressed problem 0.13 GB: larger than L2"},
           "phases_ms_per_pass": {"build_J_r_grad": dst["build_ms"] / max(dst["points"], 1.0), "tsqr": dst["tsqr_ms"] / nfac,
                                  "small_stage_device": dst["small_stage_ms"] / nfac,
                                  "host_other": (dst["solve_wall_ms"] - dst["build_ms"] - dst["tsqr_ms"] - dst["small_stage_ms"]
                                                 - dst["linesearch_ms"]) / nfac},
           "device_qrcp_per_solve": dst["device_qrcp"] / args.c5_steps, "gpu_launches": int(dst["launches"]),
           "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                        "traffic": None, "peak_source": peak_src,
                        "kernel": "one pass of the iteration: TSQR of [J | r] (tsqr_*), blocked QRCP of A_act', R_A' and J2 "
                                  "(qr_panel_persist_kernel: one cooperative kernel per dlaqps panel, + rank-32 trailing update), "
                                  "compact-WY J~ Q1 (gemm_dmma_*), cooperative WY vector products and triangular solves",
                        "algorithmic_flops_per_pass": flops_mean,
                        "note": "algorithmic flops of the REFERENCE's math per pass (SURVEY.md 8d formula at the measured working-set "
                                "sizes) / wall time of a pass; the engine itself executes fewer flops (it pivots on the compressed "
                                "(n+1) x (n+1) problem), and the pivoted panels are BLAS-2 (L2-bandwidth bound) by nature"}}
    # the dominant kernel family of a pass, timed alone: the blocked pivoted QR of a J2-sized matrix (4097 x 3587) through the
    # known-answer hook (CUDA events around its kernels).  Its BLAS-2 half reads the trailing matrix once per column:
    # algorithmic bytes = sum over the blocked columns k of 8 (rows - k) (cols - k - 1).
    try:
        import ctypes
        rows_q, cols_q = C5_N + 1, C5_N - 509
        Aq = np.asfortranarray(np.random.default_rng(1).standard_normal((rows_q, cols_q)))
        tq = np.zeros(min(rows_q, cols_q)); jq = np.zeros(cols_q, np.int32)
        L = E.capi.lib()
        vp = ctypes.c_void_p
        best = None
        for _ in range(2):
            f = Aq.copy(order="F")
            E.capi.check_large(L.enlsipb200_dense_qrcp(rows_q, cols_q, f.ctypes.data_as(vp), tq.ctypes.data_as(vp), jq.ctypes.data_as(vp), local))
            ms = float(L.enlsipb200_dense_last_ms())
            best = ms if best is None else min(best, ms)
        kb = min(rows_q, cols_q) - 128
        kk = np.arange(kb, dtype=np.float64)
        qbytes = float(np.sum(8.0 * (rows_q - kk) * (cols_q - kk - 1)))
        hbm_peak, hbm_src = measured_peaks()
        res["roofline_qrcp"] = {"bound": "hbm", "achieved": qbytes / (best * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                "frac": qbytes / (best * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "traffic": None,
                                "kernel": "qrcp_device on %d x %d (qr_panel_persist_kernel: one cooperative kernel per dlaqps panel, "
                                          "two grid barriers per pivoted column; rank-32 trailing updates; dlaqp2 tail)" % (rows_q, cols_q),
                                "kernel_ms": best, "algorithmic_bytes": qbytes,
                                "note": "whole factorisation: the trailing matrix streamed once per blocked column (dlaqps is BLAS-2 by "
                                        "construction); per column about half of the time is that streaming pass, the rest the "
                                        "latency chain pivot -> column -> norm -> F column across two grid barriers "
                                        "(profiles/r2_qr_panel_persist_phases.txt)"}
    except Exception as ex:       # measurement aid only
        res["roofline_qrcp"] = {"error": str(ex)}
    if args.large_e2e_steps > 0:
        W_h = torch.from_numpy(d["W"]).pin_memory()
        y_h = torch.from_numpy(d["y"]).pin_memory()
        mod.close()
        del W, y, mod
        hm = E.LargeCnlsModel("single_index", d["x0"], {"W": W_h.numpy(), "y": y_h.numpy(), "rho": d["rho"]}, ineq=True,
                              x_low=lo, x_upp=up, device=local)
        E.solve(hm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it2 = 0
        for _ in range(args.large_e2e_steps):
            hm.set_data(0, W_h.numpy())
            hm.set_data(1, y_h.numpy())
            E.solve(hm)
            it2 += int(hm.iterations[0])
        torch.cuda.synchronize()
        dt2 = time.perf_counter() - t0
        res["e2e"] = {"value": it2 / dt2, "unit": "iters/s", "h2d_bytes_per_step": int(C5_M * (C5_N + 1) * 8 + C5_N * 8),
                      "d2h_bytes_per_step": C5_N * 8 + 8 + 16}
        hm.close()
    else:
        mod.close()
    return res


def large_arm(args, torch, dist, E, rank, world, local, dev):
    """One step = one complete solve of the row-sharded problem from x0 (every rank holds m/world rows; R factors
    all-gathered, linesearch sums all-reduced over NCCL).  Strong scaling: the problem size is fixed."""
    m_global = args.large_rows
    rows = m_global // world
    row0 = rank * rows
    if rank == world - 1:
        rows = m_global - row0
    W, y, x0, rho = gen_large_shard(torch, dev, m_global, row0, rows)
    mod = E.LargeCnlsModel("single_index", x0, {"W": W, "y": y, "rho": rho}, m_global=m_global, device=local)
    mod.join(rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, args.large_warmup)):
        E.solve(mod)
    st0 = mod.stats()
    barrier()
    t0 = time.perf_counter()
    iters_solver = 0
    for _ in range(args.large_steps):
        E.solve(mod)
        iters_solver += int(mod.iterations[0])
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, "large_", large_outputs(mod))
    st1 = mod.stats()
    dst = {k: st1[k] - st0[k] for k in st1 if k != "rows_pad"}
    nfac = max(dst["factorisations"], 1.0)
    npts = max(dst["points"], 1.0)
    # `value` counts the iterations the solver reports (length of iterations_detail, 3 for this problem) -- the same
    # count in both arms.  Every pass of the `while exit_code == 0` loop (EF:2776-2878) ends with one new_point!, one
    # more precedes the loop, so passes = points - solves (4: the last pass terminates); the point at which the solve
    # terminates is evaluated (r, J'r, c) but not factored: factorisations = passes.
    iters = iters_solver
    passes = int(npts) - args.large_steps
    tsqr_ms = dst["tsqr_ms"] / nfac
    flops = 2.0 * m_global * (LARGE_N + 1) ** 2          # Householder R factor of the augmented [J | r] (SURVEY.md 8d)
    peak, peak_src = fp64_tensor_peak()
    achieved = flops / world / (tsqr_ms * 1e-3) / 1e12  # per GPU: its m/world rows in its own tsqr time
    res = {"metric": LARGE_METRIC, "value": iters / dt, "unit": "iters/s", "n_gpus": world, "steps": args.large_steps,
           "warmup": max(1, args.large_warmup), "scaling": "strong", "higher_is_better": True, "dtype": "f64",
           "ms_per_iteration": dt * 1e3 / iters, "iterations_reported_by_solver_per_solve": iters_solver / args.large_steps,
           "passes_of_the_loop_per_solve": passes / args.large_steps, "ms_per_pass": dt * 1e3 / max(passes, 1),
           "exit_code": int(mod.exit_code[0]), "status": int(mod.status_code[0]), "objective": float(mod.obj_value[0]),
           "config": {"workload": "C4 single-index m=%d n=256 q=64 (BASELINE.json config 4), analytic Jacobian" % m_global,
                      "rows_per_gpu": rows, "sharding": "row blocks; all-gather of R factors + all-reduce of linesearch sums (NCCL)",
                      "l2": "[J | r] is %.1f GB per GPU, larger than L2" % (rows * (LARGE_N + 8) * 8 / 1e9)},
           "phases_ms_per_factorisation": {"build_J_r_grad": dst["build_ms"] / npts, "tsqr": tsqr_ms},
           "phases_ms_per_solve": {"linesearch_kernels": dst["linesearch_ms"] / args.large_steps,
                                   "small_stage_device": dst["small_stage_ms"] / args.large_steps,
                                   "host_other": (dst["solve_wall_ms"] - dst["build_ms"] - dst["tsqr_ms"] - dst["small_stage_ms"]
                                                  - dst["linesearch_ms"]) / args.large_steps,
                                   "total": dst["solve_wall_ms"] / args.large_steps,
                                   "factorisations": nfac / args.large_steps,
                                   "points_evaluated": npts / args.large_steps,
                                   "linesearch_evals": dst["linesearch_evals"] / args.large_steps},
           "gpu_launches": int(dst["launches"]),
           "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                        "traffic": NCU_TRAIL_DRAM_BYTES_PER_ROW_COL * rows * 224.0, "peak_source": peak_src,
                        "traffic_source": "largest launch of the factorisation (tsqr_trail_staged_kernel, panel 0, level 0: 224 "
                                          "trailing columns): ncu --set full at 1M rows (profiles/r1_c4_trail_staged_v0_ncu.txt) "
                                          "2.25 GB read + 1.83 GB written = 1.04x its algorithmic bytes (trailing block read once, "
                                          "written once, V read once), scaled linearly to this run's rows",
                        "kernel": "tsqr_panel_cg_kernel + tsqr_trail_staged_kernel (one TSQR of [J | r])",
                        "kernel_ms": tsqr_ms, "algorithmic_flops_per_launch": flops / world,
                        "note": "2 m (n+1)^2 flops per factorisation; trailing updates on mma.sync.m8n8k4.f64, panels on the FP64 FMA pipe"}}
    # ---- end to end: W and y start in pinned HOST memory every step, result read back ---------------
    if args.large_e2e_steps > 0:
        W_h = torch.empty(W.shape, dtype=torch.float64).pin_memory()
        y_h = torch.empty(y.shape, dtype=torch.float64).pin_memory()
        W_h.copy_(W); y_h.copy_(y)
        mod.close()
        del W, y, mod
        torch.cuda.empty_cache()
        hm = E.LargeCnlsModel("single_index", x0, {"W": W_h.numpy(), "y": y_h.numpy(), "rho": rho}, m_global=m_global,
                              device=local)
        hm.join(rank, world)
        E.solve(hm)
        barrier()
        t0 = time.perf_counter()
        it2 = 0
        for _ in range(args.large_e2e_steps):
            hm.set_data(0, W_h.numpy())          # H2D of the step's inputs inside the timed region
            hm.set_data(1, y_h.numpy())
            E.solve(hm)                          # x, f, exit code come back to host arrays
            it2 += int(hm.iterations[0])
        barrier()
        dt2 = time.perf_counter() - t0
        t = torch.tensor([dt2], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["e2e"] = {"value": it2 / float(t.item()), "unit": "iters/s",
                      "h2d_bytes_per_step": int(rows * (LARGE_N + 1) * 8 + LARGE_N * 8), "d2h_bytes_per_step": LARGE_N * 8 + 8 + 16,
                      "note": "per GPU; W (%.1f GB) and y copied from pinned host memory every step" % (rows * LARGE_N * 8 / 1e9)}
        hm.close()
    else:
        mod.close()
    return res


def reference_arm(args):
    """`--impl reference`: the CPU implementation of the path on the host cores.

    Enlsip.jl is pure Julia and no Julia binary exists in this image, so oracle/_ref cannot be built;
    the arm times the compiled C++ port of the oracle restatement (oracle/hostport), all host threads.
    """
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = args.cpu_sample
    run, iters = cpu_port(sample, cores)
    for _ in range(args.warmup):
        run()
    times = [run() for _ in range(args.steps)]
    dt = float(np.mean(times))
    v = sample / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C3 gauss-peaks n=6 m=128 q=1 l=13 FD-jacobian (BASELINE.json config 3)",
                       "problems_per_step": sample, "note": "bounded sample of the 4M-problem workload"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d problems (seed 128 stream, first chunk), compiled C++ port of the oracle, OpenMP "
                                       "over problems, every qr(., ColumnNorm()) in OpenBLAS dgeqp3: %s" % (sample, cpu_port.lapack)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mean_iterations": float(np.mean(iters))}
    if not args.skip_large:
        # the reference arm has minutes, not seconds: the C4 pass runs on ALL rows when the host has the memory for W, J
        # and the LAPACK workspace (3 x 8.6 GB), otherwise on the bounded sample
        rows = args.large_rows
        try:
            import psutil
            if psutil.virtual_memory().available < 3.5 * rows * LARGE_N * 8:
                rows = args.large_cpu_rows
        except Exception:
            rows = args.large_cpu_rows
        if args.large_ref_rows > 0:
            rows = args.large_ref_rows
        lb = large_cpu_baseline(rows, args.large_rows)
        line["large"] = {"impl": "reference", "metric": LARGE_METRIC, "value": lb["value"], "unit": "iters/s",
                         "higher_is_better": True, "cpu_baseline": lb,
                         "config": {"workload": "C4 single-index m=%d n=256 q=64 (BASELINE.json config 4)" % args.large_rows}}
        if not args.skip_c5:
            cb = c5_cpu_baseline(scale=1 if args.c5_ref_full else 2)
            line["large5"] = {"impl": "reference", "metric": C5_METRIC, "value": cb["value"], "unit": "iters/s",
                              "higher_is_better": True, "cpu_baseline": cb,
                              "config": {"workload": "C5 single-index n=4096 m=16384, 1024 inequalities + 8192 bounds (BASELINE.json config 5)"}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--problems", type=int, default=int(os.environ.get("ENLSIP_BENCH_PROBLEMS", 4_000_000)),
                    help="problems per GPU per step (named size: 4,000,000)")
    ap.add_argument("--cpu-sample", type=int, default=60_000)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-large", action="store_true", help="skip the large-Jacobian half of the metric (config 4)")
    ap.add_argument("--large-rows", type=int, default=int(os.environ.get("ENLSIP_BENCH_LARGE_ROWS", 1 << 22)))
    ap.add_argument("--large-steps", type=int, default=3)
    ap.add_argument("--large-warmup", type=int, default=1)
    ap.add_argument("--large-e2e-steps", type=int, default=1)
    ap.add_argument("--large-cpu-rows", type=int, default=1 << 19,
                    help="rows of the C4 problem the cpu_baseline leg of the default run times (scaled linearly to --large-rows)")
    ap.add_argument("--large-ref-rows", type=int, default=0, help="--impl reference: rows to time (0 = all rows if memory allows)")
    ap.add_argument("--skip-c5", action="store_true", help="skip BASELINE.json config 5 (one GPU, replicas only)")
    ap.add_argument("--skip-c2", action="store_true", help="skip BASELINE.json config 2 (batched HS65)")
    ap.add_argument("--c2-problems", type=int, default=1_000_000, help="HS65 instances per GPU (config 2)")
    ap.add_argument("--c5-steps", type=int, default=2)
    ap.add_argument("--c5-ref-full", action="store_true", help="--impl reference: time the C5 pass at the named size (minutes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of each arm's last timed step as DIR/<name>.npy (float64; batched outputs as a "
                         "fixed, seeded sample of problems, with their indices in index.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA engine (--impl ours)")
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import enlsip_jl_b200 as E
    from enlsip_jl_b200.model import last_kernel_ms

    rank, world, local = dist_env()
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner there) are pointed at
    # stderr for the whole run, the line goes to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.problems

    # ---- synthetic inputs of this rank's shard, pinned on the host ---------------------------------
    y_np, S_np, x0_np, _ = E.synth.gen_gauss_peaks_batch(B, start=rank * B)
    y_h = torch.from_numpy(np.ascontiguousarray(y_np)).pin_memory()
    S_h = torch.from_numpy(np.ascontiguousarray(S_np)).pin_memory()
    x0_h = torch.from_numpy(np.ascontiguousarray(x0_np)).pin_memory()
    del y_np, S_np, x0_np
    y_d, S_d, x0_d = y_h.to(dev), S_h.to(dev), x0_h.to(dev)

    model = E.CnlsModel("gauss_peaks", x0_d, data={"y": y_d, "S": S_d}, x_low=E.synth.GP_LOW, x_upp=E.synth.GP_UPP,
                        jacobian="forward_diff", device=local)
    out = {"x": torch.empty(B, 6, dtype=torch.float64, device=dev), "f": torch.empty(B, dtype=torch.float64, device=dev)}
    for k in ("exit_code", "status", "iters", "nact"):
        out[k] = torch.empty(B, dtype=torch.int32, device=dev)

    def step():
        E.solve(model, want_active=False, want_counters=False, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = model.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
        kernel_ms.append(None)
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    kms = last_kernel_ms(model)    # the dominant (only) kernel: CUDA events on its launch stream, last timed step
    clocks = sampler.stop() if rank == 0 else None
    launches = model.launch_count() - launches0
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    # rank 0's shard; 2^19 of the 4M problems keep the outputs of every arm under 64 MB
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, "", out, sample_rows(B, 1 << 19))
    ms_per_step = elapsed_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    status = out["status"].cpu().numpy()
    iters = out["iters"].cpu().numpy()
    conv = float(np.mean(status == 1))

    # ---- the evaluation phase alone (SURVEY.md 8d, last row): forward-difference Jacobian + residuals of every problem,
    #      written to HBM (enlsipb200_eval_batch); the one phase of the solve with no replicated work ----------------
    fdj = None
    stepk = None
    if rank == 0:
        Bf = min(B, 1_000_000)
        xs = x0_d[:Bf].contiguous()
        fm = E.CnlsModel("gauss_peaks", xs, data={"y": y_d[:Bf].contiguous(), "S": S_d[:Bf].contiguous()}, x_low=E.synth.GP_LOW,
                         x_upp=E.synth.GP_UPP, jacobian="forward_diff", device=local)
        E.evaluate(fm, xs, want=("r", "J"))
        torch.cuda.synchronize()
        ms = []
        for _ in range(3):
            E.evaluate(fm, xs, want=("r", "J"))
            torch.cuda.synchronize()
            ms.append(last_kernel_ms(fm))
        t_ms = float(np.median(ms))
        # algorithmic work of jac_forward_diff + res_eval! (cnls_model.jl:40-82): n + 1 = 7 evaluations of the 128 residuals,
        # each 2 exponentials (det_exp: 15 FMA + 7 other FP64 instructions = 37 flop) + 12 flop of model arithmetic
        flop = 7 * 128 * (2 * 37 + 12) * float(Bf)
        wbytes = Bf * (128 * 6 + 128) * 8.0
        fdj = {"problems": Bf, "kernel_ms": t_ms, "kernel": "enlsip_eval_batch_kernel<GaussPeaks> (r and J of every problem to HBM)",
               "achieved_tflops": flop / (t_ms * 1e-3) / 1e12, "peak_tflops": fp64_fma_peak(),
               "frac_of_fp64_fma_peak": flop / (t_ms * 1e-3) / 1e12 / fp64_fma_peak(),
               "algorithmic_flop_per_problem": flop / Bf, "hbm_write_gbs": wbytes / (t_ms * 1e-3) / 1e9,
               "note": "the engine's FD kernel re-uses the unperturbed exponentials (6 instead of 14 det_exp per row, bit-identical "
                       "values), so it executes fewer flops than the algorithmic count it is credited with"}
        # ---- the batched STEP kernel from materialised inputs (SURVEY.md 8d, the HBM-roofline row): reads J, r, A, c of
        #      every problem from HBM (written by the evaluation kernel above), one update_working_set each ----
        ev = E.evaluate(fm, xs)
        E.gn_step(fm, xs, ev)
        torch.cuda.synchronize()
        ms = []
        for _ in range(3):
            E.gn_step(fm, xs, ev)
            torch.cuda.synchronize()
            ms.append(last_kernel_ms(fm))
        s_ms = float(np.median(ms))
        step_bytes = 8.0 * (128 * 6 + 128 + 13 * 6 + 13 + 2 * 6)          # SURVEY.md 8d: 8 (mn + m + ln + l + 2n) = 7992 B
        hbm_peak, hbm_src = measured_peaks()
        stepk = {"problems": Bf, "kernel_ms": s_ms, "kernel": "enlsip_eval_batch_kernel<GaussPeaks> in step mode (enlsipb200_step_batch)",
                 "algorithmic_bytes_per_problem": step_bytes, "steps_per_s": Bf / (s_ms * 1e-3),
                 "roofline": {"bound": "hbm", "achieved": step_bytes * Bf / (s_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                              "frac": step_bytes * Bf / (s_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "traffic": None},
                 "note": "one warp per problem with the n = 6 logic replicated over its lanes (the solve kernel's building blocks): "
                         "latency / instruction bound, far from the HBM roofline the survey assigns to this kernel"}
        del ev
        fm.close()
        del fm

    # ---- end to end through the C ABI with pinned host buffers -------------------------------------
    x_h = torch.empty(B, 6, dtype=torch.float64).pin_memory()
    f_h = torch.empty(B, dtype=torch.float64).pin_memory()
    ints_h = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(4)]
    hmodel = E.CnlsModel("gauss_peaks", x0_h.numpy(), data={"y": y_h.numpy(), "S": S_h.numpy()}, x_low=E.synth.GP_LOW,
                         x_upp=E.synth.GP_UPP, jacobian="forward_diff", device=local)
    hout = {"x": x_h.numpy(), "f": f_h.numpy(), "exit_code": ints_h[0].numpy(), "status": ints_h[1].numpy(),
            "iters": ints_h[2].numpy(), "nact": ints_h[3].numpy()}

    def e2e_step():
        hmodel.set_data(0, y_h.numpy())          # H2D of the step's inputs, inside the timed region
        hmodel.set_data(1, S_h.numpy())
        E.solve(hmodel, want_active=False, want_counters=False, out=hout)   # H2D x0, kernel, D2H results (blocking)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.e2e_steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B / float(t.item())
    h2d = B * (128 + 1 + 6) * 8
    d2h = B * (6 * 8 + 8 + 4 * 4)
    same = bool(np.array_equal(hout["status"], status)) and bool(np.array_equal(hout["iters"], iters))

    c2 = None if args.skip_c2 else c2_arm(args, torch, dist, E, rank, world, local, dev)

    # ---- the other half of the metric: GN iterations/s of the large-Jacobian regime (config 4) -------
    kernel_info = model.kernel_info()
    large = None
    if not args.skip_large:
        del hmodel, model, y_d, S_d, x0_d, y_h, S_h, x0_h, x_h, f_h, out, hout
        torch.cuda.empty_cache()
        large = large_arm(args, torch, dist, E, rank, world, local, dev)
    large5 = None
    if not args.skip_large and not args.skip_c5 and world == 1:
        torch.cuda.empty_cache()
        large5 = c5_arm(args, torch, E, dev, local)

    if rank == 0:
        peak, peak_src = measured_peaks()
        achieved = ALG_BYTES_PER_SOLVE * B / (kms * 1e-3) / 1e9
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C3 gauss-peaks n=6 m=128 q=1 l=13 FD-jacobian (BASELINE.json config 3)",
                           "problems_per_gpu": B, "seed": 128, "sharding": "contiguous shards, no collective",
                           "l2": "inputs (%.2f GB/GPU) larger than L2" % (B * 135 * 8 / 1e9)},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "same_results_as_device_path": same},
                "gpu_launches": int(launches),
                "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": NCU_DRAM_BYTES_PER_SOLVE * B, "peak_source": peak_src,
                             "kernel": "enlsip_solve_batch_kernel<GaussPeaks>",
                             "kernel_ms": kms, "algorithmic_bytes_per_solve": ALG_BYTES_PER_SOLVE,
                             "traffic_source": "ncu --set full, 30000 solves (profiles/r1_c3_v4_ncu.txt): 1.12 KB read + 30.0 KB "
                                               "written per solve; the writes are stack (local-memory) lines leaving L2, not data",
                             "note": "fused whole-solve kernel: every intermediate stays on chip, so it is FP64/latency bound "
                                     "and not HBM bound by construction (DESIGN.md 5.1); see roofline_fp64"},
                "roofline_fp64": {"bound": "fp64 pipe", "achieved": value / world * ALG_FLOP_PER_SOLVE / 1e12,
                                  "peak": fp64_fma_peak(), "unit": "TFLOP/s",
                                  "frac": value / world * ALG_FLOP_PER_SOLVE / 1e12 / fp64_fma_peak(),
                                  "algorithmic_flop_per_solve": ALG_FLOP_PER_SOLVE,
                                  "note": "algorithmic flops (SURVEY.md 8d: ~2e5 per Gauss-Newton iteration x the mean iteration "
                                          "count); ncu: FP64 pipe 12.7 % active, issue slots 34 % (profiles/r1_c3_v4_ncu.txt)"},
                "fd_jacobian_phase": fdj,
                "step_kernel": stepk if rank == 0 else None,
                "quality": {"converged_fraction": conv, "mean_iterations": float(iters.mean()),
                            "kernel_info": kernel_info}}
        if not args.skip_cpu and world == 1:      # cpu_baseline: rank 0 at N = 1 only
            cores = os.cpu_count() or 1
            run, cit = cpu_port(args.cpu_sample, cores)
            run()
            dt = min(run() for _ in range(2))
            line["cpu_baseline"] = {"value": args.cpu_sample / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d problems of the same stream, compiled C++ port of the oracle "
                                              "(oracle/hostport), OpenMP over problems, every qr(., ColumnNorm()) in OpenBLAS "
                                              "dgeqp3 (%s); Enlsip.jl itself needs Julia, absent from this image"
                                              % (args.cpu_sample, cpu_port.lapack),
                                    "mean_iterations": float(np.mean(cit))}
        if c2 is not None:
            line["batched_hs65"] = c2
            line["gpu_launches"] += c2["gpu_launches"]
        if large is not None:
            if not args.skip_cpu and world == 1:
                large["cpu_baseline"] = large_cpu_baseline(args.large_cpu_rows, args.large_rows)
            line["large"] = large
            line["gpu_launches"] += large["gpu_launches"]
        if large5 is not None:
            if not args.skip_cpu:
                large5["cpu_baseline"] = c5_cpu_baseline()
            line["large5"] = large5
            line["gpu_launches"] += large5["gpu_launches"]
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
