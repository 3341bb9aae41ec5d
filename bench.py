#!/usr/bin/env python
"""bench.py - headline benchmark of the Krylov matrix-function hot path (BASELINE.json).

Workload (config C3, SURVEY.md 8d): synthetic power-law graph n = 1M, nnz = 20M (Chung-Lu,
seed 20260310), A scaled by 1/lambda_max-estimate, 512 Rademacher probes PER GPU, m = 30 Lanczos
steps per probe, trace(exp(A)) by stochastic Lanczos quadrature.  One "step" = one full pass
(512 x 30 = 15 360 Krylov matvecs per GPU).  A is replicated, probes are sharded across ranks, one
NCCL all-reduce of the partial trace per step (weak scaling: per-GPU work is fixed).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric: Krylov matvecs/sec (an n x k SpMM counts k).  `value` = device-resident probes;
`e2e` = through the public host-buffer call kr_slq_trace (pinned host probes -> device, result back).
`--impl reference` times the reference's CPU algorithm (the NumPy/SciPy oracle: the reference is
MATLAB-only and cannot run here) on the host cores with the same metric.

`--steps K` is the number of timed steps of every C3 arm (device probes, host probes, int8 sign probes, strong
scaling); the C5, C4 and C2 arms time fixed calls.  At least 3 untimed steps precede the C3 timing whatever
`--warmup` says with `--impl ours` (the first steps load modules and size the memory pool); the JSON line reports
the number run.

`--dump-outputs DIR` writes, after the run, what the timed calls returned to their caller as DIR/<name>.npy
(float64): c3_trace (the trace of the last timed step), c5_edge_scores, c2_entries and c4_expmv_sample (4096
seeded rows of the n x 64 result), each for the arms that ran.  All inputs are seeded, so the same arguments give
the same inputs and two builds can be compared output for output.  The inputs that the device itself derives are
written next to them, so that a difference there shows up as an input change: c5_candidates (the 1-based node
pairs picked by the device centrality), c4_tscale (from the device norm estimate) and c2_tol (likewise).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_NODES = int(os.environ.get("KR_BENCH_N", 1_000_000))
NNZ = int(os.environ.get("KR_BENCH_NNZ", 20_000_000))
K_PROBES = int(os.environ.get("KR_BENCH_K", 512))
M_STEPS = int(os.environ.get("KR_BENCH_M", 30))
GRAPH_SEED = 20260310
PROBE_SEED = 1
METRIC = "krylov_matvecs_per_sec"
UNIT = "matvec/s"


def build_graph():
    from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate
    A = power_law_graph(N_NODES, NNZ, 2.2, GRAPH_SEED)
    lam = spectral_radius_estimate(A, 30)
    A = A * (1.0 / lam)          # uniform value -> stored pattern-only on the device
    A = A.tocsr()
    reorder = os.environ.get("KR_BENCH_REORDER", "")      # experiment knob: symmetric relabelling of the nodes
    if reorder:
        if reorder == "degree":
            perm = np.argsort(-np.diff(A.indptr), kind="stable")
        elif reorder == "rcm":
            from scipy.sparse.csgraph import reverse_cuthill_mckee
            perm = reverse_cuthill_mckee(A, symmetric_mode=True)
        else:
            raise SystemExit("KR_BENCH_REORDER must be degree or rcm")
        A = A[perm][:, perm].tocsr()
        A.sort_indices()
    return A, lam


def config_dict(world):
    return {"workload": "C3: power-law n=%d nnz=%d, %d Rademacher probes/GPU, Lanczos m=%d, trace(exp(A)) by SLQ"
                        % (N_NODES, NNZ, K_PROBES, M_STEPS),
            "n": N_NODES, "nnz": NNZ, "probes_per_gpu": K_PROBES, "lanczos_steps": M_STEPS,
            "sharding": "A replicated, probes split across %d rank(s), 1 all-reduce/step" % world,
            "cache": "inputs larger than L2 (each dense block is %.1f GB)" % (N_NODES * K_PROBES * 8 / 1e9)}


# ------------------------------------------------------------------------------- CPU arms
_CPU_A = None      # set before forking so the workers inherit the matrix instead of unpickling it


def _cpu_worker(args):
    col_offset, cols, m = args
    import oracle
    Z = _rademacher(_CPU_A.shape[0], cols, PROBE_SEED, col_offset)
    return oracle.slq_trace(_CPU_A, Z, m, "exp")[0]


def _rademacher(n, k, seed, col_offset):
    """Same counter-based +-1 stream as the device (splitmix64 of seed ^ (col << 32 | row)); restated here
    so the CPU arms do not touch the engine package."""
    i = np.arange(n, dtype=np.uint64)[:, None]
    c = (np.arange(k, dtype=np.uint64) + np.uint64(col_offset))[None, :]
    x = np.uint64(seed) ^ ((c << np.uint64(32)) | i)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return np.where((x >> np.uint64(63)) == 1, -1.0, 1.0)


def cpu_slq_rate(A, cols_per_proc, procs, m):
    """matvecs/s of the oracle's SLQ on `procs` host processes (each: cols_per_proc probes)."""
    import multiprocessing as mp
    global _CPU_A
    _CPU_A = A
    jobs = [(p * cols_per_proc, cols_per_proc, m) for p in range(procs)]
    t0 = time.perf_counter()
    if procs == 1:
        _cpu_worker(jobs[0])
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_cpu_worker, jobs)
    dt = time.perf_counter() - t0
    return procs * cols_per_proc * m / dt, dt


def cpu_block_sweep(A, m):
    """Pick the per-process probe-block width for the CPU arm: SciPy's CSR x dense product re-reads A once per
    block, so a 2-column block (round 1) starves it.  One core, 8 Lanczos steps, widths 8 / 16 / 32."""
    best = (0.0, 16)
    for cols in (16, 32):
        rate, _ = cpu_slq_rate(A, cols, 1, min(m, 4))
        best = max(best, (rate, cols))
    return best[1]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import shutil
    interp = [x for x in ("octave", "octave-cli", "matlab") if shutil.which(x)]
    A, _ = build_graph()
    cores = os.cpu_count() or 1
    cols = int(os.environ.get("KR_BENCH_CPU_COLS", 0)) or cpu_block_sweep(A, M_STEPS)
    # bounded sample per step: every process runs `cols` probes for m_cpu Lanczos steps (the per-matvec cost of the
    # recurrence does not depend on the step count), ~8 s per step on 16 cores
    m_cpu = int(os.environ.get("KR_BENCH_CPU_M", 4))
    times = []
    for it in range(args.warmup + args.steps):
        rate, dt = cpu_slq_rate(A, cols, cores, m_cpu)
        if it >= args.warmup:
            times.append((rate, dt))
    rate = float(np.mean([r for r, _ in times]))
    ms = float(np.mean([d for _, d in times]) * 1e3)
    sample = "%d probes (%d per process x %d processes, block width picked by a one-core sweep over 16/32) x %d Lanczos " \
             "steps of the same graph per step" % (cols * cores, cols, cores, m_cpu)
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(max(int(args.gpus), 1)),      # the arm's config at this N (the CPU rate does not scale with N)
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "interpreters_found": interp,
            "note": "reference is MATLAB-only; probed for octave / octave-cli / matlab on PATH: %s. This is the NumPy/SciPy "
                    "oracle port of functions/*.m on the host cores" % (interp or "none")}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------- our arm
PEAK_SOURCE = ["fallback"]


def peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            v = float(json.load(f)["hbm_gbs"])
        PEAK_SOURCE[0] = "measured"
        return v
    except Exception:
        PEAK_SOURCE[0] = "fallback"
        return 6650.0


def dump_outputs(outdir, outputs):
    os.makedirs(outdir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(outdir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def bench_c2(kr, ctx, outputs):
    """Config C2 (datasets_paper/Transport, gradient over ALL edges): gr = -2 cosh(A + Delta(X))_Omega on the largest road
    network of the reference's data (Vermont after the scripts' preprocessing, committed fixture), through
    function_multiple_entries - one single-vector Krylov space per distinct row index, each run whole in one CTA on the
    ball around its start node (csrc/entries_local.cuh).  Setup as scripts/bench_c2.py / Tests/test_weighted_sinh_lbfgs.m:52."""
    import warnings
    import scipy.sparse as sp
    path = os.path.join(ROOT, "tests", "golden", "graph_transport_Vermont.npz")
    if not os.path.exists(path):
        return {"unavailable": "tests/golden/graph_transport_Vermont.npz not found"}
    z = np.load(path)
    n = int(z["n"])
    A = sp.csr_matrix((z["data"], z["indices"], z["indptr"]), shape=(n, n)).astype(np.float64)
    A = (A / A.max()).tocsr()
    L = sp.tril(A, -1).tocoo()
    Om = np.stack([L.row + 1, L.col + 1], 1).astype(np.int64)
    X = 0.1 * L.data * np.random.default_rng(4).random(L.nnz)
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (A + D + D.T).tocsr()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        tol = 1e-8 * float(np.cosh(float(kr.normest(A, 1e-2)[0])))
        t0 = time.perf_counter()
        M = kr.Matrix(At, ctx)
        ctx.sync()
        t_mat = time.perf_counter() - t0
        kr.function_multiple_entries(M, Om[:256], "cosh", tol, 100)          # warm-up
        ctx.sync()
        times, c0 = [], ctx.counters()
        for _ in range(3):
            t0 = time.perf_counter()
            v, it = kr.function_multiple_entries(M, Om, "cosh", tol, 100)
            ctx.sync()
            times.append(time.perf_counter() - t0)
        c1 = ctx.counters()
    outputs["c2_entries"] = v
    outputs["c2_tol"] = np.array([tol])
    t = min(times)
    return {"metric": "gradient_entries_per_sec", "value": Om.shape[0] / t, "unit": "entry/s",
            "workload": "C2: transport_Vermont (n=%d, %d edges), gradient of trace sinh(A+X) over ALL edges = %d entries of "
                        "cosh(A+Delta) from %d single-vector Arnoldi spaces (full CGS2 + third pass)"
                        % (n, Om.shape[0], Om.shape[0], int(np.unique(Om[:, 0]).size)),
            "call_s": t, "calls_timed": len(times), "iterations": int(it), "matrix_analysis_upload_s": t_mat,
            "matvecs_per_call": (c1["matvecs"] - c0["matvecs"]) // len(times),
            "gpu_launches_per_call": (c1["launches"] - c0["launches"]) // len(times),
            "gradient_checksum": float(np.sum(-2.0 * v)), "max_abs_entry": float(np.max(np.abs(2.0 * v))),
            "timing": "host clock around kr_function_multiple_entries incl. index upload and result download (resident matrix)",
            "dense_batch_reference_s": 11.7,
            "note": "round-2 dense batch (all spaces advanced by n x R SpMMs): 11.5-11.9 s for the same call, see DESIGN.md 6"}


def bench_c4(kr, ctx, outputs):
    """expmv (Al-Mohy-Higham) on the C4 graph: ms per fused Taylor term and its fraction of the HBM roofline
    (algorithmic bytes 4*nnz [pattern-only CSR] + 4*(n+1) + 32*n*q: read b, write b', read-modify-write f)."""
    from krylov_robustness_b200.graphs import rmat_graph_device
    scale = int(os.environ.get("KR_BENCH_C4_SCALE", 24))
    nnz_t = int(os.environ.get("KR_BENCH_C4_NNZ", 1 << (scale + 4)))
    q = int(os.environ.get("KR_BENCH_C4_Q", 64))
    t0 = time.perf_counter()
    indptr, indices = rmat_graph_device(scale, nnz_t, seed=2, device=ctx.device)
    n, nnz = indptr.size - 1, indices.size
    gen_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    M4 = kr.Matrix.from_csr_arrays(n, indptr, indices, 1.0, ctx)
    del indptr, indices
    upload_s = time.perf_counter() - t0
    lam4 = float(kr.normest(M4, 1e-3)[0])                 # symmetric: ||A||_2 (device power iteration)
    tscale = 8.0 / lam4                                   # ||tA||_2 ~ 8: s*m = O(10^2), e^{t lambda} finite
    b = np.random.default_rng(3).standard_normal((n, q))
    kr.expmv(tscale, M4, b[:, :8])                        # warm-up
    ctx.set_timing(True)
    ctx.spmm_time(reset=True)
    c0 = ctx.counters()
    t0 = time.perf_counter()
    f, s, mdeg, mv, mvd, unA = kr.expmv(tscale, M4, b)
    wall = time.perf_counter() - t0
    ms, launches = ctx.spmm_time(reset=True)
    c1 = ctx.counters()
    ctx.set_timing(False)
    terms = mv - mvd
    # the timed SpMM launches are the Taylor terms (q columns each); the 1-norm power sequence runs on the SpMV kernel
    ms_term = ms / max(launches, 1)
    bytes_term = 4.0 * nnz + 4.0 * (n + 1) + 32.0 * n * q
    peak = peak_gbs()
    out = {"metric": "expmv_taylor_term", "workload": "C4: R-MAT scale %d, %d stored entries, %d right-hand sides, ||tA||_2 ~ 8, "
                                                      "normAm / degree selection on the device" % (scale, nnz, q),
           "n": n, "nnz": nnz, "q": q, "s": int(s), "m": int(mdeg), "mv": int(mv), "mvd": int(mvd), "unA": int(unA),
           "taylor_terms_timed": int(launches), "ms_per_taylor_term": ms_term,
           "matvecs_per_sec": launches * q / (ms * 1e-3) if ms > 0 else None,
           "algorithmic_bytes_per_term": bytes_term, "achieved_GBs": bytes_term / (ms_term * 1e-3) / 1e9,
           "peak_GBs": peak, "frac": bytes_term / (ms_term * 1e-3) / 1e9 / peak,
           "expmv_call_wall_s_incl_h2d_d2h": wall, "graph_gen_s": gen_s, "matrix_analysis_upload_s": upload_s,
           "gpu_launches": c1["launches"] - c0["launches"], "lambda_max_est": lam4}
    rows = np.sort(np.random.default_rng(0).choice(n, min(n, 4096), replace=False))
    outputs["c4_expmv_sample"] = f[rows]
    outputs["c4_tscale"] = np.array([tscale])
    del M4, f, b
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import krylov_robustness_b200 as kr

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU fallback")
    torch.cuda.set_device(local)
    from krylov_robustness_b200.parallel import bind_to_gpu_numa_node
    numa = bind_to_gpu_numa_node(local)          # before any pinned allocation: keep the probes socket-local
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from krylov_robustness_b200 import parallel as P
    A, lam = build_graph()
    n, nnz = A.shape[0], A.nnz
    ctx = kr.Context(local)
    M = kr.Matrix(A, ctx)
    pattern_only = M.info()["pattern_only"]
    k, m = K_PROBES, M_STEPS
    Zdev = kr.Dense(n, k, ctx).fill_rademacher(PROBE_SEED, col_offset=rank * k)
    # pinned host copy of the same probes for the end-to-end arm (column-major n x k)
    Zpin = torch.empty((k, n), dtype=torch.float64, pin_memory=True)
    for c0 in range(0, k, 64):                      # chunked: bounded host memory with 8 ranks per node
        cw = min(64, k - c0)
        Zpin.numpy()[c0:c0 + cw] = kr.Dense(n, cw, ctx).fill_rademacher(PROBE_SEED, col_offset=rank * k + c0).download().T
    zptr = Zpin.data_ptr()
    # the same probes as int8 signs (Rademacher probes carry one bit per entry): kr_slq_trace_sign
    Zpin8 = torch.empty((k, n), dtype=torch.int8, pin_memory=True)
    Zpin8.copy_(Zpin.to(torch.int8))
    zptr8 = Zpin8.data_ptr()
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    acc = torch.zeros(1, dtype=torch.float64, device="cuda")

    def reduce_trace(tr_local):
        # one collective per step: sum of the per-rank partial traces (tiny; latency-bound)
        acc.fill_(tr_local / world)
        if world > 1:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        return acc

    def step_dev():
        return reduce_trace(kr.slq_trace(M, Zdev, m, "exp"))

    import ctypes as C
    from krylov_robustness_b200._lib import check

    def step_e2e():
        tr = C.c_double()
        check(ctx.lib.kr_slq_trace(ctx.h, M.h, k, C.c_void_p(zptr), n, m, 0, C.byref(tr), None, None, None))
        return float(reduce_trace(tr.value).item())       # device -> host read of the step's result

    def step_e2e_sign():
        tr = C.c_double()
        check(ctx.lib.kr_slq_trace_sign(ctx.h, M.h, k, C.c_void_p(zptr8), n, m, 0, C.byref(tr), None, None, None))
        return float(reduce_trace(tr.value).item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        last = None
        for _ in range(steps):
            last = fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    for _ in range(max(args.warmup, 3)):
        step_dev()
    ctx.set_timing(True)
    ctx.spmm_time(reset=True)
    c0 = ctx.counters()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, tr_dev = timed(step_dev, args.steps)
    clocks = sampler.stop() if sampler else None
    c1 = ctx.counters()
    spmm_ms, spmm_launches = ctx.spmm_time(reset=True)
    ctx.set_timing(False)
    tr_value = float(tr_dev.item())
    outputs = {"c3_trace": np.array([tr_value])}

    # ---- strong scaling of the headline (SURVEY.md 8e: the 512 probe columns SPLIT across the ranks)
    strong = None
    if world > 1 and os.environ.get("KR_BENCH_STRONG", "1") != "0":
        lo, hi = P.shard_bounds(k)
        Zs = kr.Dense(n, hi - lo, ctx).fill_rademacher(PROBE_SEED, col_offset=lo)

        def step_strong():
            s_local = kr.slq_trace(M, Zs, m, "exp") * (hi - lo)
            acc.fill_(s_local / k)
            dist.all_reduce(acc, op=dist.ReduceOp.SUM)
            return acc
        step_strong()
        ms_s, tr_s = timed(step_strong, args.steps)
        strong = {"value": k * m * args.steps / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s / args.steps,
                  "probes_total": k, "probes_per_gpu": hi - lo, "trace_estimate": float(tr_s.item()),
                  "note": "same 512 probes split across the ranks (strong scaling); the headline `value` is weak scaling"}
        del Zs

    # ---- secondary metric of BASELINE.json (config C5): candidate edges scored per second.  10^5 missing-edge
    # candidates from find_top_missing_edges(A, leading-eigenvector centrality, 1e5, 'min') on the same graph, SPLIT
    # across the ranks (12 500 per GPU at 8), scored by the batched rank-2 trace_fun_update path, one all-gather of
    # the scores + the reference's first-wins arg-max per round.
    secondary = None
    if os.environ.get("KR_BENCH_EDGES", "1") != "0":
        ncand = int(os.environ.get("KR_BENCH_C5_CAND", 100_000))
        t0 = time.perf_counter()
        cvec = kr.compute_centrality(M, "eig", 1e-10)
        E = kr.find_top_missing_edges(A, cvec, ncand, "min")
        t_cand = time.perf_counter() - t0
        tol_e = 1e-6 * float(np.exp(1.0))                 # 1e-6 * exp(||A||), A scaled to spectral radius ~1
        b_off = 1.0 / lam                                 # an edge of the unscaled graph, in the scaled units

        def score_round(Ecand):
            its = []

            def local(Es):
                x, it, _ = kr.trace_fun_update_edges(M, Es, b_off, tol_e, 100, "exp")
                its.append(it)
                return x
            vals = P.sharded_edge_scores(local, Ecand)
            return vals, (np.concatenate(its) if its else np.zeros(0))
        score_round(E[:64 * world])                       # warm-up (allocations, attribute setup)
        ms_edges, (vals, its) = timed(lambda: score_round(E), 1)
        outputs["c5_edge_scores"] = vals
        outputs["c5_candidates"] = E
        lo, hi = P.shard_bounds(E.shape[0])
        # edge roofline of SURVEY.md 8(d): matvec roofline / (2 * mean steps)
        b_mv = ((4.0 if pattern_only else 12.0) * nnz + 4.0 * (n + 1)) / 512 + 16.0 * n
        secondary = {"metric": "edges_scored_per_sec", "value": E.shape[0] / (ms_edges * 1e-3), "unit": "edge/s",
                     "workload": "C5: %d candidates of find_top_missing_edges(A, eig centrality, 'min') on the C3 graph, "
                                 "split across %d rank(s)" % (E.shape[0], world),
                     "candidates": int(E.shape[0]), "candidates_this_gpu": int(hi - lo), "ms_per_round": ms_edges,
                     "distinct_nodes": int(np.unique(E).size),
                     "mean_block_lanczos_steps": float(its.mean()) if its.size else None,
                     "steps_histogram_rank0": {int(a): int(b) for a, b in zip(*np.unique(its, return_counts=True))},
                     "candidate_generation_s": t_cand,
                     "best_candidate": [int(v) for v in E[int(np.argmax(vals))]],
                     "scaling": "strong",
                     "note": "one greedy 'make' round: all candidates scored + all-gather + first-wins arg-max"}
        if its.size:
            secondary["roofline_edges_per_sec_per_gpu"] = peak_gbs() * 1e9 / b_mv / (2.0 * float(its.mean()))
            secondary["frac_of_edge_roofline"] = secondary["value"] / world / secondary["roofline_edges_per_sec_per_gpu"]
        # ---- the same greedy round with the node-basis screen (kr_greedy_round, csrc/nodepairs.cuh): shared per-node
        # Krylov bases rule out the candidates that cannot win (values to 1e-9..1e-8, NOT the parity path); only the
        # contenders take the exact path and the selection runs on exact values.  Each rank screens its own shard, one
        # all-gather of (index, value) pairs, first-wins over the rank order.
        if os.environ.get("KR_BENCH_SCREEN", "1") != "0":
            def screened_round(Ecand):
                lo_, hi_ = P.shard_bounds(Ecand.shape[0])
                b, v, sc, mask, info = kr.greedy_round(M, Ecand[lo_:hi_], b_off, tol_e, 100, "exp", "make", screen=True)
                mine = torch.tensor([float(lo_ + b) if b >= 0 else -1.0, v if b >= 0 else float("-inf"), float(info["exact"]),
                                     float(info["nodes"])], dtype=torch.float64, device="cuda")
                allr = [torch.zeros_like(mine) for _ in range(world)] if world > 1 else [mine]
                if world > 1:
                    dist.all_gather(allr, mine)
                rows = torch.stack(allr).cpu().numpy()
                best_i, best_v = -1, float("-inf")
                for r in rows:                       # rank order = candidate order: strict > keeps the first
                    if r[0] >= 0 and r[1] > best_v:
                        best_i, best_v = int(r[0]), float(r[1])
                return best_i, best_v, rows, sc, mask
            screened_round(E)                        # warm-up at full size (pool blocks of the round's own shapes)
            ms_scr, (bi, bv, rows, sc, mask) = timed(lambda: screened_round(E), 1)
            ex_best = int(np.argmax(vals))
            lo, hi = P.shard_bounds(E.shape[0])
            dev = np.abs(sc - vals[lo:hi]) / np.abs(vals[lo:hi])
            secondary["screened_round"] = {
                "metric": "edges_scored_per_sec", "value": E.shape[0] / (ms_scr * 1e-3), "unit": "edge/s", "ms_per_round": ms_scr,
                "same_edge_and_value_as_exact_round": bool(bi == ex_best and bv == float(vals[ex_best])),
                "exactly_rescored_candidates": int(rows[:, 2].sum()), "distinct_nodes_rank0": int(rows[0, 3]),
                "screen_max_rel_deviation_rank0": float(dev.max()), "speedup_vs_exact_round": ms_edges / ms_scr,
                "note": "NOT the 1e-10 parity path for the discarded candidates: the screen's values deviate by up to ~1e-8 "
                        "relative; the selected edge and its value are those of the exact round (checked here)"}

    for _ in range(1):
        step_e2e()
    h0 = ctx.counters()
    ms_e2e, tr_e2e = timed(step_e2e, args.steps)
    h1 = ctx.counters()
    step_e2e_sign()
    g0 = ctx.counters()
    ms_e2e8, tr_e2e8 = timed(step_e2e_sign, args.steps)
    g1 = ctx.counters()

    # ---- config C4: expmv Taylor path on R-MAT 2^24 nodes / 2^28 stored entries, 64 right-hand sides, normAm on the
    # device.  One GPU's worth of work (A replicated, columns would be split): measured on rank 0 when N == 1.
    secondary_c4 = None
    if rank == 0 and os.environ.get("KR_BENCH_C4", "1" if world == 1 else "0") != "0":
        secondary_c4 = bench_c4(kr, ctx, outputs)
    # ---- config C2: gradient over all edges of the largest Transport road network (rank 0, N == 1)
    secondary_c2 = None
    if rank == 0 and os.environ.get("KR_BENCH_C2", "1" if world == 1 else "0") != "0":
        secondary_c2 = bench_c2(kr, ctx, outputs)

    if rank == 0:
        mv_step = k * m * world
        value = mv_step * args.steps / (ms_dev * 1e-3)
        e2e = mv_step * args.steps / (ms_e2e * 1e-3)
        peak = peak_gbs()
        src = PEAK_SOURCE[0]
        # algorithmic bytes with the matrix as it is actually stored (pattern-only CSR: 4 B per nonzero)
        # columns one SpMM launch covers: k unsplit; k/2 when the SLQ step runs its two column groups half a step
        # apart (csrc/slq.cuh, split mode) - derived from the launches counted in the timed region
        cols_per_launch = float(k) * m * args.steps / max(spmm_launches, 1)
        b_spmm = (4.0 if pattern_only else 12.0) * nnz + 4.0 * (n + 1) + 16.0 * n * cols_per_launch
        per_launch_ms = spmm_ms / max(spmm_launches, 1)
        achieved = b_spmm / (per_launch_ms * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "spmm_traffic.json")) as f:
                # measured on one k = 512 launch; a launch over fewer columns moves proportionally less
                traffic = json.load(f).get("dram_bytes_per_launch") * cols_per_launch / 512.0
        except Exception:
            pass
        # bounded CPU sample: the oracle on one core, 4 probes x m steps of the same graph
        cpu_rate, cpu_dt = cpu_slq_rate(A, 4, 1, m)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world),
            "trace_estimate": tr_value, "lambda_scale": lam,
            "clocks": clocks, "numa": numa,
            "e2e": {"value": e2e, "unit": UNIT,
                    "h2d_bytes_per_step": (h1["h2d_bytes"] - h0["h2d_bytes"]) // args.steps,
                    "d2h_bytes_per_step": (h1["d2h_bytes"] - h0["d2h_bytes"]) // args.steps + 8,
                    "ms_per_step": ms_e2e / args.steps, "trace_estimate": tr_e2e},
            # same call path with the probes handed over as int8 signs (kr_slq_trace_sign): 1/8 of the upload
            "e2e_sign_probes": {"value": mv_step * args.steps / (ms_e2e8 * 1e-3), "unit": UNIT,
                                "h2d_bytes_per_step": (g1["h2d_bytes"] - g0["h2d_bytes"]) // args.steps,
                                "ms_per_step": ms_e2e8 / args.steps, "trace_estimate": tr_e2e8},
            "gpu_launches": c1["launches"] - c0["launches"],
            "roofline": {"bound": "hbm", "kernel": "spmm_kernel<EpiDot> (CSR x %d-wide fp64 block + fused alpha dot)" % int(round(cols_per_launch)),
                         "columns_per_launch": cols_per_launch,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": "%s copy bandwidth (MEASURED_PEAKS.json)" % src if src == "measured"
                         else "fallback 6650 GB/s (B200_PROFILING.md)",
                         "algorithmic_bytes_per_launch": b_spmm, "ms_per_launch": per_launch_ms,
                         "launches_timed": spmm_launches,
                         "share_of_step": spmm_ms / ms_dev, "traffic": traffic,
                         # what actually binds on a random power-law graph (DESIGN.md section 5.1): every
                         # (nonzero, column) operand crosses L2 -> SM once; the pure-gather ceiling on a
                         # 128 MB window was measured with scripts/l2_gather.cu
                         "gather": {"bytes_per_launch": 8.0 * nnz * cols_per_launch,
                                    "achieved_tb_per_s": 8.0 * nnz * cols_per_launch / (per_launch_ms * 1e-3) / 1e12,
                                    "microbench_ceiling_tb_per_s": 14.8,
                                    "source": "profiles/r01_l2_gather_microbench.json"}},
            "secondary": secondary, "secondary_c4": secondary_c4, "secondary_c2": secondary_c2, "strong_scaling": strong,
            "cpu_baseline": {"value": cpu_rate, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": "oracle.slq_trace (NumPy/SciPy port of the reference path) on 4 probes x %d steps "
                                       "of the same graph, %.1f s" % (m, cpu_dt)},
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every C3 arm")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before the C3 timing (--impl ours runs at least 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed calls returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
