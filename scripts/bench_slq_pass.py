#!/usr/bin/env python
"""The SLQ pass on an int8 sign panel against the same probes as fp64, on the C3 workload (power-law n = 1M,
nnz = 20M, 512 Rademacher probes), one JSON line.  Alternated `--reps` times in this one process:
  step0_spmm   the step-0 SpMM (spmm_kernel<EpiDotT<signed char, true>> against <double, true>): per-launch time
               from the library's SpMM events, m = 1 with alpha / beta asked for (so Y is stored, as at step 0 of a
               whole pass)
  pass         one whole pass, m = 30, vals only (what bench.py times as `value`): a block filled by
               kr_dense_fill_rademacher (sign panel) against the same values uploaded as fp64 (no sign panel),
               CUDA events around the call
The per-probe values of every pair of runs must agree to the bit.
  python scripts/bench_slq_pass.py [--out FILE] [--reps 3]"""
import argparse, ctypes as C, json, os, subprocess, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import krylov_robustness_b200 as kr
    from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate
    A = power_law_graph(1_000_000, 20_000_000, 2.2, 20260310)
    lam = spectral_radius_estimate(A, 30)
    A = (A * (1.0 / lam)).tocsr()
    n, k = A.shape[0], 512
    ctx = kr.Context.default(0)
    M = kr.Matrix(A, ctx)
    Zs = kr.Dense(n, k, ctx).fill_rademacher(1)
    Zh = np.empty((n, k), order="F")                 # the same values as fp64, through the host
    for c0 in range(0, k, 64):
        Zh[:, c0:c0 + 64] = kr.Dense(n, 64, ctx).fill_rademacher(1, col_offset=c0).download()
    Zf = kr.Dense(n, k, ctx).upload(Zh)
    del Zh
    stream = torch.cuda.ExternalStream(ctx.stream())

    def call(Z, m, want_ab):
        tr = C.c_double()
        vals = np.empty(k)
        al = np.empty((m, k), order="F") if want_ab else None
        be = np.empty((m, k), order="F") if want_ab else None
        p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        assert ctx.lib.kr_slq_trace_dev(ctx.h, M.h, Z.h, m, 0, C.byref(tr), p(vals), p(al), p(be)) == 0
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), vals

    for Z in (Zs, Zf):                                # warm-up: every kernel flavour of both paths
        call(Z, 1, True)
        call(Z, 30, False)
    runs = {"step0_spmm_sign_ms": [], "step0_spmm_fp64_ms": [], "pass_sign_ms": [], "pass_fp64_ms": []}
    bitwise = True
    for _ in range(args.reps):
        v = {}
        for name, Z in (("sign", Zs), ("fp64", Zf)):
            ctx.set_timing(True)
            ctx.spmm_time(reset=True)
            _, v["s0" + name] = call(Z, 1, True)
            ms, launches = ctx.spmm_time(reset=True)
            ctx.set_timing(False)
            assert launches == 1
            runs["step0_spmm_%s_ms" % name].append(ms)
        for name, Z in (("sign", Zs), ("fp64", Zf)):
            ms, v["p" + name] = call(Z, 30, False)
            runs["pass_%s_ms" % name].append(ms)
        bitwise &= bool(np.array_equal(v["s0sign"].view(np.int64), v["s0fp64"].view(np.int64)))
        bitwise &= bool(np.array_equal(v["psign"].view(np.int64), v["pfp64"].view(np.int64)))
    med = {key: float(np.median(x)) for key, x in runs.items()}
    line = {"gpu": gpu_info(), "workload": "C3: power-law n=1000000 nnz=20000000, 512 probes, m=30, exp",
            "reps": args.reps, "runs": runs, "median": med, "bitwise_equal_vals": bitwise,
            "step0_spmm_speedup": med["step0_spmm_fp64_ms"] / med["step0_spmm_sign_ms"],
            "pass_speedup": med["pass_fp64_ms"] / med["pass_sign_ms"]}
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
