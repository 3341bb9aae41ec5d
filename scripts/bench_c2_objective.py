#!/usr/bin/env python
"""Config C2 objective (BASELINE.json configs[1]) on one B200: f = -(tr sinh(Ã) - tr sinh(A)) over all edges of a road
network, by the Gauss-Legendre quadrature of kr_trace_fun_sparse_update, against the SLQ estimate of bench_c2.py.

  python scripts/bench_c2_objective.py [--graph transport_Vermont] [--repeat 5] [--probes 64]

The inputs are those of bench_c2.py: A <- A / max(A), Omega = all lower-triangular edges, X = 0.1 * A_Omega * uniform(0,1)
(seed 4), tol = 1e-8 * cosh(normest(A)).  Timed, each call ended by a device synchronise, median of --repeat after one
warm-up call of the same shape:
  * gradient alone:          fun_and_grad_all_edges(X, A, Omega, sinh, cosh, tol, 100)
  * objective + gradient:    the same call with objective=True (one upload of Ã for both)
  * objective alone:         trace_fun_sparse_update on a prebuilt device copy of Ã
  * SLQ objective:           two slq_trace calls (common Rademacher probes, 40 steps) as in bench_c2.py
It reports q, the step count, the columns per budget tier of the local path and those through the dense batch, and
how far the SLQ estimate is from the quadrature value.  Prints one JSON line (and writes it to --out if given).
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_description():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(ctx, fn, repeat):
    out, ts = None, []
    for _ in range(repeat):
        t0 = time.perf_counter()
        out = fn()
        ctx.sync()
        ts.append(time.perf_counter() - t0)
    return out, float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graph", default="transport_Vermont")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--probes", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    warnings.simplefilter("ignore")
    import krylov_robustness_b200 as kr
    from conftest import load_graph
    A = load_graph(args.graph).astype(np.float64)
    A = (A / A.max()).tocsr()
    n = A.shape[0]
    L = sp.tril(A, -1).tocoo()
    Om = np.stack([L.row + 1, L.col + 1], 1).astype(np.int64)
    X = 0.1 * L.data * np.random.default_rng(4).random(L.nnz)
    ctx = kr.Context.default()
    nrm = float(kr.normest(A, 1e-2)[0])
    tol = 1e-8 * float(np.cosh(nrm))
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (A + D + D.T).tocsr()
    out = {"workload": "C2 objective: %s, trace sinh change over all %d edges" % (args.graph, Om.shape[0]),
           "gpu": gpu_description(), "n": n, "edges": int(Om.shape[0]), "tol": tol, "repeat": args.repeat}
    # warm-up of every timed shape
    kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100, objective=True)
    ctx.sync()
    gr, out["gradient_s"], out["gradient_s_all"] = timed(
        ctx, lambda: kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100), args.repeat)
    (f, gr2), out["objective_and_gradient_s"], out["objective_and_gradient_s_all"] = timed(
        ctx, lambda: kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100, objective=True), args.repeat)
    out["gradient_bitwise_equal"] = bool(np.array_equal(gr, gr2))
    Mt = kr.Matrix(At, ctx)
    res, out["objective_prebuilt_matrix_s"], _ = timed(
        ctx, lambda: kr.trace_fun_sparse_update(Mt, X, Om, "sinh", tol, 100, return_info=True), args.repeat)
    dtr, q, it, info = res
    out.update({"objective": f, "objective_equal_to_direct_call": bool(-dtr == f), "q": q, "iter": it,
                "tier_columns": info["tier_columns"], "dense_columns": info["dense_columns"],
                "columns": int(q * np.unique(Om[:, 0]).size)})
    Z = kr.rademacher_host(n, args.probes, 9)
    kr.slq_trace(At, Z, 40, "sinh")
    f_slq, out["objective_slq_s"], _ = timed(
        ctx, lambda: -(kr.slq_trace(At, Z, 40, "sinh") - kr.slq_trace(A, Z, 40, "sinh")), args.repeat)
    out["objective_slq"] = f_slq
    out["slq_minus_quadrature"] = f_slq - f
    out["slq_rel_err"] = abs(f_slq - f) / abs(f)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
