#!/usr/bin/env python
"""Hessian-vector product of the config C2 callbacks (kr_frechet_hessian_multiply) on one B200, with the gradient and
the objective of the same inputs timed in the same process, and the product against hessianfcn_fun + a matmul on
Anaheim's 634 edges.

  python scripts/bench_c2_hessp.py [--graph transport_Vermont] [--pairs 0] [--repeat 5] [--out FILE]

The inputs are those of bench_c2.py: A <- A / max(A), Omega = all lower-triangular edges, X = 0.1 * A_Omega * uniform(0,1)
(seed 4), tol = 1e-8 * cosh(normest(A)); Y is standard normal (seed 5) with p = 1 and p = 8.  --pairs k > 0 runs the
product on the first k rows of Omega only (Atilde still carries all of X).  Timed, each call ended by a device
synchronise, median of --repeat after one warm-up call of the same shape.  Prints one JSON line (and writes it to --out).
"""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_c2_objective import gpu_description, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graph", default="transport_Vermont")
    ap.add_argument("--pairs", type=int, default=0)
    ap.add_argument("--repeat", type=int, default=5)
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
    tol = 1e-8 * float(np.cosh(float(kr.normest(A, 1e-2)[0])))
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (A + D + D.T).tocsr()
    Mt = kr.Matrix(At, ctx)
    k = args.pairs if args.pairs > 0 else Om.shape[0]
    Omk = Om[:k]
    out = {"workload": "C2 Hessian-vector product: %s, %d of %d edges" % (args.graph, k, Om.shape[0]),
           "gpu": gpu_description(), "n": n, "edges": int(Om.shape[0]), "pairs": k, "tol": tol, "repeat": args.repeat}
    kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100)
    ctx.sync()
    _, out["gradient_s"], _ = timed(ctx, lambda: kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100),
                                    args.repeat)
    kr.trace_fun_sparse_update(Mt, X, Om, "sinh", tol, 100)
    _, out["objective_s"], _ = timed(ctx, lambda: kr.trace_fun_sparse_update(Mt, X, Om, "sinh", tol, 100), args.repeat)
    rng = np.random.default_rng(5)
    for p in (1, 8):
        Y = rng.standard_normal((k, p))
        kr.hessp_all_edges(None, Mt, Omk, "cosh", Y, tol, 100)
        res, t, ts = timed(ctx, lambda: kr.hessp_all_edges(None, Mt, Omk, "cosh", Y, tol, 100, return_info=True),
                           args.repeat)
        W, it, info = res
        out["hessp_p%d_s" % p] = t
        out["hessp_p%d_s_all" % p] = ts
        out["hessp_p%d_iter" % p] = it
        out["hessp_p%d_tier_pairs" % p] = info["tier_pairs"]
        out["hessp_p%d_dense_pairs" % p] = info["dense_pairs"]
        out["hessp_p%d_max_abs" % p] = float(np.abs(W).max())
    # Anaheim, all 634 edges: the product against the assembled reference Hessian followed by a matmul
    An = load_graph("transport_Anaheim").astype(np.float64)
    An = (An / An.max()).tocsr()
    La = sp.tril(An, -1).tocoo()
    Oa = np.stack([La.row + 1, La.col + 1], 1).astype(np.int64)
    Xa = 0.1 * La.data * np.random.default_rng(4).random(La.nnz)
    tola = 1e-8 * float(np.cosh(float(kr.normest(An, 1e-2)[0])))
    ya = rng.standard_normal(len(Oa))
    kr.hessp_all_edges(Xa, An, Oa, "cosh", ya, tola, 100, reference_form=True)
    Wa, out["anaheim_hessp_s"], _ = timed(
        ctx, lambda: kr.hessp_all_edges(Xa, An, Oa, "cosh", ya, tola, 100, reference_form=True), args.repeat)
    kr.hessianfcn_fun(Xa, An, Oa, "cosh", tola, 100)
    Ha, out["anaheim_hessianfcn_matmul_s"], _ = timed(
        ctx, lambda: kr.hessianfcn_fun(Xa, An, Oa, "cosh", tola, 100) @ ya, args.repeat)
    out["anaheim_edges"] = int(len(Oa))
    out["anaheim_rel_gap"] = float(np.abs(Wa - Ha).max() / np.abs(Ha).max())
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
