#!/usr/bin/env python
"""One call of one entry point on one of the reference's graphs (for launch lists):
  python scripts/one_call.py fun_and_grad|tfu_rank2|edges250|centrality|normest|tfu_set [graph]"""
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
warnings.simplefilter("ignore")


def main():
    import krylov_robustness_b200 as kr
    import oracle as O
    from conftest import load_graph
    what = sys.argv[1]
    name = sys.argv[2] if len(sys.argv) > 2 else "grid_England"
    A = load_graph(name)
    A = (A / A.max()).tocsr()
    n = A.shape[0]
    M = kr.Matrix(A)
    c = O.compute_centrality(A, "eig")
    nrm = float(O.normest(A, 1e-2)[0])
    E = O.find_top_edges(A, c, 100, "min")
    tol_df = 1e-6 * float(np.cosh(nrm))
    vals, _ = O.function_multiple_entries(A, E, "cosh", tol_df, 100)
    ind = np.argsort(-vals, kind="stable")[:30]
    Om, dfA = E[ind], vals[ind]
    x = 0.05 * np.ones(30)
    tol = 1e-6 * float(np.sinh(nrm))
    calls = {
        "fun_and_grad": lambda: kr.fun_and_grad_krylov_fun(x, M, Om, "sinh", "cosh", dfA, tol, 100),
        "tfu_rank2": lambda: kr.trace_fun_update(M, *O.edge2low_rank(Om[:1], n, 1.0)[:2], tol, 100, 0, "sinh"),
        "tfu_set": lambda: kr.trace_fun_update(M, *O.edge2low_rank(Om[:10], n, 1.0)[:2], tol, 100, 0, "sinh"),
        "edges250": lambda: kr.trace_fun_update_edges(M, O.find_top_edges(A, c, 250, "min"), -1.0, tol, 100, "sinh"),
        "centrality": lambda: kr.compute_centrality(M, "eig"),
        "normest": lambda: kr.normest(M, 1e-2),
    }
    f = calls[what]
    f()                       # warm-up: attribute setup, pool allocations
    M.ctx.sync()
    c0 = M.ctx.counters()
    t0 = time.perf_counter()
    f()
    M.ctx.sync()
    dt = time.perf_counter() - t0
    c1 = M.ctx.counters()
    print("%s on %s: %.3f ms, %d launches" % (what, name, dt * 1e3, c1["launches"] - c0["launches"]))


if __name__ == "__main__":
    main()
