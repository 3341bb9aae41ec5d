#!/usr/bin/env python
"""Node-removal scoring (kr_trace_fun_update_nodes, csrc/nodes.cuh) on the GPU, three measurements in one JSON line:
  c3_nodes      candidate nodes scored per second: the 4096 top-centrality nodes of the C3 power-law graph
                (n = 1M, 20M stored entries, scaled to spectral radius ~1, exp, tol = 1e-12 * e)
  a7_round      one node-removal round on Oregon A7: the Q = 250 top-centrality nodes, device against the oracle
  a0_greedy     greedy_krylov_nodes with k = 10, Q = 250 on Oregon A0, device against the oracle
  python scripts/bench_nodes.py [--out FILE] [--skip-c3]"""
import argparse, json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def hist(it):
    return {int(k): int(v) for k, v in zip(*np.unique(it, return_counts=True))}


def c3_nodes(kr, count):
    from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate
    A = power_law_graph(1_000_000, 20_000_000, 2.2, 20260310)
    lam = spectral_radius_estimate(A, 30)
    A = (A * (1.0 / lam)).tocsr()
    ctx = kr.Context.default(0)
    M = kr.Matrix(A, ctx)
    c = kr.compute_centrality(M, "eig", 1e-10)
    V = np.argsort(-c, kind="stable")[:count] + 1
    tol = 1e-12 * float(np.exp(1.0))
    kr.trace_fun_update_nodes(M, V[:64], tol, 100, "exp")            # warm-up (allocations, attributes)
    ctx.set_timing(True)
    ctx.spmm_time(reset=True)
    c0 = ctx.counters()
    t0 = time.perf_counter()
    x, it, lk = kr.trace_fun_update_nodes(M, V, tol, 100, "exp")
    dt = time.perf_counter() - t0
    ms, nl = ctx.spmm_time(reset=True)
    ctx.set_timing(False)
    c1 = ctx.counters()
    again = kr.trace_fun_update_nodes(M, V, tol, 100, "exp")
    return {"nodes": int(V.size), "seconds": dt, "nodes_per_sec": V.size / dt, "steps_histogram": hist(it),
            "lucky": int(lk.sum()), "spmm_ms": ms, "spmm_launches": nl, "spmm_share": ms * 1e-3 / dt,
            "launches": c1["launches"] - c0["launches"], "matvecs": c1["matvecs"] - c0["matvecs"],
            "repeat_bit_identical": bool(np.array_equal(x, again[0]) and np.array_equal(it, again[1])),
            "best_node": int(V[int(np.argmin(x))]), "best_value": float(np.min(x))}


def a7_round(kr, O, ON, load_graph, Q):
    A = load_graph("oregon_A7").astype(float)
    c = O.compute_centrality(A, "eig")
    V = np.argsort(-c, kind="stable")[:Q] + 1
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-12 * float(np.exp(nrm))
    M = kr.Matrix(A)
    kr.trace_fun_update_nodes(M, V[:16], tol, 100, "exp")
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        x, it, lk = kr.trace_fun_update_nodes(M, V, tol, 100, "exp")
    dt = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    ref = [ON.trace_fun_update_node(A, int(v), tol, 100, "exp") for v in V]
    dt_o = time.perf_counter() - t0
    xo = np.array([r[0] for r in ref])
    return {"n": int(A.shape[0]), "nnz": int(A.nnz), "Q": int(Q), "device_ms": dt * 1e3, "oracle_ms": dt_o * 1e3,
            "speedup_vs_oracle": dt_o / dt, "steps_histogram": hist(it),
            "max_rel_diff_vs_oracle": float(np.max(np.abs(x - xo) / np.abs(xo))),
            "iter_equal": bool(np.array_equal(it, [r[1] for r in ref])),
            "same_best": bool(int(np.argmin(x)) == int(np.argmin(xo)))}


def a0_greedy(kr, O, ON, load_graph, k, Q):
    A = load_graph("oregon_A0").astype(float)
    c = O.compute_centrality(A, "eig")
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-12 * float(np.exp(nrm))
    kr.greedy_krylov_nodes(A, 1, 8, c, tol, None, "exp")               # warm-up
    t0 = time.perf_counter()
    nd, rd, _ = kr.greedy_krylov_nodes(A, k, Q, c, tol, None, "exp")
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    no, ro, _ = ON.greedy_krylov_nodes(A, k, Q, c, tol, None, "exp")
    dt_o = time.perf_counter() - t0
    return {"n": int(A.shape[0]), "k": k, "Q": Q, "device_s": dt, "oracle_s": dt_o, "speedup_vs_oracle": dt_o / dt,
            "nodes": [int(v) for v in nd], "same_nodes_as_oracle": bool(list(nd) == list(no)),
            "rob_variation": float(rd), "rel_diff_rob_vs_oracle": float(abs(rd - ro) / abs(ro))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--nodes", type=int, default=4096)
    ap.add_argument("--skip-c3", action="store_true")
    args = ap.parse_args()
    import krylov_robustness_b200 as kr
    import oracle as O
    import oracle.nodes as ON
    from conftest import load_graph
    res = {"gpu": gpu_info()}
    res["a7_round"] = a7_round(kr, O, ON, load_graph, 250)
    res["a0_greedy"] = a0_greedy(kr, O, ON, load_graph, 10, 250)
    if not args.skip_c3:
        res["c3_nodes"] = c3_nodes(kr, args.nodes)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
