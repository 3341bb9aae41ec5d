#!/usr/bin/env python
"""Per-candidate values in edge scoring (kr_trace_fun_update_edges_w, kr_greedy_round_w) on the GPU, one JSON line:
  c5_list       the 10^5-candidate C5 list (find_top_missing_edges(..., 'min') on the C3 power-law graph, n = 1M, 20M
                stored entries, spectral radius ~1, exp, tol = 1e-6 e) scored exactly three ways, alternated `--reps`
                times in this one process: random values d_h in [0.5, 1.5] / lam and the uniform d_h = 1 / lam through
                trace_fun_update_edges_w, and the scalar 1 / lam through trace_fun_update_edges_ex.  Uniform against
                scalar is the same work (bitwise the same results), so it isolates the cost of the per-candidate load;
                random values change the step counts.  Edges/s of each run, so the spread is visible next to the
                difference.  Also the screened round (greedy_round_w / greedy_round, screen on) once each.
  grid_greedy   greedy_krylov_weighted on the England power grid ('break', k = 10, Q = 250, the grid's own weights),
                device against the oracle driver (oracle.weighted_edges)
  python scripts/bench_edges_w.py [--out FILE] [--reps 3] [--skip-c5]"""
import argparse, json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def c5_list(kr, reps, ncand):
    from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate
    A = power_law_graph(1_000_000, 20_000_000, 2.2, 20260310)
    lam = spectral_radius_estimate(A, 30)
    A = (A * (1.0 / lam)).tocsr()
    ctx = kr.Context.default(0)
    M = kr.Matrix(A, ctx)
    E = kr.find_top_missing_edges(A, kr.compute_centrality(M, "eig", 1e-10), ncand, "min")
    d = np.random.default_rng(20261022).uniform(0.5, 1.5, len(E)) / lam
    tol = 1e-6 * float(np.exp(1.0))
    kr.trace_fun_update_edges_w(M, E[:4000], d[:4000], tol, 100, "exp")              # warm-up, both flavours
    kr.trace_fun_update_edges(M, E[:4000], 1.0 / lam, tol, 100, "exp")
    du = np.full(len(E), 1.0 / lam)
    runs = {"weighted": [], "uniform_w": [], "scalar": []}
    out = {}
    for _ in range(reps):
        for kind in runs:
            t0 = time.perf_counter()
            if kind == "scalar":
                x, it, _ = kr.trace_fun_update_edges(M, E, 1.0 / lam, tol, 100, "exp")
            else:
                x, it, _ = kr.trace_fun_update_edges_w(M, E, d if kind == "weighted" else du, tol, 100, "exp")
            runs[kind].append(len(E) / (time.perf_counter() - t0))
            out[kind] = (x, it)
    res = {"candidates": int(len(E)), "distinct_nodes": int(np.unique(E).size)}
    for kind, v in runs.items():
        res[kind + "_edges_per_sec"] = v
        res[kind + "_steps_mean"] = float(out[kind][1].mean())
        res[kind + "_edges_per_sec_spread"] = float((max(v) - min(v)) / np.median(v))
    res["uniform_w_over_scalar_median"] = float(np.median(runs["uniform_w"]) / np.median(runs["scalar"]))
    res["weighted_over_scalar_median"] = float(np.median(runs["weighted"]) / np.median(runs["scalar"]))
    res["uniform_values_bitwise_equal_scalar"] = bool(np.array_equal(out["uniform_w"][0], out["scalar"][0]) and
                                                      np.array_equal(out["uniform_w"][1], out["scalar"][1]))
    t0 = time.perf_counter()
    bw, vw, _, _, iw = kr.greedy_round_w(M, E, d, tol, 100, "exp", "make", screen=True)
    res["screened_round_weighted_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    kr.greedy_round(M, E, 1.0 / lam, tol, 100, "exp", "make", screen=True)
    res["screened_round_scalar_s"] = time.perf_counter() - t0
    xw = out["weighted"][0]
    res["screened_weighted_winner_is_exact_winner"] = bool((bw, vw) == kr.select_candidate(xw, "make"))
    res["screened_weighted_info"] = iw
    return res


def grid_greedy(kr, k, Q):
    import oracle as O
    import oracle.weighted_edges as OW
    from conftest import load_graph
    A = load_graph("grid_England").astype(float)
    c = O.compute_centrality(A, "eig")
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-8 * float(np.exp(nrm))
    kr.greedy_krylov_weighted(A, 1, 8, c, "mult", tol, None, "exp", "break")          # warm-up
    t0 = time.perf_counter()
    ed, rd, _, ad = kr.greedy_krylov_weighted(A, k, Q, c, "mult", tol, None, "exp", "break")
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    eo, ro, _, _ = OW.greedy_krylov_weighted(A, k, Q, c, "mult", tol, None, "exp", "break")
    dt_o = time.perf_counter() - t0
    return {"graph": "grid_England", "n": int(A.shape[0]), "nnz": int(A.nnz), "k": k, "Q": Q, "device_s": dt,
            "oracle_s": dt_o, "speedup_vs_oracle": dt_o / dt, "edges": ed.tolist(), "applied": ad.tolist(),
            "same_edges_as_oracle": bool(np.array_equal(ed, eo)), "rob_variation": float(rd),
            "rel_diff_rob_vs_oracle": float(abs(rd - ro) / abs(ro))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ncand", type=int, default=100_000)
    ap.add_argument("--skip-c5", action="store_true")
    args = ap.parse_args()
    import krylov_robustness_b200 as kr
    res = {"gpu": gpu_info()}
    res["grid_greedy"] = grid_greedy(kr, 10, 250)
    if not args.skip_c5:
        res["c5_list"] = c5_list(kr, args.reps, args.ncand)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
