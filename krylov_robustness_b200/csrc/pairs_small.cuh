// pairs_small.cuh - the candidate loop of functions/krylov_miobi.m:76-99 (trace_fun_update on U = [e_i e_j],
// functions/trace_fun_update.m:60-125 over functions/lanczos_krylov.m:73-101) for graphs whose CSR is L2-resident
// (the reference's own data sets: Oregon AS graphs, road networks, power grids - config C1 of BASELINE.json).
//
// On those graphs the batched path of pairs.cuh is launch-bound: ~10 launches and one host synchronisation per
// block-Lanczos step.  Here the WHOLE evaluation of a candidate - seed, every block-Lanczos step (product, CGS2,
// QR-from-Gram, projected eigen-solves, lag-2 stop) - runs inside ONE persistent CTA, candidates are handed out by
// a ticket counter, and a scoring round is ONE kernel launch and ONE device-to-host copy.  The arithmetic is the
// batched path's, function for function (pair_coef1_math / pair_coef2_math / pair_qr_from_gram /
// pair_projected_trace are shared); only the summation order of the Gram reductions differs (fixed, so results are
// bit-reproducible run to run).
//
// Per-CTA work space in global memory (L1/L2 resident): three n x 2 blocks P (previous), C (current), Y (work),
// one double2 per row.
#pragma once
#include "pairs.cuh"

namespace kr {

constexpr int PS_THREADS = 512;
constexpr int PS_WARPS = PS_THREADS / 32;
constexpr int PS_ILP = 4;               // rows per lane group kept in flight in the product
constexpr int PS_RLP = 2;               // rows per thread kept in flight in the streaming passes
constexpr int PS_SMEM_NN = 48;          // projections up to 48 x 48 (24 block steps) live in shared memory
constexpr size_t PS_DYN_SMEM = (size_t)(2 * PS_SMEM_NN * (PS_SMEM_NN | 1) + 2 * PS_SMEM_NN) * sizeof(double);

struct PairSmallArgs {
    CsrDevView A;
    int rows_cta, rows_warp;            // stored rows [0, rows_cta): whole CTA each; next rows_warp: a warp each; rest: 4 lanes
    const int* ei;                      // [np] 0-based end points
    const int* ej;
    int np, it, fun;
    double tol, b_off;
    double2* ws;                        // [ctas][3][n]
    double* hbuf;                       // [ctas][3][it][4]: Hd, Hs, Hr
    double* gscratch;                   // [ctas][gstride] projected matrices once 2j > PS_SMEM_NN (may be null if it is small)
    int64_t gstride;
    int* ticket;
    double* res_Xm;
    long long* res_iter;
    int* res_lucky;
};

// fixed-order CTA sum of NV per-thread values; totals land in out[0..NV) (shared), valid after the trailing barrier
template <int NV>
__device__ __forceinline__ void ps_reduce(double (&v)[NV], double (*wred)[8], double* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = v[i];
        for (int off = 16; off; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
        v[i] = x;
    }
    __syncthreads();                                   // wred / out may still be read from the previous use
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < NV; ++i) wred[warp][i] = v[i];
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0.0;
        for (int w = 0; w < PS_WARPS; ++w) s += wred[w][threadIdx.x];
        out[threadIdx.x] = s;
    }
    __syncthreads();
}

// Y = A * X for the CTA's n x 2 block (X, Y indexed by ORIGINAL row).  Rows are stored by decreasing length.
__device__ __forceinline__ void ps_spmv2(const PairSmallArgs& a, const double2* __restrict__ X, double2* __restrict__ Y,
                                         double* red2) {
    const CsrDevView& A = a.A;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool hv = A.val != nullptr;
    const double uv = A.uval;
    // ---- the few hub rows: whole CTA per row
    for (int s = 0; s < a.rows_cta; ++s) {
        const int p0 = A.row_ptr[s], p1 = A.row_ptr[s + 1];
        double ax = 0.0, ay = 0.0;
#pragma unroll 4
        for (int p = p0 + tid; p < p1; p += PS_THREADS) {
            const double2 x = X[A.col[p]];
            const double v = hv ? A.val[p] : 1.0;
            ax = fma(v, x.x, ax);
            ay = fma(v, x.y, ay);
        }
        for (int off = 16; off; off >>= 1) {
            ax += __shfl_xor_sync(0xffffffffu, ax, off);
            ay += __shfl_xor_sync(0xffffffffu, ay, off);
        }
        __syncthreads();
        if (lane == 0) { red2[2 * warp] = ax; red2[2 * warp + 1] = ay; }
        __syncthreads();
        if (tid == 0) {
            double sx = 0.0, sy = 0.0;
            for (int w = 0; w < PS_WARPS; ++w) { sx += red2[2 * w]; sy += red2[2 * w + 1]; }
            if (!hv) { sx *= uv; sy *= uv; }
            Y[A.row_order[s]] = make_double2(sx, sy);
        }
    }
    // ---- medium rows: a warp per row
    const int m1 = a.rows_cta + a.rows_warp;
    for (int s = a.rows_cta + warp; s < m1; s += PS_WARPS) {
        const int p0 = A.row_ptr[s], p1 = A.row_ptr[s + 1];
        double ax = 0.0, ay = 0.0;
#pragma unroll 4
        for (int p = p0 + lane; p < p1; p += 32) {
            const double2 x = X[A.col[p]];
            const double v = hv ? A.val[p] : 1.0;
            ax = fma(v, x.x, ax);
            ay = fma(v, x.y, ay);
        }
        for (int off = 16; off; off >>= 1) {
            ax += __shfl_xor_sync(0xffffffffu, ax, off);
            ay += __shfl_xor_sync(0xffffffffu, ay, off);
        }
        if (lane == 0) {
            if (!hv) { ax *= uv; ay *= uv; }
            Y[A.row_order[s]] = make_double2(ax, ay);
        }
    }
    // ---- short rows: four lanes per row, PS_ILP rows of a lane group in flight at once (the chain row pointer ->
    // column index -> X row is three dependent L2 accesses; one CTA per SM cannot hide them with warps alone)
    const int sub = lane & 3;
    constexpr int G = PS_THREADS / 4;                     // lane groups per CTA
    for (int base = m1 + warp * 8; base < A.n; base += G * PS_ILP) {
        int q0[PS_ILP], q1[PS_ILP];
        double ax[PS_ILP], ay[PS_ILP];
        int maxlen = 0;
#pragma unroll
        for (int u = 0; u < PS_ILP; ++u) {
            const int s = base + u * G + (lane >> 2);
            q0[u] = q1[u] = 0;
            ax[u] = ay[u] = 0.0;
            if (s < A.n) {
                q0[u] = A.row_ptr[s];
                q1[u] = A.row_ptr[s + 1];
            }
            maxlen = max(maxlen, q1[u] - q0[u]);
        }
        for (int off = sub; off < maxlen; off += 4) {
#pragma unroll
            for (int u = 0; u < PS_ILP; ++u) {
                const int p = q0[u] + off;
                if (p < q1[u]) {
                    const double2 x = X[A.col[p]];
                    const double v = hv ? A.val[p] : 1.0;
                    ax[u] = fma(v, x.x, ax[u]);
                    ay[u] = fma(v, x.y, ay[u]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < PS_ILP; ++u) {
            const int s = base + u * G + (lane >> 2);
            double bx = ax[u], by = ay[u];
            bx += __shfl_xor_sync(0xffffffffu, bx, 1);
            by += __shfl_xor_sync(0xffffffffu, by, 1);
            bx += __shfl_xor_sync(0xffffffffu, bx, 2);
            by += __shfl_xor_sync(0xffffffffu, by, 2);
            if (sub == 0 && s < A.n) {
                if (!hv) { bx *= uv; by *= uv; }
                Y[A.row_order[s]] = make_double2(bx, by);
            }
        }
    }
    __syncthreads();
    // ---- pending edge edits (kr_matrix_set_edges): A = stored CSR + delta entries, sorted by stored row; the thread
    // that owns the first entry of a row walks the row's run
    for (int e = tid; e < A.dl_count; e += PS_THREADS) {
        const int pos = A.dl_pos[e];
        if (e > 0 && A.dl_pos[e - 1] == pos) continue;
        const int r = A.row_order[pos];
        double2 y = Y[r];
        for (int q = e; q < A.dl_count && A.dl_pos[q] == pos; ++q) {
            const double2 x = X[A.dl_col[q]];
            const double d = A.dl_val[q];
            y.x = fma(d, x.x, y.x);
            y.y = fma(d, x.y, y.y);
        }
        Y[r] = y;
    }
    if (A.dl_count > 0) __syncthreads();
}

__global__ void __launch_bounds__(PS_THREADS, 1)
pair_small_kernel(PairSmallArgs a) {
    extern __shared__ double dyn[];
    __shared__ JacobiShared sh;
    __shared__ double wred[PS_WARPS][8];
    __shared__ double gsum[8];
    __shared__ double cf[12], Tp[4], Tc[4], Tn[4], hp[4], hc[4], aij[3], Xs[2];
    __shared__ int s_cand, s_lucky, s_done;
    const CsrDevView& A = a.A;
    const int n = A.n, tid = threadIdx.x;
    double2* P = a.ws + (size_t)blockIdx.x * 3 * n;
    double2* C = P + n;
    double2* Y = C + n;
    double* Hd = a.hbuf + (size_t)blockIdx.x * 3 * a.it * 4;
    double* Hs = Hd + (size_t)a.it * 4;
    double* Hr = Hs + (size_t)a.it * 4;
    double* gwork = a.gscratch ? a.gscratch + (size_t)blockIdx.x * a.gstride : nullptr;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_cand = atomicAdd(a.ticket, 1);
        __syncthreads();
        const int cand = s_cand;
        if (cand >= a.np) break;
        const int i = a.ei[cand], j = a.ej[cand];
        // ------------------------------------------------------------------ step 1 from the CSR rows of i and j
        // P = [e_i e_j], C = W1 = A(:, [i j]) with rows i, j zeroed (= A*U - U*(U'AU): the second CGS pass finds
        // exactly zero coefficients, lanczos_krylov.m:86-88), hc = U'AU
        for (int r = tid; r < n; r += PS_THREADS) {
            P[r] = make_double2(0.0, 0.0);
            C[r] = make_double2(0.0, 0.0);
        }
        if (tid < 3) aij[tid] = 0.0;
        __syncthreads();
        {
            const int si = A.row_pos[i], sj = A.row_pos[j];
            double* Cd = reinterpret_cast<double*>(C);
            for (int p = A.row_ptr[si] + tid; p < A.row_ptr[si + 1]; p += PS_THREADS) {
                const int r = A.col[p];
                const double v = A.val ? A.val[p] : A.uval;
                if (r == i) aij[0] = v;
                else if (r == j) aij[1] = v;
                else Cd[2 * (size_t)r] = v;
            }
            for (int p = A.row_ptr[sj] + tid; p < A.row_ptr[sj + 1]; p += PS_THREADS) {
                const int r = A.col[p];
                const double v = A.val ? A.val[p] : A.uval;
                if (r == j) aij[2] = v;
                else if (r != i) Cd[2 * (size_t)r + 1] = v;
            }
            __syncthreads();
            if (tid == 0) {
                for (int side = 0; side < 2 && A.dl_count > 0; ++side) {          // pending edits of the two rows
                    const int pos = side == 0 ? si : sj;
                    int lo = 0, hi = A.dl_count;
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (A.dl_pos[mid] < pos) lo = mid + 1; else hi = mid; }
                    for (int e = lo; e < A.dl_count && A.dl_pos[e] == pos; ++e) {
                        const int r = A.dl_col[e];
                        const double d = A.dl_val[e];
                        if (r == i || r == j) {
                            if (side == 0 && r == i) aij[0] += d;
                            else if (side == 1 && r == j) aij[2] += d;
                            else if (side == 0) aij[1] += d;                       // the (j, i) twin carries the same delta
                        } else {
                            Cd[2 * (size_t)r + side] += d;
                        }
                    }
                }
                reinterpret_cast<double*>(P)[2 * (size_t)i] = 1.0;
                reinterpret_cast<double*>(P)[2 * (size_t)j + 1] = 1.0;
                hc[0] = aij[0]; hc[1] = aij[1]; hc[2] = aij[1]; hc[3] = aij[2];
                for (int k = 0; k < 4; ++k) {
                    hp[k] = 0.0;
                    Tp[k] = Tc[k] = (k == 0 || k == 3) ? 1.0 : 0.0;
                }
                Xs[0] = Xs[1] = 0.0;
            }
            __syncthreads();
        }
        double2* W = C;                                  // the block the step routine factorises
        int step = 0;
        for (;;) {
            if (step > 0) {
                // -------------------------------------------------------------- one dense block-Lanczos step
                ps_spmv2(a, C, Y, &wred[0][0]);                                       // pass A: Y = A*C
                double acc[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] = 0.0;
                for (int r0 = tid; r0 < n; r0 += PS_THREADS * PS_RLP) {               //         raw Grams P'Y, C'Y
                    double2 y[PS_RLP], p[PS_RLP], c[PS_RLP];
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        const int r = r0 + u * PS_THREADS;
                        if (r < n) { y[u] = Y[r]; p[u] = P[r]; c[u] = C[r]; }
                    }
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        if (r0 + u * PS_THREADS < n) {
                            acc[0] += p[u].x * y[u].x; acc[1] += p[u].x * y[u].y; acc[2] += p[u].y * y[u].x; acc[3] += p[u].y * y[u].y;
                            acc[4] += c[u].x * y[u].x; acc[5] += c[u].x * y[u].y; acc[6] += c[u].y * y[u].x; acc[7] += c[u].y * y[u].y;
                        }
                    }
                }
                ps_reduce<8>(acc, wred, gsum);
                if (tid == 0) pair_coef1_math(gsum, Tp, Tc, cf, hp, hc);
                __syncthreads();
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] = 0.0;
                for (int r0 = tid; r0 < n; r0 += PS_THREADS * PS_RLP) {               // pass B: first CGS update + Grams
                    double2 yv[PS_RLP], pv[PS_RLP], cv[PS_RLP];
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        const int r = r0 + u * PS_THREADS;
                        if (r < n) { yv[u] = Y[r]; pv[u] = P[r]; cv[u] = C[r]; }
                    }
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        const int r = r0 + u * PS_THREADS;
                        if (r < n) {
                            const double2 y = yv[u], p = pv[u], c = cv[u];
                            double2 w;
                            w.x = y.x * cf[0] + y.y * cf[2] - (p.x * cf[4] + p.y * cf[6]) - (c.x * cf[8] + c.y * cf[10]);
                            w.y = y.x * cf[1] + y.y * cf[3] - (p.x * cf[5] + p.y * cf[7]) - (c.x * cf[9] + c.y * cf[11]);
                            Y[r] = w;
                            acc[0] += p.x * w.x; acc[1] += p.x * w.y; acc[2] += p.y * w.x; acc[3] += p.y * w.y;
                            acc[4] += c.x * w.x; acc[5] += c.x * w.y; acc[6] += c.y * w.x; acc[7] += c.y * w.y;
                        }
                    }
                }
                ps_reduce<8>(acc, wred, gsum);
                if (tid == 0) pair_coef2_math(gsum, Tp, Tc, cf, hp, hc);
                __syncthreads();
                W = Y;
            }
            double g[3] = {0.0, 0.0, 0.0};
            if (step > 0) {
                for (int r0 = tid; r0 < n; r0 += PS_THREADS * PS_RLP) {               // pass C: second CGS update + W'W
                    double2 yv[PS_RLP], pv[PS_RLP], cv[PS_RLP];
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        const int r = r0 + u * PS_THREADS;
                        if (r < n) { yv[u] = Y[r]; pv[u] = P[r]; cv[u] = C[r]; }
                    }
#pragma unroll
                    for (int u = 0; u < PS_RLP; ++u) {
                        const int r = r0 + u * PS_THREADS;
                        if (r < n) {
                            const double2 y = yv[u], p = pv[u], c = cv[u];
                            double2 w;
                            w.x = y.x - (p.x * cf[4] + p.y * cf[6]) - (c.x * cf[8] + c.y * cf[10]);
                            w.y = y.y - (p.x * cf[5] + p.y * cf[7]) - (c.x * cf[9] + c.y * cf[11]);
                            Y[r] = w;
                            g[0] += w.x * w.x; g[1] += w.x * w.y; g[2] += w.y * w.y;
                        }
                    }
                }
            } else {
                for (int r = tid; r < n; r += PS_THREADS) {                           // Gram of W1
                    const double2 w = C[r];
                    g[0] += w.x * w.x; g[1] += w.x * w.y; g[2] += w.y * w.y;
                }
            }
            ps_reduce<3>(g, wred, gsum);
            // ------------------------------------------------------------------ QR from the Gram, H, projections, stop
            const int jj = step + 1;
            if (tid == 0) {
                double R[4], T[4];
                double* w1 = reinterpret_cast<double*>(W);
                pair_qr_from_gram(gsum[0], gsum[1], gsum[2], w1, w1 + 1, 2, n, R, T);
                for (int k = 0; k < 4; ++k) {
                    Tn[k] = T[k];
                    Hd[(jj - 1) * 4 + k] = hc[k];
                    Hs[(jj - 1) * 4 + k] = hp[k];
                    Hr[(jj - 1) * 4 + k] = R[k];
                }
                s_lucky = sqrt(R[0] * R[0] + R[1] * R[1] + R[2] * R[2] + R[3] * R[3]) < 1e-8;   // lanczos_krylov.m:91
            }
            __syncthreads();
            double* work = 2 * jj <= PS_SMEM_NN ? dyn : gwork;
            const double Xm = pair_projected_trace<PS_THREADS>(Hd, Hs, Hr, jj, a.b_off, a.fun, work, &sh);
            if (tid == 0) {
                bool done = false;
                if (jj <= 2) {
                    Xs[jj - 1] = Xm;
                } else {
                    const double err = fabs(Xm - Xs[0]);                              // trace_fun_update.m:104-118
                    if (err < a.tol) done = true;
                    else { Xs[0] = Xs[1]; Xs[1] = Xm; }
                }
                if (!done && s_lucky) done = true;
                if (jj == a.it) done = true;
                a.res_Xm[cand] = Xm;
                a.res_iter[cand] = jj;
                a.res_lucky[cand] = s_lucky;
                s_done = done;
                for (int k = 0; k < 4; ++k) { Tp[k] = Tc[k]; Tc[k] = Tn[k]; }
            }
            __syncthreads();
            if (s_done) break;
            if (step > 0) {                              // rotate blocks: previous <- current, current <- W
                double2* oldP = P;
                P = C;
                C = Y;
                Y = oldP;
            }
            step += 1;
        }
        // restore the canonical block order for the next candidate (pointers are per-thread copies of the same values)
        P = a.ws + (size_t)blockIdx.x * 3 * n;
        C = P + n;
        Y = C + n;
    }
}

// Where the single-launch path wins (profiles/r02n_time_pairs_small_*.jsonl): the CSR and one CTA's three n x 2 blocks
// must stay cache-resident, and with more candidates than SMs a CTA's latency-bound row loops are no longer hidden
// by other CTAs - there the batched pipeline catches up (n = 13 947, 250 candidates: 3.6 vs 3.4 ms).
inline bool use_pairs_small(const kr_ctx* ctx, const kr_matrix* M, int64_t np) {
    if (getenv("KR_PAIR_SLOTS")) return false;                   // test hook of the batched pipeline
    const int64_t n = M->dev.n;
    if (M->dev.nnz > CSR_L2_RESIDENT_NNZ || n > 20000) return false;
    return np <= ctx->num_sms || n <= 8192;
}

// Same contract as pairs_run (pairs.cuh); one launch, one synchronisation.
inline void pairs_small_run(kr_ctx* ctx, const kr_matrix* M, const int64_t* Ei, const int64_t* Ej, int64_t np, double b_off,
                            double tol, int it, int fun, double* Xm_out, int64_t* iter_out, int* lucky_out) {
    if (np <= 0) return;
    const CsrDev& A = M->dev;
    const int64_t n = A.n;
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(pair_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PS_DYN_SMEM));
    const int ctas = (int)std::min<int64_t>(np, (int64_t)ctx->num_sms);      // 128 registers x 512 threads: one resident CTA per SM
    PairSmallArgs a;
    a.A = A.view();
    a.rows_cta = a.rows_warp = 0;
    for (const RowTile& t : A.tiles_host) {
        if (t.lanes_log2 == 6) a.rows_cta += t.count;
        else if (t.lanes_log2 >= 2) a.rows_warp += t.count;
    }
    std::vector<int> e2((size_t)2 * np);
    for (int64_t q = 0; q < np; ++q) {
        e2[(size_t)q] = (int)(Ei[q] - 1);
        e2[(size_t)(np + q)] = (int)(Ej[q] - 1);
    }
    DevBuf<int> de(ctx, (size_t)2 * np + 1);
    de.upload(e2.data(), (size_t)2 * np);
    KR_CUDA(cudaMemsetAsync(de.p + 2 * np, 0, sizeof(int), ctx->stream));
    DevBuf<double2> ws(ctx, (size_t)ctas * 3 * n);
    DevBuf<double> hbuf(ctx, (size_t)ctas * 3 * it * 4), gs;
    a.gstride = 0;
    a.gscratch = nullptr;
    if (2 * it > PS_SMEM_NN) {
        const int nn = 2 * it;
        a.gstride = (int64_t)2 * nn * (nn | 1) + 2 * nn;
        gs.reset(ctx, (size_t)ctas * a.gstride);
        a.gscratch = gs.p;
    }
    // results packed in one buffer: Xm | iter | lucky
    DevBuf<double> rx(ctx, (size_t)np);
    DevBuf<long long> ri(ctx, (size_t)np);
    DevBuf<int> rl(ctx, (size_t)np);
    a.ei = de.p; a.ej = de.p + np; a.ticket = de.p + 2 * np;
    a.np = (int)np; a.it = it; a.fun = fun; a.tol = tol; a.b_off = b_off;
    a.ws = ws.p; a.hbuf = hbuf.p;
    a.res_Xm = rx.p; a.res_iter = ri.p; a.res_lucky = rl.p;
    KR_LAUNCH(ctx, pair_small_kernel, ctas, PS_THREADS, PS_DYN_SMEM, a);
    std::vector<long long> itv((size_t)np);
    KR_CUDA(cudaMemcpyAsync(Xm_out, rx.p, np * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(itv.data(), ri.p, np * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(lucky_out, rl.p, np * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->counters[3] += np * 8;
    ctx->counters[4] += np * 20;
    for (int64_t q = 0; q < np; ++q) iter_out[q] = itv[(size_t)q];
}

}  // namespace kr
