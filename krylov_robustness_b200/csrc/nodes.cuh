// nodes.cuh - node-removal scores: for every candidate node v, tr f(Ã) - tr f(A) where Ã is A with the off-diagonal
// entries of row and column v set to zero (a_vv kept, n unchanged).
//
// The reference scores such a rank-two edit with trace_fun_update(A, U, B) and U = [e_v, a'], a' = the off-diagonal
// part of row v (functions/trace_fun_update.m:72-124).  range(U) lies in K_2(A, e_v), so K_j(A, U) = K_{j+1}(A, e_v):
// the projected update is a single-vector Lanczos run from e_v (functions/lanczos_krylov.m:73-101 with bs = 1), and at
// step j
//     Gm  = T_{j+1}                        (symmetric tridiagonal of the first j+1 Lanczos vectors)
//     tGm = alpha_1 (+) T_{j+1}(2:, 2:)    (Gm with its (1,2) and (2,1) entries set to zero: Ã projected)
//     Xm  = trace formula (trace_fun_update.m:83-89) on d1 = sort(eig(tGm)), d2 = sort(eig(Gm))
// with the lag-2 stopping rule (:104-118) and the lucky-breakdown exit (:119-124, beta_{j+1} < 1e-8).  A node whose
// row has no off-diagonal entry (beta_1 < 1e-8) scores 0 with iter = 1, lucky.
//
// One probe column per candidate, panel-major, advanced by the SLQ step kernels (dense.cuh: spmm_kernel<EpiDot> for
// alpha, combine3_norm_kernel + slq_beta_kernel for beta; pending kr_matrix_set_edges entries, those of v's own row
// included, enter through the DELTA flavour of the SpMM).  The Lanczos coefficients of a column do not depend on when
// it stops, so the steps run in batches of NODE_BATCH and the host reads one active count per batch.
// node_step_kernel takes, per candidate and per step of the batch, every eigenvalue of both tridiagonals by Sturm
// bisection (one thread per eigenvalue), evaluates the formula in a fixed order and applies the stopping rules.
// Every reduction has a fixed order: scores, iteration counts and flags are bit-reproducible run to run.
#pragma once
#include "dense.cuh"
#include "smalldense.cuh"

namespace kr {

constexpr int NODE_THREADS = 128;
constexpr int NODE_BATCH = 8;                      // Lanczos steps between two host reads of the active count
constexpr int NODE_MAX_N = SLQ_MAX_M + 1;          // step j = it <= SLQ_MAX_M needs T_{it+1}

struct NodeState {
    double* Xstop;     // [2][tc] lag-2 history
    double* Xm;        // [tc]
    int* iter;         // [tc]
    int* lucky;        // [tc]
    int* active;       // [tc]
};

// e_v into column c of the zeroed panel-major block U1, unit scale; padding columns stay zero with scale 0
__global__ void node_seed_kernel(double* __restrict__ U1, int64_t n, const int64_t* __restrict__ V, int cols, int tc,
                                 SlqState st, NodeState ns) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= tc) return;
    const bool real = c < cols;
    if (real) U1[(int64_t)(c / PW) * n * PW + V[c] * PW + (c % PW)] = 1.0;
    st.s1[c] = real ? 1.0 : 0.0;
    st.s0[c] = 0.0;
    st.beta_prev[c] = 0.0;
    ns.Xstop[c] = 0.0;
    ns.Xstop[tc + c] = 0.0;
    ns.Xm[c] = 0.0;
    ns.iter[c] = 0;
    ns.lucky[c] = 0;
    ns.active[c] = real;
}

// k-th smallest (0-based) eigenvalue of the tridiagonal (d, e2 = squared off-diagonals) of order n inside [lo, hi],
// bisected down to an absolute width of eps/4 * tn (tn >= ||T||, LAPACK dstebz's accuracy class)
__device__ double node_bisect(const double* d, const double* e2, int n, int k, double lo, double hi, double tn) {
    const double goal = 0.25 * 2.220446049250313e-16 * tn;
    for (int r = 0; r < 96 && hi - lo > goal; ++r) {
        const double mid = 0.5 * (lo + hi);
        if (mid <= lo || mid >= hi) break;
        if (sturm_count(d, e2, n, mid) > k) hi = mid;
        else lo = mid;
    }
    return 0.5 * (lo + hi);
}

// One CTA per candidate column: node steps j0..j1 (1-based) of every still-active column.  alpha / beta: [step][tc] as
// written by slq_alpha_kernel / slq_beta_kernel (index i holds alpha_{i+1}, beta_{i+1}); steps 0..j1 must be done.
__global__ void __launch_bounds__(NODE_THREADS)
node_step_kernel(const double* __restrict__ alpha, const double* __restrict__ beta, int tc, int j0, int j1, int it,
                 double tol, int fun, NodeState ns) {
    __shared__ double d[NODE_MAX_N], e2[NODE_MAX_N], e2t[NODE_MAX_N], ev1[NODE_MAX_N], ev2[NODE_MAX_N];
    __shared__ double gb[3];
    __shared__ int s_done;
    const int c = blockIdx.x;
    if (!ns.active[c]) return;
    const int tid = threadIdx.x;
    for (int i = tid; i <= j1; i += NODE_THREADS) {
        d[i] = alpha[(int64_t)i * tc + c];
        const double b = beta[(int64_t)i * tc + c];
        e2[i] = b * b;
        e2t[i] = i == 0 ? 0.0 : b * b;
    }
    __syncthreads();
    for (int j = j0; j <= j1; ++j) {
        const int N = j + 1;
        if (j == 1 && !(beta[c] >= 1e-8)) {                // no off-diagonal entry in row v: A e_v = a_vv e_v
            if (tid == 0) {
                ns.Xm[c] = 0.0;
                ns.iter[c] = 1;
                ns.lucky[c] = 1;
                ns.active[c] = 0;
            }
            return;
        }
        if (tid == 0) {                                    // Gershgorin bounds of T_N (they also enclose tGm)
            double mn = 1e300, mx = -1e300;
            for (int i = 0; i < N; ++i) {
                const double r = (i > 0 ? sqrt(e2[i - 1]) : 0.0) + (i + 1 < N ? sqrt(e2[i]) : 0.0);
                mn = fmin(mn, d[i] - r);
                mx = fmax(mx, d[i] + r);
            }
            const double tn = fmax(fmax(fabs(mn), fabs(mx)), 1e-300);
            const double pad = 4.0 * tn * 2.220446049250313e-16 * N + 1e-290;
            gb[0] = mn - pad;
            gb[1] = mx + pad;
            gb[2] = tn;
        }
        __syncthreads();
        for (int t = tid; t < 2 * N; t += NODE_THREADS) {
            const int m = t / N, k = t - m * N;
            const double x = node_bisect(d, m ? e2 : e2t, N, k, gb[0], gb[1], gb[2]);
            (m ? ev2 : ev1)[k] = x;
        }
        __syncthreads();
        if (tid == 0) {
            double Xm = 0.0;                               // fixed summation order
            for (int i = 0; i < N; ++i) {
                if (fun == KR_FUN_EXP) Xm += exp(ev1[i]) * (1.0 - exp(ev2[i] - ev1[i]));
                else Xm += fun_eval(fun, ev1[i]) - fun_eval(fun, ev2[i]);
            }
            const int lk = !(beta[(int64_t)j * tc + c] >= 1e-8);
            bool done = false;
            double* Xs = ns.Xstop;
            if (j <= 2) {
                Xs[(j - 1) * tc + c] = Xm;
            } else if (fabs(Xm - Xs[c]) < tol) {
                done = true;
            } else {
                Xs[c] = Xs[tc + c];
                Xs[tc + c] = Xm;
            }
            done = done || lk || j == it;
            ns.Xm[c] = Xm;
            ns.iter[c] = j;
            ns.lucky[c] = lk;
            if (done) ns.active[c] = 0;
            s_done = done;
        }
        __syncthreads();
        if (s_done) return;
    }
}

// count[0] = active columns; panel_active[q] = any active column in panel q (the SpMM skips the others)
__global__ void __launch_bounds__(256)
node_active_kernel(const int* __restrict__ active, int panels, int* __restrict__ panel_active, int* __restrict__ count) {
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int cnt = 0;
    for (int q = threadIdx.x; q < panels; q += blockDim.x) {
        int any = 0;
        for (int i = 0; i < PW; ++i) any += active[q * PW + i];
        panel_active[q] = any > 0;
        cnt += any;
    }
    atomicAdd(&s_cnt, cnt);                                // integer: the total does not depend on the order
    __syncthreads();
    if (threadIdx.x == 0) count[0] = s_cnt;
}

// Scores the candidates V[0..cols) (0-based node numbers) with the three n x cols work blocks of one chunk.
inline void nodes_chunk(kr_ctx* ctx, const kr_matrix* M, const int64_t* V, int cols, double tol, int it, int fun,
                        double* Xm_out, int64_t* iter_out, int* lucky_out) {
    const CsrDev& A = M->dev;
    const int64_t n = A.n;
    PanelBuf U1b(ctx, n, cols), U0b(ctx, n, cols), Y(ctx, n, cols);
    const int panels = U1b.panels, tc = panels * PW;
    U1b.buf.zero();
    U0b.buf.zero();
    const int rb = col_row_blocks(n);
    DevBuf<double> partial(ctx, (size_t)std::max(rb, A.ntiles) * tc), sums(ctx, tc), scal(ctx, (size_t)tc * 6);
    DevBuf<double> ab(ctx, (size_t)2 * (it + 1) * tc), nsd(ctx, (size_t)3 * tc);
    DevBuf<int> nsi(ctx, (size_t)3 * tc + panels + 1);
    DevBuf<int64_t> vdev(ctx, (size_t)cols);
    vdev.upload(V, (size_t)cols);
    SlqState st;
    st.s1 = scal.p;
    st.s0 = scal.p + tc;
    st.beta_prev = scal.p + 2 * tc;
    st.coef = scal.p + 3 * tc;
    st.alpha = ab.p;
    st.beta = ab.p + (size_t)(it + 1) * tc;
    NodeState ns;
    ns.Xstop = nsd.p;
    ns.Xm = nsd.p + 2 * tc;
    ns.iter = nsi.p;
    ns.lucky = nsi.p + tc;
    ns.active = nsi.p + 2 * tc;
    int* pact = nsi.p + 3 * tc;
    int* count = pact + panels;
    const int sb = (int)ceil_div(tc, 128);
    const dim3 cgrid((unsigned)rb, (unsigned)panels);
    KR_LAUNCH(ctx, node_seed_kernel, sb, 128, 0, U1b.p(), n, vdev.p, cols, tc, st, ns);
    double* U1 = U1b.p();
    double* U0 = U0b.p();
    int steps = 0, jdone = 0, live = cols;
    while (jdone < it && live > 0) {
        const int j1 = std::min(it, jdone + NODE_BATCH);
        for (; steps <= j1; ++steps) {                     // Lanczos step index `steps` -> alpha_{steps+1}, beta_{steps+1}
            EpiDot epi;
            epi.Y = Y.p();
            epi.X = U1;
            epi.partial = partial.p;
            epi.total_cols = tc;
            launch_spmm(ctx, A, U1, panels, epi, nullptr, live, jdone > 0 ? pact : nullptr);
            sum_partials(ctx, partial.p, A.ntiles, tc, sums.p);
            KR_LAUNCH(ctx, slq_alpha_kernel, sb, 128, 0, sums.p, tc, st, steps);
            KR_LAUNCH(ctx, combine3_norm_kernel, cgrid, COL_THREADS, 0, Y.p(), U1, U0, U0, n, st.coef, tc, partial.p);
            sum_partials(ctx, partial.p, rb, tc, sums.p);
            KR_LAUNCH(ctx, slq_beta_kernel, sb, 128, 0, sums.p, tc, st, steps);
            std::swap(U0, U1);
        }
        KR_LAUNCH(ctx, node_step_kernel, cols, NODE_THREADS, 0, st.alpha, st.beta, tc, jdone + 1, j1, it, tol, fun, ns);
        jdone = j1;
        KR_LAUNCH(ctx, node_active_kernel, 1, 256, 0, ns.active, panels, pact, count);
        KR_CUDA(cudaMemcpyAsync(&live, count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->counters[4] += (int64_t)sizeof(int);
    }
    std::vector<double> x(cols);
    std::vector<int> iv((size_t)2 * tc);
    KR_CUDA(cudaMemcpyAsync(x.data(), ns.Xm, cols * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(iv.data(), ns.iter, (size_t)2 * tc * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->counters[4] += (int64_t)(cols * sizeof(double) + 2 * tc * sizeof(int));
    for (int c = 0; c < cols; ++c) {
        Xm_out[c] = x[(size_t)c];
        iter_out[c] = iv[(size_t)c];
        lucky_out[c] = iv[(size_t)(tc + c)];
    }
}

// All candidates, in column chunks that keep the three n x cols work blocks within ~48 GB (whole panels).
inline void nodes_run(kr_ctx* ctx, const kr_matrix* M, const int64_t* V, int64_t nV, double tol, int it, int fun,
                      double* Xm, int64_t* iter, int* lucky) {
    const int64_t n = M->dev.n;
    const int64_t budget = (int64_t)48 << 30;
    const int64_t chunk = std::min<int64_t>(std::max<int64_t>(PW, budget / (3 * std::max<int64_t>(n, 1) * 8) / PW * PW), 1 << 20);
    for (int64_t c0 = 0; c0 < nV; c0 += chunk) {
        const int cols = (int)std::min<int64_t>(chunk, nV - c0);
        nodes_chunk(ctx, M, V + c0, cols, tol, it, fun, Xm + c0, iter + c0, lucky + c0);
    }
}

}  // namespace kr
