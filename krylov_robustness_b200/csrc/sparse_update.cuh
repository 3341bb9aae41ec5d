// sparse_update.cuh - tr f(Ã) - tr f(Ã - D) for a sparse symmetric direction D = Δ(X, Ω) (kr_trace_fun_sparse_update):
// the objective of the all-edges callback (config C2) without two large traces that cancel.  With A_t = Ã - (1 - t) D,
//     tr f(Ã) - tr f(A_0) = ∫₀¹ φ'(t) dt,   φ'(t) = tr(f'(A_t) D) = Σ_h c_h X_h f'(A_t)(i_h, j_h)
// (c_h = 2 off the diagonal, 1 on it), and φ is entire in t, so a q-point Gauss-Legendre rule converges fast.  Every
// node is one set of entries f'(A_t)_Ω - the entries the gradient computes, at another t - so all (start node, quadrature
// node) pairs run as the columns of one direction-flavour launch of entries_local_kernel per budget tier.  This file
// holds the host-side rule (nodes, weights, the choice of q) and the fixed-order reduction of the entries.
#pragma once
#include <cmath>
#include "entries_local.cuh"

namespace kr {

constexpr int SU_QCAP = 32;          // largest quadrature order
constexpr int SU_THREADS = 256;
constexpr int SU_BLOCKS = 256;       // partials of the first reduction stage (fixed by the input size only)

// q-point Gauss-Legendre rule on [0, 1]: nodes ascending, weights summing to 1.  Newton's method on P_q from the usual
// cosine guesses, weights 2 / ((1 - x^2) P_q'(x)^2) at the converged root; the rule is symmetric about 1/2.
inline void gauss_legendre01(int q, std::vector<double>& t, std::vector<double>& w) {
    t.assign(q, 0.0);
    w.assign(q, 0.0);
    const double pi = 3.14159265358979323846;
    for (int i = 0; i < (q + 1) / 2; ++i) {
        double x = std::cos(pi * (i + 0.75) / (q + 0.5)), dp = 1.0;
        for (int iter = 0; iter < 100; ++iter) {
            double p0 = 1.0, p1 = x;
            for (int k = 2; k <= q; ++k) {
                const double p2 = ((2 * k - 1) * x * p1 - (k - 1) * p0) / k;
                p0 = p1;
                p1 = p2;
            }
            dp = q * (x * p1 - p0) / (x * x - 1.0);
            const double dx = p1 / dp;
            x -= dx;
            if (std::fabs(dx) <= 1e-16) break;
        }
        double p0 = 1.0, p1 = x;
        for (int k = 2; k <= q; ++k) {
            const double p2 = ((2 * k - 1) * x * p1 - (k - 1) * p0) / k;
            p0 = p1;
            p1 = p2;
        }
        dp = q == 1 ? 1.0 : q * (x * p1 - p0) / (x * x - 1.0);
        const double wi = 1.0 / ((1.0 - x * x) * dp * dp);      // half of the weight on [-1, 1]
        t[q - 1 - i] = 0.5 * (1.0 + x);
        t[i] = 0.5 * (1.0 - x);
        w[q - 1 - i] = wi;
        w[i] = wi;
    }
}

// Smallest q in 1..qcap whose Gauss-Legendre error bound (q!)^4 / ((2q+1) ((2q)!)^3) * max |φ^(2q)| is at most
// tol * sumw, with max |φ^(2q)| <= n ||D||^{2q} e^{ρ}, ρ = ||Ã|| + ||D|| (oracle/sparse_update.py derives the bound);
// qcap when none is.  Evaluated in logarithms.
inline int su_choose_q(int64_t n, double normD, double normA, double tol, double sumw, int qcap) {
    const double target = std::log(tol * sumw);
    for (int q = 1; q < qcap; ++q) {
        const double lb = 4.0 * std::lgamma(q + 1.0) - std::log(2.0 * q + 1.0) - 3.0 * std::lgamma(2.0 * q + 1.0) +
                          std::log((double)n) + 2.0 * q * std::log(normD) + normA + normD;
        if (lb <= target) return q;
    }
    return qcap;
}

// partial[b] = sum over the fixed grid-stride slice of block b of wq[i / k] * (cx[i % k] * E[i]),  i < q * k
__global__ void __launch_bounds__(SU_THREADS)
su_partial_kernel(const double* __restrict__ E, const double* __restrict__ cx, const double* __restrict__ wq, int64_t k,
                  int64_t total, double* __restrict__ partial) {
    __shared__ double red[64];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * SU_THREADS + threadIdx.x; i < total; i += (int64_t)gridDim.x * SU_THREADS)
        s += wq[i / k] * (cx[i % k] * E[i]);
    s = block_sum<SU_THREADS>(s, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(SU_THREADS)
su_final_kernel(const double* __restrict__ partial, int nb, double* __restrict__ out) {
    __shared__ double red[64];
    double s = 0.0;
    for (int i = threadIdx.x; i < nb; i += SU_THREADS) s += partial[i];
    s = block_sum<SU_THREADS>(s, red);
    if (threadIdx.x == 0) *out = s;
}

// E[idx[m]] = v[m]: entries of the columns that went through the dense batch
__global__ void su_scatter_kernel(double* __restrict__ E, const int64_t* __restrict__ idx, const double* __restrict__ v,
                                  int64_t m) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) E[idx[i]] = v[i];
}

// Σ_i wq[i / k] cx[i % k] E[i] over q * k device entries: two stages in a fixed order, no atomics (bit-identical run to run)
inline double su_reduce(kr_ctx* ctx, const double* E, const std::vector<double>& cx, const std::vector<double>& wq) {
    const int64_t k = (int64_t)cx.size(), total = k * (int64_t)wq.size();
    DevBuf<double> dcx(ctx, cx.size()), dwq(ctx, wq.size()), part(ctx, SU_BLOCKS + 1);
    dcx.upload(cx.data(), cx.size());
    dwq.upload(wq.data(), wq.size());
    const int nb = (int)std::max<int64_t>(1, std::min<int64_t>(SU_BLOCKS, ceil_div(total, SU_THREADS)));
    KR_LAUNCH(ctx, su_partial_kernel, nb, SU_THREADS, 0, E, dcx.p, dwq.p, k, total, part.p);
    KR_LAUNCH(ctx, su_final_kernel, 1, SU_THREADS, 0, part.p, nb, part.p + SU_BLOCKS);
    double r = 0.0;
    KR_CUDA(cudaMemcpyAsync(&r, part.p + SU_BLOCKS, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->counters[4] += (int64_t)sizeof(double);
    return r;
}

}  // namespace kr
