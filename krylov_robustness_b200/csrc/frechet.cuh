// frechet.cuh - Hessian callbacks of the weighted experiments (SURVEY.md section 8, row f3):
// functions/multiple_frechet_eval.m + functions/hessianfcn_exp.m / hessianfcn_fun.m.
//
// For every pair (i, j) in omega the reference builds K(A, e_i) and K(A', e_j) with bs = 1 Arnoldi and
// takes the (1,2) block of f([G, C; 0, H']) with C = (V'e_i)(W'e_j)' = +-e1 e1'
// (multiple_frechet_eval.m:150-159).  Here the two families of spaces are two ArnoldiBatch objects (one
// wide SpMM per family per step) and the block-triangular function is evaluated per pair by one CTA in
// shared memory through the Daleckii-Krein formula: with G = P diag(lambda) P', H = Q diag(mu) Q'
// (both symmetric up to rounding on this path; symmetrised as in entries.cuh),
//     X = P [ f[lambda_a, mu_b] * P(1,a) Q(1,b) ]_{ab} Q'
// where f[.,.] is the first divided difference, written in the cancellation-free product form
// exp[l,m] = e^{(l+m)/2} sinh(d)/d, sinh[l,m] = cosh((l+m)/2) sinh(d)/d, cosh[l,m] = sinh((l+m)/2) sinh(d)/d,
// d = (l-m)/2.  The lag-3 stopping rule uses ||X_j - pad(X_{j-3})||_2 (:172) = sqrt(lambda_max(D'D)).
#pragma once
#include "entries.cuh"

namespace kr {

constexpr int FRECHET_CAP = 64;     // largest projected size handled in shared memory (5 matrices)

__device__ __forceinline__ double divided_difference(int fun, double l, double m) {
    const double mean = 0.5 * (l + m), d = 0.5 * (l - m);
    const double shc = d == 0.0 ? 1.0 : sinh(d) / d;
    const double w = fun == KR_FUN_EXP ? exp(mean) : fun == KR_FUN_SINH ? cosh(mean) : sinh(mean);
    return w * shc;
}

// One CTA per pair.  HcI/HcJ: Hessenberg columns of the row / column families (entries.cuh layout);
// sa[p], sb[p]: space (column) of pair p in each family.  hist[pair][4][CAP*CAP]; xfin[pair][CAP*CAP].
__global__ void __launch_bounds__(JAC_THREADS)
frechet_step_kernel(const double* __restrict__ HcI, const double* __restrict__ HcJ, int it1, int jj, int fun, double tol,
                    const int* __restrict__ sa, const int* __restrict__ sb, double* __restrict__ hist,
                    double* __restrict__ xfin, int* __restrict__ nfin, int* __restrict__ conv, int* __restrict__ nactive) {
    extern __shared__ double dyn[];
    __shared__ JacobiShared sh;
    __shared__ double lam[FRECHET_CAP], mu[FRECHET_CAP];
    const int p = blockIdx.x;
    if (conv[p]) return;
    const int lda = jj | 1;
    double* G = dyn;
    double* P = G + jj * lda;
    double* H = P + jj * lda;
    double* Q = H + jj * lda;
    double* T = Q + jj * lda;
    const double* HI = HcI + (int64_t)sa[p] * it1 * (it1 + 1);
    const double* HJ = HcJ + (int64_t)sb[p] * it1 * (it1 + 1);
    for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
        const int r = e % jj, c = e / jj;
        const double g1 = r <= c + 1 ? HI[(int64_t)c * (it1 + 1) + r] : 0.0;
        const double g2 = c <= r + 1 ? HI[(int64_t)r * (it1 + 1) + c] : 0.0;
        const double h1 = r <= c + 1 ? HJ[(int64_t)c * (it1 + 1) + r] : 0.0;
        const double h2 = c <= r + 1 ? HJ[(int64_t)r * (it1 + 1) + c] : 0.0;
        G[r + c * lda] = 0.5 * (g1 + g2);
        H[r + c * lda] = 0.5 * (h1 + h2);
        P[r + c * lda] = r == c ? 1.0 : 0.0;
        Q[r + c * lda] = r == c ? 1.0 : 0.0;
    }
    __syncthreads();
    block_jacobi(G, jj, lda, P, lda, &sh);
    block_jacobi(H, jj, lda, Q, lda, &sh);
    for (int i = threadIdx.x; i < jj; i += JAC_THREADS) {
        lam[i] = G[i + i * lda];
        mu[i] = H[i + i * lda];
    }
    __syncthreads();
    // T = [f[lam_a, mu_b] P(0,a) Q(0,b)]
    for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
        const int a = e % jj, b = e / jj;
        T[a + b * lda] = divided_difference(fun, lam[a], mu[b]) * P[0 + a * lda] * Q[0 + b * lda];
    }
    __syncthreads();
    // G <- P * T
    for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
        const int r = e % jj, c = e / jj;
        double s = 0.0;
        for (int k = 0; k < jj; ++k) s += P[r + k * lda] * T[k + c * lda];
        G[r + c * lda] = s;
    }
    __syncthreads();
    // H <- X = G * Q'
    for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
        const int r = e % jj, c = e / jj;
        double s = 0.0;
        for (int k = 0; k < jj; ++k) s += G[r + k * lda] * Q[c + k * lda];
        H[r + c * lda] = s;
    }
    __syncthreads();
    double* hp = hist + (int64_t)p * 4 * FRECHET_CAP * FRECHET_CAP;
    double err = 0.0;
    if (jj > 3) {
        const double* old = hp + (int64_t)((jj - 3) & 3) * FRECHET_CAP * FRECHET_CAP;   // (jj-3) x (jj-3), ld jj-3
        const int on = jj - 3;
        for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
            const int r = e % jj, c = e / jj;
            T[r + c * lda] = H[r + c * lda] - ((r < on && c < on) ? old[r + c * on] : 0.0);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {       // G <- T' T
            const int r = e % jj, c = e / jj;
            double s = 0.0;
            for (int k = 0; k < jj; ++k) s += T[k + r * lda] * T[k + c * lda];
            G[r + c * lda] = s;
        }
        __syncthreads();
        block_jacobi(G, jj, lda, nullptr, 0, &sh);
        double m = 0.0;
        for (int i = threadIdx.x; i < jj; i += JAC_THREADS) m = fmax(m, G[i + i * lda]);
        for (int off = 16; off; off >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, off));
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh.red[threadIdx.x >> 5] = m;
        __syncthreads();
        for (int w = 0; w < JAC_THREADS / 32; ++w) m = fmax(m, sh.red[w]);
        err = sqrt(fmax(m, 0.0));
    }
    double* cur = hp + (int64_t)(jj & 3) * FRECHET_CAP * FRECHET_CAP;
    double* fin = xfin + (int64_t)p * FRECHET_CAP * FRECHET_CAP;
    for (int e = threadIdx.x; e < jj * jj; e += JAC_THREADS) {
        const int r = e % jj, c = e / jj;
        const double v = H[r + c * lda];
        cur[r + c * jj] = v;
        fin[r + c * jj] = v;
    }
    if (threadIdx.x == 0) {
        nfin[p] = jj;
        if (jj > 3 && !(err > tol)) {
            conv[p] = 1;
            atomicSub(nactive, 1);
        }
    }
}

// Hes(j, l) = -2 * U_{a_j}(O(l,1), 1:sz) * X_j * V_{b_j}(O(l,2), 1:sz)'  for l >= j, mirrored
// (hessianfcn_exp.m:9-15).  One CTA per j, one thread per l.
__global__ void hessian_assemble_kernel(const double* const* __restrict__ VI, const double* const* __restrict__ VJ,
                                        int64_t n, const int64_t* __restrict__ omega, int m, const int* __restrict__ sa,
                                        const int* __restrict__ sb, const double* __restrict__ xfin,
                                        const int* __restrict__ nfin, double* __restrict__ Hes) {
    const int j = blockIdx.x;
    const int sz = nfin[j];
    const double* X = xfin + (int64_t)j * FRECHET_CAP * FRECHET_CAP;      // sz x sz, ld sz
    const int ca = sa[j], cb = sb[j];
    for (int l = j + threadIdx.x; l < m; l += blockDim.x) {
        const int64_t offa = (int64_t)(ca / PW) * n * PW + (omega[l] - 1) * PW + (ca % PW);
        const int64_t offb = (int64_t)(cb / PW) * n * PW + (omega[m + l] - 1) * PW + (cb % PW);
        double u[FRECHET_CAP];
        for (int r = 0; r < sz; ++r) u[r] = VI[r][offa];
        double acc = 0.0;
        for (int c = 0; c < sz; ++c) {
            double t = 0.0;
            for (int r = 0; r < sz; ++r) t += u[r] * X[r + c * sz];
            acc += t * VJ[c][offb];
        }
        Hes[j + (int64_t)l * m] = -2.0 * acc;
        Hes[l + (int64_t)j * m] = -2.0 * acc;
    }
}

// The stepping of multiple_frechet_eval (:86-195) for the pairs omega (m x 2 col-major, 1-based, checked by the caller):
// two ArnoldiBatch families (one space per distinct first / second index) advanced together until every pair met the
// lag-3 rule or it steps were taken.  xfin[p] (nfin[p] x nfin[p], ld nfin[p]) is X of pair p at its stop step.
struct FrechetPairs {
    std::vector<int64_t> rowsI, rowsJ;
    std::vector<int> sa, sb;
    std::unique_ptr<ArnoldiBatch> BI, BJ;
    DevBuf<int> dsa, dsb, istate;               // istate: nfin[m], conv[m], nactive
    DevBuf<double> hist, xfin;
    int64_t iter = 0;
    const int* nfin() const { return istate.p; }
};

inline void frechet_pairs_run(kr_ctx* ctx, const kr_matrix* M, int64_t m, const int64_t* omega, int fun, double tol,
                              int it, FrechetPairs& F) {
    const int it1 = it + 1;
    F.sa.resize(m);
    F.sb.resize(m);
    std::map<int64_t, int> pi, pj;
    for (int64_t p = 0; p < m; ++p) {
        const int64_t i = omega[p], j = omega[m + p];
        auto fi = pi.find(i);
        if (fi == pi.end()) { pi[i] = (int)F.rowsI.size(); F.sa[p] = (int)F.rowsI.size(); F.rowsI.push_back(i); } else F.sa[p] = fi->second;
        auto fj = pj.find(j);
        if (fj == pj.end()) { pj[j] = (int)F.rowsJ.size(); F.sb[p] = (int)F.rowsJ.size(); F.rowsJ.push_back(j); } else F.sb[p] = fj->second;
    }
    F.BI.reset(new ArnoldiBatch(ctx, M->dev, F.rowsI, it));
    F.BJ.reset(new ArnoldiBatch(ctx, M->T(), F.rowsJ, it));
    F.dsa.reset(ctx, m);
    F.dsb.reset(ctx, m);
    F.istate.reset(ctx, (size_t)2 * m + 1);
    F.dsa.upload(F.sa.data(), m);
    F.dsb.upload(F.sb.data(), m);
    F.hist.reset(ctx, (size_t)m * 4 * FRECHET_CAP * FRECHET_CAP);
    F.xfin.reset(ctx, (size_t)m * FRECHET_CAP * FRECHET_CAP);
    F.hist.zero(); F.xfin.zero(); F.istate.zero();
    int* nfin = F.istate.p;
    int* conv = F.istate.p + m;
    int* nactive = F.istate.p + 2 * m;
    int nact = (int)m;
    KR_CUDA(cudaMemcpyAsync(nactive, &nact, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    static bool attr_set[64] = {};              // per device: the attribute lives in the device's primary context
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(frechet_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JAC_SMEM_LIMIT));
    int j = 0;
    for (j = 0; j < it; ++j) {
        F.BI->step(j);
        F.BJ->step(j);
        const int jj = j + 1;
        const size_t smem = (size_t)(5 * jj * (jj | 1)) * sizeof(double);
        KR_LAUNCH(ctx, frechet_step_kernel, (int)m, JAC_THREADS, smem, F.BI->Hc.p, F.BJ->Hc.p, it1, jj, fun, tol, F.dsa.p,
                  F.dsb.p, F.hist.p, F.xfin.p, nfin, conv, nactive);
        KR_CUDA(cudaMemcpyAsync(&nact, nactive, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        if (nact <= 0) { ++j; break; }
    }
    F.iter = std::min(j, it);
}

struct HessianResult { std::vector<double> Hes; int64_t iter = 0; };

// omega: m x 2 column-major on the host (1-based)
inline HessianResult frechet_hessian_run(kr_ctx* ctx, const kr_matrix* M, int64_t m, const int64_t* omega, int fun,
                                         double tol, int it) {
    const int64_t n = M->dev.n;
    it = std::min(it, FRECHET_CAP);
    for (int64_t q = 0; q < 2 * m; ++q)
        if (omega[q] < 1 || omega[q] > n) fail(KR_ERR_ARG, "Omega index out of range");
    FrechetPairs F;
    frechet_pairs_run(ctx, M, m, omega, fun, tol, it, F);
    DevBuf<int64_t> dom(ctx, 2 * m);
    dom.upload(omega, 2 * m);
    HessianResult out;
    out.iter = F.iter;
    DevBuf<const double*> pI = F.BI->block_pointers(), pJ = F.BJ->block_pointers();
    DevBuf<double> dH(ctx, (size_t)m * m);
    dH.zero();
    KR_LAUNCH(ctx, hessian_assemble_kernel, (int)m, 64, 0, pI.p, pJ.p, n, dom.p, (int)m, F.dsa.p, F.dsb.p, F.xfin.p,
              F.nfin(), dH.p);
    out.Hes = dH.to_host();
    return out;
}

// ----------------------------------------------------------------------------- Hessian times vectors
// W(h, r) = -2 <X_h, U_h' S_r V_h>_F = -2 sum_e S_r(a_e, b_e) U_h(a_e, :) X_h V_h(b_e, :)'  over the entries e of S
// (entry list sorted by (a, b), sval[e * p + r]).  One CTA per pair; the entries go in blocks of HESSP_THREADS: thread t
// forms g_e for entry e0 + t, then thread t sums column r = r0 + t over the block in entry order.  Every sum has a
// fixed order: results are bit-identical run to run.
constexpr int HESSP_THREADS = 128;
__global__ void __launch_bounds__(HESSP_THREADS)
hessp_contract_kernel(const double* const* __restrict__ VI, const double* const* __restrict__ VJ, int64_t n,
                      const int* __restrict__ sa, const int* __restrict__ sb, const double* __restrict__ xfin,
                      const int* __restrict__ nfin, const int64_t* __restrict__ ea, const int64_t* __restrict__ eb,
                      const double* __restrict__ sval, int64_t nnzS, int p, double* __restrict__ W, int64_t ldw) {
    __shared__ double X[FRECHET_CAP * FRECHET_CAP];
    __shared__ double g[HESSP_THREADS];
    const int h = blockIdx.x, tid = threadIdx.x;
    const int sz = nfin[h];
    for (int e = tid; e < sz * sz; e += HESSP_THREADS) X[e] = xfin[(int64_t)h * FRECHET_CAP * FRECHET_CAP + e];
    const int ca = sa[h], cb = sb[h];
    const int64_t ca0 = (int64_t)(ca / PW) * n * PW + (ca % PW), cb0 = (int64_t)(cb / PW) * n * PW + (cb % PW);
    for (int r0 = 0; r0 < p; r0 += HESSP_THREADS) {
        double acc = 0.0;
        for (int64_t e0 = 0; e0 < nnzS; e0 += HESSP_THREADS) {
            __syncthreads();
            const int64_t e = e0 + tid;
            if (e < nnzS) {
                const int64_t offa = ca0 + ea[e] * PW, offb = cb0 + eb[e] * PW;
                double u[FRECHET_CAP];
                bool any = false;
                for (int k = 0; k < sz; ++k) { u[k] = VI[k][offa]; any |= u[k] != 0.0; }
                double s = 0.0;
                if (any)
                    for (int c = 0; c < sz; ++c) {
                        const double v = VJ[c][offb];
                        if (v == 0.0) continue;
                        double t = 0.0;
                        for (int k = 0; k < sz; ++k) t += u[k] * X[k + c * sz];
                        s += t * v;
                    }
                g[tid] = s;
            }
            __syncthreads();
            const int r = r0 + tid;
            if (r < p) {
                const int64_t ne = nnzS - e0 < HESSP_THREADS ? nnzS - e0 : HESSP_THREADS;
                for (int q = 0; q < ne; ++q) acc += g[q] * sval[(e0 + q) * p + r];
            }
        }
        if (r0 + tid < p) W[h + (int64_t)(r0 + tid) * ldw] = -2.0 * acc;
    }
}

// Bytes a chunk of the dense path holds, approximately: both families' bases (n x (it + 2) per space, worst case one space
// per pair and family) and the 4 + 1 lag-3 / final X matrices of every pair.  ArnoldiBatch's Hessenberg columns, its
// partial-sum buffers and the padding of a panel to PW columns come on top (a few percent at n = 10^5).
constexpr size_t HESSP_DENSE_BUDGET = (size_t)16 << 30;

// The pairs sel of omega (m x 2, 1-based, checked) through the dense families, in chunks that fit HESSP_DENSE_BUDGET;
// row h of W (m x p, ld ldw, host) gets -2 <X_h, U_h' S V_h>.  S: entries (ea, eb) (0-based, sorted) with values
// sval[e * p + r].  Returns the largest stop step of any pair.
inline int64_t hessp_dense_run(kr_ctx* ctx, const kr_matrix* M, int64_t m, const int64_t* omega,
                               const std::vector<int64_t>& sel, int fun, double tol, int it,
                               const std::vector<int64_t>& ea, const std::vector<int64_t>& eb,
                               const std::vector<double>& sval, int p, double* W, int64_t ldw) {
    const int64_t n = M->dev.n, nnzS = (int64_t)ea.size();
    it = std::min(it, FRECHET_CAP);
    const size_t per_pair = (size_t)2 * (size_t)n * (it + 2) * sizeof(double) +
                            (size_t)5 * FRECHET_CAP * FRECHET_CAP * sizeof(double);
    const int64_t chunk = std::max<int64_t>(1, (int64_t)(HESSP_DENSE_BUDGET / per_pair));
    DevBuf<int64_t> dea(ctx, nnzS), deb(ctx, nnzS);
    DevBuf<double> dsv(ctx, sval.size());
    dea.upload(ea.data(), nnzS);
    deb.upload(eb.data(), nnzS);
    dsv.upload(sval.data(), sval.size());
    int64_t iter = 0;
    for (int64_t c0 = 0; c0 < (int64_t)sel.size(); c0 += chunk) {
        const int64_t mc = std::min<int64_t>(chunk, (int64_t)sel.size() - c0);
        std::vector<int64_t> om(2 * mc);
        for (int64_t q = 0; q < mc; ++q) {
            om[q] = omega[sel[c0 + q]];
            om[mc + q] = omega[m + sel[c0 + q]];
        }
        FrechetPairs F;
        frechet_pairs_run(ctx, M, mc, om.data(), fun, tol, it, F);
        iter = std::max(iter, F.iter);
        DevBuf<const double*> pI = F.BI->block_pointers(), pJ = F.BJ->block_pointers();
        DevBuf<double> dW(ctx, (size_t)mc * p);
        KR_LAUNCH(ctx, hessp_contract_kernel, (int)mc, HESSP_THREADS, 0, pI.p, pJ.p, n, F.dsa.p, F.dsb.p, F.xfin.p,
                  F.nfin(), dea.p, deb.p, dsv.p, nnzS, p, dW.p, mc);
        std::vector<double> Wc = dW.to_host();
        for (int r = 0; r < p; ++r)
            for (int64_t q = 0; q < mc; ++q) W[sel[c0 + q] + (int64_t)r * ldw] = Wc[q + (int64_t)r * mc];
    }
    return iter;
}

}  // namespace kr
