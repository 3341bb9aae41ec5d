// hessp_local.cuh - kr_frechet_hessian_multiply on graphs whose Krylov vectors stay LOCAL (road networks): ONE CTA runs
// one Frechet pair h = (i, j) of multiple_frechet_eval (functions/multiple_frechet_eval.m:86-195) whole, in shared memory,
// on the ball around {i, j}:
//   * the ball grows one BFS level per step with the hash table and the deterministic level sort of entries_local.cuh;
//     basis vector l of either space lives on the nodes within l hops, so it is stored with len[l] entries (BFS order);
//   * the spaces K(A, e_i) (U) and K(A, e_j) (V) advance in lockstep, each by w = A v_l and CGS2 + the third pass of
//     arnoldi_krylov.m:104-106;
//   * X_h = P [f[lam_a, mu_b] P(0,a) Q(0,b)] Q' (Daleckii-Krein, frechet.cuh) from the eigen-decompositions of the two
//     symmetrised tridiagonals by one warp each (EISPACK tql2, as warp_tridiag_fx), the lag-3 rule on the spectral norm
//     ||X_j - pad(X_{j-3})||_2 (:172) by the block Jacobi solve of the dense path;
//   * at the stop, W(h, r) = -2 sum_{a in ball} sum_{b in S row a, b in ball} S_r(a, b) U(a,:) X_h V(b,:)': the entries of S
//     outside the ball meet a zero row of U or V, so this is exact, not a truncation.  S is a CSR by global row.
// Pairs are handed out by a ticket counter.  A pair whose ball outgrows the budget is flagged (1) and run again with the
// next tier; one that outgrows the last tier, or that has not stopped after EL_IT steps while the caller allows more (2),
// takes the dense families of frechet.cuh.  Every sum has a fixed order and there are no floating-point atomics.
#pragma once
#include "entries_local.cuh"
#include "frechet.cuh"

namespace kr {

struct HesspLocalBudget { int maxn, hcap, arena; };     // arena: doubles per space
constexpr int HL_NTIERS = 3;
constexpr HesspLocalBudget HL_TIERS[HL_NTIERS] = {{384, 1024, 2048}, {768, 2048, 4096}, {1536, 4096, 6144}};
constexpr int HL_X = EL_IT * EL_IT;                     // one X_h (jj x jj, ld jj)
constexpr int HL_LDG = EL_IT | 1;

struct HesspLocalArgs {
    const int64_t* omega;            // [2m] 1-based, col-major
    const int* sel;                  // pairs to run (null: all of 0..m-1)
    int nsel, m;
    const int* srow;                 // [n + 1] S by global row
    const int* scol;                 // [nnzS]
    const double* sval;              // [nnzS * p]
    int p;
    double* W;                       // [m x p], ld m
    int* steps;                      // [m]
    int* flag;                       // [m]
    int* ticket;
    int itl, it_is_cap, fun;
    int maxn, hcap, hshift, arena;
    double tol;
};

// eigenvalues d and eigenvectors (Q, lane k owns row k) of the symmetric tridiagonal part of H (Hessenberg columns of
// it1 + 1): the tql2 loop of warp_tridiag_fx, run by ONE warp without a barrier.
__device__ __forceinline__ void hl_warp_tql2(const double* H, int it1, int n, double* Q, double* dout) {
    const int lane = threadIdx.x & 31;
    double d[EL_IT], e[EL_IT];
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        d[i] = H[(int64_t)i * (it1 + 1) + i];
        e[i] = i + 1 < n ? 0.5 * (H[(int64_t)i * (it1 + 1) + i + 1] + H[(int64_t)(i + 1) * (it1 + 1) + i]) : 0.0;
    }
    if (lane < n)
        for (int i = 0; i < n; ++i) Q[lane * EL_LDQ + i] = lane == i ? 1.0 : 0.0;
    double f = 0.0, tst1 = 0.0;
    const double eps = 2.220446049250313e-16;
#pragma unroll 1
    for (int l = 0; l < n; ++l) {
        tst1 = fmax(tst1, fabs(d[l]) + fabs(e[l]));
        int m = l;
        while (m < n) {
            if (fabs(e[m]) <= eps * tst1) break;
            ++m;
        }
        if (m > l) {
            int iter = 0;
            do {
                ++iter;
                double g = d[l];
                double p = (d[l + 1] - g) / (2.0 * e[l]);
                double r = sqrt(fma(p, p, 1.0));
                if (p < 0.0) r = -r;
                d[l] = e[l] / (p + r);
                d[l + 1] = e[l] * (p + r);
                const double dl1 = d[l + 1];
                double h = g - d[l];
                for (int i = l + 2; i < n; ++i) d[i] -= h;
                f += h;
                p = d[m];
                double c = 1.0, c2 = 1.0, c3 = 1.0, s = 0.0, s2 = 0.0;
                const double el1 = e[l + 1];
#pragma unroll 1
                for (int i = m - 1; i >= l; --i) {
                    c3 = c2;
                    c2 = c;
                    s2 = s;
                    g = c * e[i];
                    h = c * p;
                    const double r2 = fma(p, p, e[i] * e[i]);
                    const double rinv = rsqrt(r2);
                    r = r2 * rinv;
                    e[i + 1] = s * r;
                    s = e[i] * rinv;
                    c = p * rinv;
                    p = c * d[i] - s * g;
                    d[i + 1] = h + s * (c * g + s * d[i]);
                    if (lane < n) {
                        const double q1 = Q[lane * EL_LDQ + i + 1], q0 = Q[lane * EL_LDQ + i];
                        Q[lane * EL_LDQ + i + 1] = s * q0 + c * q1;
                        Q[lane * EL_LDQ + i] = c * q0 - s * q1;
                    }
                }
                p = -s * s2 * c3 * el1 * e[l] / dl1;
                e[l] = s * p;
                d[l] = c * p;
            } while (fabs(e[l]) > eps * tst1 && iter < 60);
        }
        d[l] += f;
        e[l] = 0.0;
    }
    if (lane < n) dout[lane] = d[lane];
    __syncwarp();
}

__host__ __device__ inline int hl_scratch_doubles(int itl) {
    const int it1 = itl + 1;
    return 2 * it1 * (it1 + 1) + 2 * EL_IT * EL_LDQ + 2 * EL_IT + 5 * HL_X + EL_IT * HL_LDG;
}

inline size_t hessp_local_smem(int itl, const HesspLocalBudget& b) {
    return (size_t)(2 * b.arena + hl_scratch_doubles(itl)) * sizeof(double) + (size_t)(2 * b.hcap + 3 * b.maxn) * sizeof(int);
}

__global__ void __launch_bounds__(JAC_THREADS)
hessp_local_kernel(CsrDevView A, HesspLocalArgs a) {
    extern __shared__ double dyn[];
    __shared__ JacobiShared sh;
    __shared__ int s_pair, s_m, s_over;
    __shared__ int off[EL_IT + 2], len[EL_IT + 2];
    __shared__ double hcoef[2][EL_IT + 1];
    __shared__ double s_r[2];
    const int it1 = a.itl + 1;
    double* arU = dyn;
    double* arV = arU + a.arena;
    double* HlU = arV + a.arena;                        // it1 columns of it1 + 1
    double* HlV = HlU + it1 * (it1 + 1);
    double* QU = HlV + it1 * (it1 + 1);                 // EL_IT x EL_LDQ
    double* QV = QU + EL_IT * EL_LDQ;
    double* lam = QV + EL_IT * EL_LDQ;
    double* mu = lam + EL_IT;
    double* ring = mu + EL_IT;                          // 4 x HL_X: X of steps jj & 3
    double* T = ring + 4 * HL_X;                        // HL_X
    double* G = T + HL_X;                               // EL_IT x HL_LDG
    int* keys = reinterpret_cast<int*>(G + EL_IT * HL_LDG);
    int* vals = keys + a.hcap;
    int* L = vals + a.hcap;
    int* rs = L + a.maxn;
    int* rl = rs + a.maxn;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = JAC_THREADS / 32;
    const int hmask = a.hcap - 1;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_pair = atomicAdd(a.ticket, 1);
        __syncthreads();
        if (s_pair >= (a.sel ? a.nsel : a.m)) return;
        const int h = a.sel ? a.sel[s_pair] : s_pair;
        const int gi = (int)(a.omega[h] - 1), gj = (int)(a.omega[a.m + h] - 1);
        for (int i = tid; i < a.hcap; i += JAC_THREADS) keys[i] = -1;
        for (int i = tid; i < 2 * it1 * (it1 + 1); i += JAC_THREADS) HlU[i] = 0.0;
        __syncthreads();
        // level 0: {i, j} sorted by global id
        if (tid == 0) {
            const int g0 = min(gi, gj), g1 = max(gi, gj);
            const int nl = g0 == g1 ? 1 : 2;
            for (int t = 0; t < nl; ++t) {
                const int g = t == 0 ? g0 : g1;
                unsigned s = el_hash(g, a.hshift);
                while (keys[s] != -1) s = (s + 1) & hmask;
                keys[s] = g;
                vals[s] = t;
                L[t] = g;
                const int sp = A.row_pos[g];
                rs[t] = A.row_ptr[sp];
                rl[t] = A.row_ptr[sp + 1] - rs[t];
            }
            s_m = nl;
            s_over = 0;
            off[0] = 0;
            len[0] = nl;
            const int li = gi == g0 ? 0 : 1, lj = gj == g0 ? 0 : 1;
            arU[0] = li == 0 ? 1.0 : 0.0;
            arV[0] = lj == 0 ? 1.0 : 0.0;
            if (nl == 2) { arU[1] = li == 1 ? 1.0 : 0.0; arV[1] = lj == 1 ? 1.0 : 0.0; }
        }
        __syncthreads();
        int nsteps = 0, lev_begin = 0;
        bool over = false, done = false;
        for (int j = 0; j < a.itl; ++j) {
            // ---- next BFS level (as entries_local_kernel)
            const int m_old = s_m;
            __syncthreads();
            for (int idx = lev_begin + tid; idx < m_old; idx += JAC_THREADS) {
                const int p0 = rs[idx], p1 = p0 + rl[idx];
                for (int p = p0; p < p1; ++p) {
                    if (*(volatile int*)&s_m >= a.maxn) { s_over = 1; break; }
                    const int g = A.col[p];
                    unsigned s = el_hash(g, a.hshift);
                    for (;;) {
                        const int k = atomicCAS(&keys[s], -1, g);
                        if (k == -1) {
                            const int t = atomicAdd(&s_m, 1);
                            if (t < a.maxn) L[t] = g; else s_over = 1;
                            break;
                        }
                        if (k == g) break;
                        s = (s + 1) & hmask;
                    }
                }
            }
            __syncthreads();
            const int m = s_m;
            if (s_over || off[j] + len[j] + m > a.arena) { over = true; break; }
            const int nnew = m - m_old;
            for (int i = tid; i < nnew; i += JAC_THREADS) {
                const int g = L[m_old + i];
                int rank = 0;
                for (int q = 0; q < nnew; ++q) rank += L[m_old + q] < g;
                rl[m_old + rank] = g;
            }
            __syncthreads();
            for (int i = m_old + tid; i < m; i += JAC_THREADS) {
                const int g = rl[i];
                L[i] = g;
                unsigned s = el_hash(g, a.hshift);
                while (keys[s] != g) s = (s + 1) & hmask;
                vals[s] = i;
                rs[i] = A.row_ptr[A.row_pos[g]];
            }
            __syncthreads();
            for (int i = m_old + tid; i < m; i += JAC_THREADS) rl[i] = A.row_ptr[A.row_pos[L[i]] + 1] - rs[i];
            if (tid == 0) {
                off[j + 1] = off[j] + len[j];
                len[j + 1] = m;
            }
            __syncthreads();
            lev_begin = m_old;
            // ---- both spaces: w = A v_j, CGS2 + third pass (arnoldi_krylov.m:104-106)
            const int lj = len[j];
            for (int r = tid; r < m; r += JAC_THREADS) {
                const int p0 = rs[r], p1 = p0 + rl[r];
                double su = 0.0, sv = 0.0;
                for (int p = p0; p < p1; ++p) {
                    const int li = el_lookup(keys, vals, A.col[p], a.hshift, hmask);
                    if (li >= 0 && li < lj) {
                        const double v = A.val ? A.val[p] : A.uval;
                        su += v * arU[off[j] + li];
                        sv += v * arV[off[j] + li];
                    }
                }
                arU[off[j + 1] + r] = su;
                arV[off[j + 1] + r] = sv;
            }
            __syncthreads();
            for (int pass = 0; pass < 3; ++pass) {
                for (int q = warp; q < 2 * (j + 1); q += NW) {
                    const int sp = q & 1, l = q >> 1;
                    const double* ar = sp ? arV : arU;
                    const double* vl = ar + off[l];
                    const double* w = ar + off[j + 1];
                    double s = 0.0;
                    for (int i = lane; i < len[l]; i += 32) s += vl[i] * w[i];
                    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane == 0) hcoef[sp][l] = s;
                }
                __syncthreads();
                for (int i = tid; i < m; i += JAC_THREADS) {
                    double xu = arU[off[j + 1] + i], xv = arV[off[j + 1] + i];
                    for (int l = 0; l <= j; ++l)
                        if (i < len[l]) {
                            xu -= hcoef[0][l] * arU[off[l] + i];
                            xv -= hcoef[1][l] * arV[off[l] + i];
                        }
                    arU[off[j + 1] + i] = xu;
                    arV[off[j + 1] + i] = xv;
                }
                if (tid < 2 * (j + 1)) {
                    const int sp = tid & 1, l = tid >> 1;
                    double* Hc = (sp ? HlV : HlU) + j * (it1 + 1);
                    if (pass == 0) Hc[l] = hcoef[sp][l];
                    else if (pass == 1) Hc[l] += hcoef[sp][l];
                    else Hc[l] += hcoef[sp][l] * s_r[sp];
                }
                __syncthreads();
                if (pass == 1) {
                    for (int sp = 0; sp < 2; ++sp) {
                        double* w = (sp ? arV : arU) + off[j + 1];
                        double s = 0.0;
                        for (int i = tid; i < m; i += JAC_THREADS) s += w[i] * w[i];
                        s = block_sum(s, sh.red);
                        const double r = sqrt(s);
                        const double inv = r > 0.0 ? 1.0 / r : 0.0;
                        for (int i = tid; i < m; i += JAC_THREADS) w[i] *= inv;
                        if (tid == 0) {
                            s_r[sp] = r;
                            (sp ? HlV : HlU)[j * (it1 + 1) + j + 1] = r;
                        }
                        __syncthreads();
                    }
                }
            }
            // ---- X_h by Daleckii-Krein (frechet.cuh), then the lag-3 rule
            const int jj = j + 1;
            if (warp == 0) hl_warp_tql2(HlU, it1, jj, QU, lam);
            else if (warp == 1) hl_warp_tql2(HlV, it1, jj, QV, mu);
            __syncthreads();
            for (int e = tid; e < jj * jj; e += JAC_THREADS) {
                const int x = e % jj, y = e / jj;
                T[x + y * jj] = divided_difference(a.fun, lam[x], mu[y]) * QU[0 * EL_LDQ + x] * QV[0 * EL_LDQ + y];
            }
            __syncthreads();
            for (int e = tid; e < jj * jj; e += JAC_THREADS) {     // G <- P T (P(r, k) = QU[r * EL_LDQ + k])
                const int r = e % jj, c = e / jj;
                double s = 0.0;
                for (int k = 0; k < jj; ++k) s += QU[r * EL_LDQ + k] * T[k + c * jj];
                G[r + c * HL_LDG] = s;
            }
            __syncthreads();
            double* cur = ring + (jj & 3) * HL_X;
            for (int e = tid; e < jj * jj; e += JAC_THREADS) {     // X = G Q'
                const int r = e % jj, c = e / jj;
                double s = 0.0;
                for (int k = 0; k < jj; ++k) s += G[r + k * HL_LDG] * QV[c * EL_LDQ + k];
                cur[r + c * jj] = s;
            }
            __syncthreads();
            bool conv = false;
            if (jj > 3) {
                const double* old = ring + ((jj - 3) & 3) * HL_X;
                const int on = jj - 3;
                for (int e = tid; e < jj * jj; e += JAC_THREADS) {
                    const int r = e % jj, c = e / jj;
                    T[r + c * jj] = cur[r + c * jj] - ((r < on && c < on) ? old[r + c * on] : 0.0);
                }
                __syncthreads();
                for (int e = tid; e < jj * jj; e += JAC_THREADS) { // G <- D' D
                    const int r = e % jj, c = e / jj;
                    double s = 0.0;
                    for (int k = 0; k < jj; ++k) s += T[k + r * jj] * T[k + c * jj];
                    G[r + c * HL_LDG] = s;
                }
                __syncthreads();
                block_jacobi(G, jj, HL_LDG, nullptr, 0, &sh);
                double mx = 0.0;
                for (int i = tid; i < jj; i += JAC_THREADS) mx = fmax(mx, G[i + i * HL_LDG]);
                for (int o = 16; o; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                __syncthreads();
                if (lane == 0) sh.red[warp] = mx;
                __syncthreads();
                for (int w = 0; w < NW; ++w) mx = fmax(mx, sh.red[w]);
                conv = !(sqrt(fmax(mx, 0.0)) > a.tol);
            }
            nsteps = jj;
            __syncthreads();
            if (conv) { done = true; break; }
        }
        if (over || (!done && !a.it_is_cap)) {
            if (tid == 0) { a.flag[h] = over ? 1 : 2; a.steps[h] = 0; }
            continue;
        }
        // ---- W(h, r) = -2 sum_a sum_b S_r(a, b) U(a,:) X V(b,:)'; r in groups of 8, one fixed-order block sum each
        const int s = nsteps, mb = len[s - 1];                   // U's rows: the ball after s - 1 levels
        const double* X = ring + (s & 3) * HL_X;
        for (int r0 = 0; r0 < a.p; r0 += 8) {
            double acc[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[q] = 0.0;
            for (int la = tid; la < mb; la += JAC_THREADS) {
                const int g = L[la];
                const int e0 = a.srow[g], e1 = a.srow[g + 1];
                if (e0 == e1) continue;
                double ux[EL_IT];                              // U(a,:) X
                for (int c = 0; c < s; ++c) ux[c] = 0.0;
                for (int k = 0; k < s; ++k) {
                    if (la >= len[k]) continue;
                    const double u = arU[off[k] + la];
                    for (int c = 0; c < s; ++c) ux[c] += u * X[k + c * s];
                }
                for (int e = e0; e < e1; ++e) {
                    const int lb = el_lookup(keys, vals, a.scol[e], a.hshift, hmask);
                    if (lb < 0) continue;
                    double gsum = 0.0;
                    for (int c = 0; c < s; ++c)
                        if (lb < len[c]) gsum += ux[c] * arV[off[c] + lb];
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (r0 + q < a.p) acc[q] += gsum * a.sval[(int64_t)e * a.p + r0 + q];
                }
            }
            for (int q = 0; q < 8 && r0 + q < a.p; ++q) {
                const double t = block_sum(acc[q], sh.red);
                if (tid == 0) a.W[h + (int64_t)(r0 + q) * a.m] = -2.0 * t;
            }
        }
        if (tid == 0) { a.flag[h] = 0; a.steps[h] = nsteps; }
    }
}

struct HesspLocalResult {
    std::vector<int> steps, flag;    // [m]
    int tier_pairs[HL_NTIERS] = {};
};

// omega: m x 2 col-major (1-based, checked); S by global row (srow [n + 1], scol, sval [nnzS * p]); W (host, m x p, ld
// ldw) gets the rows of the pairs with flag 0.
inline HesspLocalResult hessp_local_run(kr_ctx* ctx, const CsrDev& M, int64_t m, const int64_t* omega,
                                        const std::vector<int>& srow, const std::vector<int>& scol,
                                        const std::vector<double>& sval, int p, int fun, double tol, int it, double* W,
                                        int64_t ldw) {
    HesspLocalResult out;
    DevBuf<int64_t> dom(ctx, 2 * m);
    DevBuf<int> dsrow(ctx, srow.size()), dscol(ctx, scol.size()), dstate(ctx, (size_t)2 * m + 1);
    DevBuf<double> dsval(ctx, sval.size()), dW(ctx, (size_t)m * p);
    dom.upload(omega, 2 * m);
    dsrow.upload(srow.data(), srow.size());
    dscol.upload(scol.data(), scol.size());
    dsval.upload(sval.data(), sval.size());
    dstate.zero();
    dW.zero();
    HesspLocalArgs a;
    a.omega = dom.p;
    a.m = (int)m;
    a.srow = dsrow.p;
    a.scol = dscol.p;
    a.sval = dsval.p;
    a.p = p;
    a.W = dW.p;
    a.steps = dstate.p;
    a.flag = dstate.p + m;
    a.ticket = dstate.p + 2 * m;
    a.itl = std::min(it, EL_IT);
    a.it_is_cap = it <= EL_IT;
    a.fun = fun;
    a.tol = tol;
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(hessp_local_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)hessp_local_smem(EL_IT, HL_TIERS[HL_NTIERS - 1])));
    DevBuf<int> dsel;
    std::vector<int> sel;
    for (int tier = 0; tier < HL_NTIERS; ++tier) {
        const HesspLocalBudget& b = HL_TIERS[tier];
        a.maxn = b.maxn;
        a.hcap = b.hcap;
        a.arena = b.arena;
        a.hshift = 32;
        for (int hh = b.hcap; hh > 1; hh >>= 1) a.hshift--;
        a.sel = sel.empty() ? nullptr : dsel.p;
        a.nsel = (int)sel.size();
        const int todo = sel.empty() ? (int)m : (int)sel.size();
        const size_t smem = hessp_local_smem(a.itl, b);
        const int per_sm = std::max(1, (int)((size_t)228 * 1024 / (smem + 4096 + 1024)));
        const int ctas = (int)std::min<int64_t>(todo, (int64_t)ctx->num_sms * per_sm);
        KR_CUDA(cudaMemsetAsync(a.ticket, 0, sizeof(int), ctx->stream));
        out.tier_pairs[tier] = todo;
        KR_LAUNCH(ctx, hessp_local_kernel, ctas, JAC_THREADS, smem, M.view(), a);
        if (tier == HL_NTIERS - 1) break;
        std::vector<int> fl(m);
        KR_CUDA(cudaMemcpyAsync(fl.data(), a.flag, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        sel.clear();
        for (int64_t q = 0; q < m; ++q)
            if (fl[q] == 1) sel.push_back((int)q);
        if (sel.empty()) break;
        dsel.reset(ctx, sel.size());
        dsel.upload(sel.data(), sel.size());
    }
    std::vector<int> st = dstate.to_host();
    out.steps.assign(st.begin(), st.begin() + m);
    out.flag.assign(st.begin() + m, st.begin() + 2 * m);
    std::vector<double> Wh = dW.to_host();
    for (int r = 0; r < p; ++r)
        for (int64_t q = 0; q < m; ++q)
            if (out.flag[q] == 0) W[q + (int64_t)r * ldw] = Wh[q + (int64_t)r * m];
    return out;
}

}  // namespace kr
