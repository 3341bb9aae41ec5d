// entries_local.cuh - function_multiple_entries (functions/function_multiple_entries.m:86-164) on graphs whose Krylov
// vectors stay LOCAL: the j-th basis vector of K(A, e_h) lives on the nodes within j hops of h, and on a road network
// (config C2: datasets_paper/Transport, degree 2-3) sixteen hops reach a few hundred of the 10^5 nodes.  The dense
// batch of entries.cuh streams n rows per column per pass for them; here ONE CTA runs the whole Arnoldi process of a
// column in shared memory on the ball around h:
//   * the ball grows one BFS level per step (hash table global id -> local index; a new level is sorted by global id,
//     so the local numbering - and with it every summation order - is deterministic),
//   * local index order = BFS order, so basis vector l is stored with |ball(l)| entries only (a triangular arena),
//   * w = A v_j by rows in stored CSR order, CGS2 + the third pass of arnoldi_krylov.m:104-106 (all inner products of
//     a pass before its update, as the reference), the projected solve by one warp + the lag-3 stop of entries_stop_test,
//   * the requested entries f(A)(h, j2) = sum_l V_l(j2) x_l straight from the arena.
// Columns are handed out by a ticket counter.  A column whose ball outgrows the CTA's budget is flagged and run again with
// the next budget tier; one that outgrows the last tier (or that has not stopped after EL_IT steps while the caller allows
// more) goes through the dense batch: results do not depend
// on which path a column took beyond rounding (test_gpu_krylov.py::test_function_multiple_entries_local_vs_dense).
// Needs a symmetric stored pattern (w's support is found from the rows of v's support) and no pending edge edits.
// The direction flavour (DIR = true, kr_trace_fun_sparse_update) runs column c on A_t = A + (t_c - 1) D instead, where D
// is given by its values aligned with the stored CSR (zero where D has no entry): one launch serves every quadrature node.
#pragma once
#include <type_traits>
#include "entries.cuh"

namespace kr {

// Budget of a CTA: nodes of a ball, hash slots (power of two, > maxn + CTA threads: the table never fills up), doubles of
// basis storage (sum over l of |ball(l)|).  Two tiers: most spaces of a road network fit the small one (five CTAs per
// SM); what it flags is run again with the next one (three CTAs per SM, then one); what the last one flags takes the dense batch.
struct EntriesLocalBudget { int maxn, hcap, arena; };
constexpr int EL_NTIERS = 3;
constexpr EntriesLocalBudget EL_TIERS[EL_NTIERS] = {{384, 1024, 2048}, {768, 2048, 4096}, {1536, 4096, 16384}};
constexpr int EL_IT = 24;            // steps a column may take on this path

struct EntriesLocalArgs {
    const int64_t* rows;             // [R] 1-based start nodes
    const int* pair_begin;           // [R + 1] pairs of column c: pair_list[pair_begin[c] .. pair_begin[c+1])
    const int* pair_list;            // pair numbers sorted by column
    const int64_t* j2;               // [k] 1-based second index of every pair
    double* X;                       // [k]
    int* steps;                      // [R] steps taken (reference's per-space iteration count)
    int* flag;                       // [R] nonzero = not handled here (1: ball outgrew the budget, 2: step limit of this path)
    int* ticket;
    int R, itl, it_is_cap, fun;      // itl = min(it, EL_IT); it_is_cap: it <= EL_IT (running out of steps is final)
    int maxn, hcap, hshift, arena;   // budget (hshift = 32 - log2 hcap)
    const int* sel;                  // columns to process (null: all of 0..R-1)
    int nsel;
    double tol;
};

// The direction flavour's arguments (a separate type: the default flavour's parameter block stays as it was)
struct EntriesLocalDirArgs : EntriesLocalArgs {
    const double* tcol;              // [R] t of column c
    const double* dval;              // [nnz] D's values in stored CSR order
};
template <bool DIR> using EntriesLocalArgsOf = std::conditional_t<DIR, EntriesLocalDirArgs, EntriesLocalArgs>;

__device__ __forceinline__ unsigned el_hash(int g, int hshift) { return ((unsigned)g * 2654435761u) >> hshift; }

__device__ __forceinline__ int el_lookup(const int* keys, const int* vals, int g, int hshift, int hmask) {
    unsigned s = el_hash(g, hshift);
    for (;;) {
        const int k = keys[s];
        if (k == g) return vals[s];
        if (k == -1) return -1;
        s = (s + 1) & hmask;
    }
}

constexpr int EL_LDQ = EL_IT + 1;   // odd: the lanes' rows of Q fall into different banks
static_assert(EL_IT <= 32 && (EL_LDQ & 1) == 1, "one lane per row of Q");
__host__ __device__ inline int el_scratch_doubles(int itl) { return itl * EL_LDQ + itl; }   // Q (itl x EL_LDQ) + x

// x = f(T) e1 for the symmetric tridiagonal part T of the projection (diagonal H(i,i), off-diagonal the mean of H(i+1,i)
// and H(i,i+1)): implicit QL with eigenvector accumulation (EISPACK tql2) run by ONE warp without any barrier - every
// lane carries the scalar recurrence redundantly in private copies of d / e, lane k owns row k of Q.  With full
// re-orthogonalisation on a symmetric A the entries of H outside the band are rounding noise (1e-16 ||A||), so this equals
// the dense path's Jacobi solve of (H + H')/2 to rounding; the warp-local form has no CTA barrier per rotation round.
__device__ __forceinline__ void warp_tridiag_fx(const double* H, int it1, int n, int fun, double* Q, double* x) {
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
                    // r = |(p, e_i)| and the rotation from one reciprocal square root (entries are O(||A||): no scaling)
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
    __syncwarp();
    if (lane < n) {
        double sum = 0.0;
        for (int k = 0; k < n; ++k) sum += Q[lane * EL_LDQ + k] * fun_eval(fun, d[k]) * Q[k];
        x[lane] = sum;
    }
}

// The same x = f(T) e1 without an eigen-decomposition: f is exp / sinh / cosh, so x comes from y+ = e^{T} e1 and
// y- = e^{-T} e1, each evaluated as (e^{T/s})^s e1 with s = ceil(||T||_inf) and a degree-20 Taylor polynomial per stage
// (||T/s|| <= 1: truncation 1/21! = 2e-20, no cancellation; the scheme of expmv.m:62-90 with theta = 1).  Lane i holds
// component i, a product with the tridiagonal T is two shuffles and three multiply-adds: 20 s short dependent steps
// instead of the ~2 n^2 dependent rotations of the QL solve.  Returns false (nothing written) when s would exceed
// EL_TAYLOR_MAX_S; the caller then takes the QL solve.
constexpr int EL_TAYLOR_MAX_S = 48;
__device__ __forceinline__ bool warp_tridiag_fx_taylor(const double* H, int it1, int n, int fun, double* x) {
    const int lane = threadIdx.x & 31;
    const unsigned full = 0xffffffffu;
    const double di = lane < n ? H[(int64_t)lane * (it1 + 1) + lane] : 0.0;
    const double eu = lane + 1 < n ? 0.5 * (H[(int64_t)lane * (it1 + 1) + lane + 1] + H[(int64_t)(lane + 1) * (it1 + 1) + lane]) : 0.0;
    double el = __shfl_up_sync(full, eu, 1);
    if (lane == 0) el = 0.0;
    double rho = fabs(di) + fabs(eu) + fabs(el);
    for (int o = 16; o; o >>= 1) rho = fmax(rho, __shfl_xor_sync(full, rho, o));
    if (!(rho <= (double)EL_TAYLOR_MAX_S)) return false;          // also catches NaN
    const int ns = rho > 1.0 ? (int)ceil(rho) : 1;
    const double inv_s = 1.0 / (double)ns;
    const bool both = fun != KR_FUN_EXP;
    double yp = lane == 0 ? 1.0 : 0.0, ym = yp;
    if (ns == 1) {
        // no scaling: the even / odd terms of the one series are cosh / sinh themselves (no cancellation for small ||T||)
        double tp = yp, ev = yp, od = 0.0;
#pragma unroll 4
        for (int k = 1; k <= 20; ++k) {
            const double up = __shfl_up_sync(full, tp, 1), dn = __shfl_down_sync(full, tp, 1);
            tp = (di * tp + el * up + eu * dn) * (1.0 / (double)k);
            if (k & 1) od += tp; else ev += tp;
        }
        if (lane < n) x[lane] = fun == KR_FUN_EXP ? ev + od : fun == KR_FUN_SINH ? od : ev;
        return true;
    }
#pragma unroll 1
    for (int stage = 0; stage < ns; ++stage) {
        double tp = yp, tm = ym;
#pragma unroll 4
        for (int k = 1; k <= 20; ++k) {
            const double ck = inv_s / (double)k;
            const double up = __shfl_up_sync(full, tp, 1), dn = __shfl_down_sync(full, tp, 1);
            tp = (di * tp + el * up + eu * dn) * ck;
            yp += tp;
            if (both) {
                const double um = __shfl_up_sync(full, tm, 1), dm = __shfl_down_sync(full, tm, 1);
                tm = -(di * tm + el * um + eu * dm) * ck;
                ym += tm;
            }
        }
    }
    if (lane < n) x[lane] = fun == KR_FUN_EXP ? yp : fun == KR_FUN_SINH ? 0.5 * (yp - ym) : 0.5 * (yp + ym);
    return true;
}

template <bool DIR>
__global__ void __launch_bounds__(JAC_THREADS)
entries_local_kernel(CsrDevView A, EntriesLocalArgsOf<DIR> a) {
    extern __shared__ double dyn[];
    __shared__ JacobiShared sh;
    __shared__ int s_col, s_m, s_over;
    __shared__ int off[EL_IT + 2], len[EL_IT + 2];
    __shared__ double hcoef[EL_IT + 1];
    __shared__ double s_r;
    const int it1 = a.itl + 1;
    double* arena = dyn;
    double* Hl = arena + a.arena;                        // it1 columns of it1 + 1
    double* ring = Hl + it1 * (it1 + 1);                  // 4 x it1
    double* Q = ring + 4 * it1;                          // QL fallback: itl x EL_LDQ
    double* fx = Q + a.itl * EL_LDQ;                     // f(T) e1 of the latest step
    int* keys = reinterpret_cast<int*>(Q + el_scratch_doubles(a.itl));
    int* vals = keys + a.hcap;
    int* L = vals + a.hcap;                              // global ids in local order
    int* rs = L + a.maxn;                                // first stored nonzero of the node's row
    int* rl = rs + a.maxn;                               // its length (also the sort buffer of a new level)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = JAC_THREADS / 32;
    const int hmask = a.hcap - 1;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_col = atomicAdd(a.ticket, 1);
        __syncthreads();
        if (s_col >= (a.sel ? a.nsel : a.R)) return;
        const int c = a.sel ? a.sel[s_col] : s_col;
        // ---- reset
        for (int i = tid; i < a.hcap; i += JAC_THREADS) keys[i] = -1;
        for (int i = tid; i < it1 * (it1 + 1); i += JAC_THREADS) Hl[i] = 0.0;
        for (int i = tid; i < 4 * it1; i += JAC_THREADS) ring[i] = 0.0;
        __syncthreads();
        const int h0 = (int)(a.rows[c] - 1);
        double tm1 = 0.0;
        const double* dv = nullptr;
        if constexpr (DIR) {
            tm1 = a.tcol[c] - 1.0;
            dv = a.dval;
        }
        if (tid == 0) {
            const unsigned s = el_hash(h0, a.hshift);
            keys[s] = h0;
            vals[s] = 0;
            L[0] = h0;
            const int sp = A.row_pos[h0];
            rs[0] = A.row_ptr[sp];
            rl[0] = A.row_ptr[sp + 1] - rs[0];
            s_m = 1;
            s_over = 0;
            off[0] = 0;
            len[0] = 1;
            arena[0] = 1.0;
        }
        __syncthreads();
        int nsteps = 0;
        bool over = false, done = false;
        int lev_begin = 0;                                 // first local index of the newest BFS level
        for (int j = 0; j < a.itl; ++j) {
            // ---- next BFS level: neighbours of level j that are not in the ball yet
            const int m_old = s_m;
            __syncthreads();
            for (int idx = lev_begin + tid; idx < m_old; idx += JAC_THREADS) {
                const int p0 = rs[idx], p1 = p0 + rl[idx];
                for (int p = p0; p < p1; ++p) {
                    // a full ball stops the insertions at once (the table must never fill up: hub rows)
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
            // ---- sort the new level by global id (rank sort; a level has tens of nodes), then index it
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
                const int sp = A.row_pos[g];
                rs[i] = A.row_ptr[sp];
            }
            __syncthreads();
            for (int i = m_old + tid; i < m; i += JAC_THREADS) rl[i] = A.row_ptr[A.row_pos[L[i]] + 1] - rs[i];
            if (tid == 0) {
                off[j + 1] = off[j] + len[j];
                len[j + 1] = m;
            }
            __syncthreads();
            lev_begin = m_old;
            // ---- w = A v_j on the ball (rows in stored order; v_j is zero beyond len[j])
            const double* vj = arena + off[j];
            const int lj = len[j];
            double* w = arena + off[j + 1];
            for (int r = tid; r < m; r += JAC_THREADS) {
                const int p0 = rs[r], p1 = p0 + rl[r];
                double s = 0.0;
                for (int p = p0; p < p1; ++p) {
                    const int li = el_lookup(keys, vals, A.col[p], a.hshift, hmask);
                    if (li >= 0 && li < lj) {
                        double v = A.val ? A.val[p] : A.uval;
                        if (DIR) v = fma(tm1, dv[p], v);
                        s += v * vj[li];
                    }
                }
                w[r] = s;
            }
            __syncthreads();
            // ---- CGS2 + third pass against V_0..V_j (arnoldi_krylov.m:104-106, :119-125)
            double* Hcol = Hl + j * (it1 + 1);
            for (int pass = 0; pass < 3; ++pass) {
                for (int l = warp; l <= j; l += NW) {
                    const double* vl = arena + off[l];
                    const int ll = len[l];
                    double s = 0.0;
                    for (int i = lane; i < ll; i += 32) s += vl[i] * w[i];
                    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane == 0) hcoef[l] = s;
                }
                __syncthreads();
                for (int i = tid; i < m; i += JAC_THREADS) {
                    double x = w[i];
                    for (int l = 0; l <= j; ++l)
                        if (i < len[l]) x -= hcoef[l] * arena[off[l] + i];
                    w[i] = x;
                }
                if (tid <= j) {
                    if (pass == 0) Hcol[tid] = hcoef[tid];
                    else if (pass == 1) Hcol[tid] += hcoef[tid];
                    else Hcol[tid] += hcoef[tid] * s_r;
                }
                __syncthreads();
                if (pass == 1) {
                    double s = 0.0;
                    for (int i = tid; i < m; i += JAC_THREADS) s += w[i] * w[i];
                    s = block_sum(s, sh.red);
                    const double r = sqrt(s);
                    const double inv = r > 0.0 ? 1.0 / r : 0.0;
                    for (int i = tid; i < m; i += JAC_THREADS) w[i] *= inv;
                    if (tid == 0) {
                        s_r = r;
                        Hcol[j + 1] = r;
                    }
                    __syncthreads();
                }
            }
            // ---- projected problem and stopping test
            const int jj = j + 1;
            if (warp == 0 && !warp_tridiag_fx_taylor(Hl, it1, jj, a.fun, fx)) warp_tridiag_fx(Hl, it1, jj, a.fun, Q, fx);
            __syncthreads();
            done = entries_stop_test(fx, it1, jj, a.tol, ring, &sh);
            nsteps = jj;
            __syncthreads();
            if (done) break;
        }
        if (over || (!done && !a.it_is_cap)) {
            if (tid == 0) { a.flag[c] = over ? 1 : 2; a.steps[c] = 0; }     // 1: a larger budget may do, 2: needs more steps
            continue;
        }
        // ---- entries: X[p] = sum_{l < nsteps} V_l(j2) x_l     (function_multiple_entries.m:162-164)
        for (int q = a.pair_begin[c] + tid; q < a.pair_begin[c + 1]; q += JAC_THREADS) {
            const int p = a.pair_list[q];
            const int li = el_lookup(keys, vals, (int)(a.j2[p] - 1), a.hshift, hmask);
            double s = 0.0;
            if (li >= 0)
                for (int l = 0; l < nsteps; ++l)
                    if (li < len[l]) s += arena[off[l] + li] * fx[l];
            a.X[p] = s;
        }
        if (tid == 0) { a.flag[c] = 0; a.steps[c] = nsteps; }
    }
}

struct EntriesLocalResult {
    std::vector<double> X;           // [k], valid where flag[colof[p]] == 0 (empty for the direction flavour)
    std::vector<int> steps, flag;    // [R]
    int tier_cols[EL_NTIERS] = {};   // columns launched per budget tier
};

// Direction flavour: column c runs on A + (t[c] - 1) D (device arrays; d aligned with the stored CSR) and the entries
// stay on the device in X (device, [k]).
struct EntriesLocalDir { const double* t; const double* d; double* X; };

inline size_t entries_local_smem(int itl, const EntriesLocalBudget& b) {
    const int it1 = itl + 1;
    return (size_t)(b.arena + it1 * (it1 + 1) + 4 * it1 + el_scratch_doubles(itl)) * sizeof(double) +
           (size_t)(2 * b.hcap + 3 * b.maxn) * sizeof(int);
}

// rows: distinct first indices (1-based); colof[p]: column of pair p; j2[p]: second index (1-based)
inline EntriesLocalResult entries_local_run(kr_ctx* ctx, const CsrDev& M, const std::vector<int64_t>& rows,
                                            const std::vector<int>& colof, const std::vector<int64_t>& j2, int fun,
                                            double tol, int it, const EntriesLocalDir* dir = nullptr) {
    const int R = (int)rows.size(), k = (int)colof.size();
    EntriesLocalResult out;
    std::vector<int> pb(R + 1, 0), pl(k);
    for (int p = 0; p < k; ++p) pb[colof[p] + 1]++;
    for (int c = 0; c < R; ++c) pb[c + 1] += pb[c];
    {
        std::vector<int> next(pb.begin(), pb.end() - 1);
        for (int p = 0; p < k; ++p) pl[next[colof[p]]++] = p;
    }
    DevBuf<int64_t> drows(ctx, R), dj2(ctx, k);
    DevBuf<int> dpb(ctx, R + 1), dpl(ctx, k), dstate(ctx, (size_t)2 * R + 1);
    DevBuf<double> dX(ctx, dir ? 0 : k);
    drows.upload(rows.data(), R);
    dj2.upload(j2.data(), k);
    dpb.upload(pb.data(), R + 1);
    dpl.upload(pl.data(), k);
    dstate.zero();
    if (!dir) dX.zero();
    EntriesLocalArgs a;
    a.rows = drows.p;
    a.pair_begin = dpb.p;
    a.pair_list = dpl.p;
    a.j2 = dj2.p;
    a.X = dir ? dir->X : dX.p;
    a.steps = dstate.p;
    a.flag = dstate.p + R;
    a.ticket = dstate.p + 2 * R;
    a.R = R;
    a.itl = std::min(it, EL_IT);
    a.it_is_cap = it <= EL_IT;
    a.fun = fun;
    a.tol = tol;
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device)) {
        const int lim = (int)entries_local_smem(EL_IT, EL_TIERS[EL_NTIERS - 1]);
        KR_CUDA(cudaFuncSetAttribute(entries_local_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        KR_CUDA(cudaFuncSetAttribute(entries_local_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    }
    DevBuf<int> dsel;
    std::vector<int> sel;                                   // empty: all columns
    for (int tier = 0; tier < EL_NTIERS; ++tier) {
        const EntriesLocalBudget& b = EL_TIERS[tier];
        a.maxn = b.maxn;
        a.hcap = b.hcap;
        a.arena = b.arena;
        a.hshift = 32;
        for (int h = b.hcap; h > 1; h >>= 1) a.hshift--;
        if (b.maxn + JAC_THREADS >= b.hcap) fail(KR_ERR_ARG, "entries_local: hash too small for the ball");
        a.sel = sel.empty() ? nullptr : dsel.p;
        a.nsel = (int)sel.size();
        const int todo = sel.empty() ? R : (int)sel.size();
        const size_t smem = entries_local_smem(a.itl, b);
        const int per_sm = std::max(1, (int)((size_t)228 * 1024 / (smem + 4096 + 1024)));      // + static + the per-CTA reserve
        const int ctas = (int)std::min<int64_t>(todo, (int64_t)ctx->num_sms * per_sm);
        KR_CUDA(cudaMemsetAsync(a.ticket, 0, sizeof(int), ctx->stream));
        out.tier_cols[tier] = todo;
        if (dir) {
            EntriesLocalDirArgs da;
            static_cast<EntriesLocalArgs&>(da) = a;
            da.tcol = dir->t;
            da.dval = dir->d;
            KR_LAUNCH(ctx, entries_local_kernel<true>, ctas, JAC_THREADS, smem, M.view(), da);
        } else {
            KR_LAUNCH(ctx, entries_local_kernel<false>, ctas, JAC_THREADS, smem, M.view(), a);
        }
        if (tier == EL_NTIERS - 1) break;
        // what this tier flagged goes to the next one
        std::vector<int> fl(R);
        KR_CUDA(cudaMemcpyAsync(fl.data(), a.flag, (size_t)R * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->counters[4] += (int64_t)R * sizeof(int);
        sel.clear();
        for (int c = 0; c < R; ++c)
            if (fl[c] == 1) sel.push_back(c);
        if (sel.empty()) break;
        dsel.reset(ctx, sel.size());
        dsel.upload(sel.data(), sel.size());
    }
    if (!dir) out.X = dX.to_host();
    std::vector<int> st = dstate.to_host();
    out.steps.assign(st.begin(), st.begin() + R);
    out.flag.assign(st.begin() + R, st.begin() + 2 * R);
    return out;
}

}  // namespace kr
