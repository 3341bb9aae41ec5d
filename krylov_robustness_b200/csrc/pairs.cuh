// pairs.cuh - trace_fun_update for MANY candidate edges at once (the candidate loop of
// functions/krylov_miobi.m:76-99 -> functions/trace_fun_update.m:60-125 -> functions/lanczos_krylov.m:73-101).
//
// A fixed set of SLOTS (two columns each) of three panel-major blocks P (previous basis block), C (current),
// Y (work) is kept busy with candidates until the whole list is scored ("continuous batching"): a slot whose
// candidate has converged is re-seeded with the next candidate of the queue, so every dense pass works on
// columns that are still iterating and the cost is the SUM of the candidates' step counts, not (slowest
// candidate of a chunk) x (chunk width) as in round 1.  Slots at different step numbers coexist: all
// per-candidate state (step count, H blocks, transforms, lag-2 buffer) is indexed by slot.
//
// Basis blocks are never normalised in memory: the orthonormal block is V = raw * T with a per-slot 2x2
// matrix T, so the thin QR of every step costs no pass over the data.
//   step 1 (seed)   U = [e_i e_j]: A*U are two COLUMNS OF A, U'AU four entries of A, and CGS2 leaves exactly
//                   W = A(:, [i j]) with rows i and j zeroed - built straight from the CSR rows (O(deg)), no
//                   SpMM and no dense pass; its Gram is two sparse norms and a sorted-list intersection
//   steps >= 2      pass A  spmm<EpiGram2>: Y = A*C, raw Grams P'Y, C'Y           (CGS pass 1 coefficients)
//                   pass B  W = Y*Ma - P*Mp - C*Mc, raw Grams P'W, C'W            (CGS pass 2 coefficients)
//                   pass C  W = W - P*Mp - C*Mc, Gram W'W                         (R of the thin QR)
// then one small CTA per slot: QR factor from the Gram (Householder conventions of LAPACK for exactly-zero
// columns, see DESIGN.md "rank-deficient blocks"), projected matrices Gm / tGm, two Jacobi eigen-solves, the
// trace formula and the reference's lag-2 stopping rule.
#pragma once
#include "dense.cuh"
#include "smalldense.cuh"

namespace kr {

// W = Y*Ma - P*Mp - C*Mc per candidate (coef[cand][12] = Ma, Mp, Mc row-major 2x2), in place in Y.
// MODE 0: partial[rb][cand][8] = {P'W, C'W};  MODE 1: partial[rb][cand][4] = {w1'w1, w1'w2, w2'w2, 0}
template <int MODE>
__global__ void __launch_bounds__(COL_THREADS)
pair_update_kernel(double* __restrict__ Y, const double* __restrict__ P, const double* __restrict__ C,
                   int64_t n, const double* __restrict__ coef, int ncand, double* __restrict__ partial,
                   const int* __restrict__ panel_active) {
    constexpr int NV = MODE == 0 ? 8 : 4;
    if (!panel_active[blockIdx.y]) return;            // all candidates of this panel have converged
    __shared__ double smem[COL_WARPS * LPT * NV];
    __shared__ double cf[LPT][12];
    const int q = blockIdx.y, sub = threadIdx.x % LPT;
    if (threadIdx.x < LPT * 12) {
        int cand = q * LPT + threadIdx.x / 12;
        cf[threadIdx.x / 12][threadIdx.x % 12] = cand < ncand ? coef[(int64_t)cand * 12 + threadIdx.x % 12] : 0.0;
    }
    __syncthreads();
    const double* m = cf[sub];
    const int64_t po = (int64_t)q * n * PW;
    const int64_t r0 = (int64_t)blockIdx.x * COL_ROWS_PER_CTA;
    const int64_t r1 = min(n, r0 + COL_ROWS_PER_CTA);
    double acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.0;
    for (int64_t r = r0 + (threadIdx.x / LPT); r < r1; r += COL_THREADS / LPT) {
        const int64_t o = po + r * PW + sub * 2;
        double2 y = *reinterpret_cast<const double2*>(Y + o);
        double2 c = *reinterpret_cast<const double2*>(C + o);
        const double2 p = *reinterpret_cast<const double2*>(P + o);
        double2 w;
        w.x = y.x * m[0] + y.y * m[2] - (p.x * m[4] + p.y * m[6]) - (c.x * m[8] + c.y * m[10]);
        w.y = y.x * m[1] + y.y * m[3] - (p.x * m[5] + p.y * m[7]) - (c.x * m[9] + c.y * m[11]);
        *reinterpret_cast<double2*>(Y + o) = w;
        if (MODE == 0) {
            acc[0] += p.x * w.x; acc[1] += p.x * w.y; acc[2] += p.y * w.x; acc[3] += p.y * w.y;
            acc[4] += c.x * w.x; acc[5] += c.x * w.y; acc[6] += c.y * w.x; acc[7] += c.y * w.y;
        } else {
            acc[0] += w.x * w.x; acc[1] += w.x * w.y; acc[2] += w.y * w.y;
        }
    }
    cta_reduce_by_sub<NV>(acc, smem);
    if (threadIdx.x < LPT) {
        int cand = q * LPT + threadIdx.x;
        double* o = partial + ((int64_t)blockIdx.x * (gridDim.y * LPT) + cand) * NV;
#pragma unroll
        for (int i = 0; i < NV; ++i) o[i] = acc[i];
    }
}

// 2x2 helpers, row-major [a b; c d]
__device__ __forceinline__ void mm2(const double* A, const double* B, double* C) {
    double c0 = A[0] * B[0] + A[1] * B[2], c1 = A[0] * B[1] + A[1] * B[3];
    double c2 = A[2] * B[0] + A[3] * B[2], c3 = A[2] * B[1] + A[3] * B[3];
    C[0] = c0; C[1] = c1; C[2] = c2; C[3] = c3;
}
__device__ __forceinline__ void mtm2(const double* A, const double* B, double* C) {   // A' * B
    double c0 = A[0] * B[0] + A[2] * B[2], c1 = A[0] * B[1] + A[2] * B[3];
    double c2 = A[1] * B[0] + A[3] * B[2], c3 = A[1] * B[1] + A[3] * B[3];
    C[0] = c0; C[1] = c1; C[2] = c2; C[3] = c3;
}

struct PairState {
    int nslots, it, fun;
    double tol, b_off;
    // ---- per slot
    long long* cand;  // [nslots] index of the candidate in the caller's list, -1 = idle
    int* ei;          // [nslots] 0-based end points
    int* ej;
    int* step;        // [nslots] block-Lanczos steps completed
    int* flag;        // [nslots] PAIR_IDLE / PAIR_NEW (seeded, step 1 pending) / PAIR_RUN
    double* Tp;       // [nslots][4]
    double* Tc;       // [nslots][4]
    double* hp;       // [nslots][4] accumulated CGS2 coefficients vs previous block (this step)
    double* hc;       // [nslots][4] vs current block
    double* coef;     // [nslots][12]
    double* Hd;       // [nslots][it][4] diagonal blocks
    double* Hs;       // [nslots][it][4] super-diagonal blocks (block (l-1, l))
    double* Hr;       // [nslots][it][4] sub-diagonal blocks (block (l+1, l))
    double* Xstop;    // [nslots][2]
    double* G3;       // [nslots][4] Gram of the new block {g11, g12, g22, -}
    // ---- finished slots of the last pair_step launch (the host re-seeds them)
    int* fin_count;   // [1]
    int* fin_slots;   // [nslots]
    // ---- results, indexed by candidate
    double* res_Xm;
    long long* res_iter;
    int* res_lucky;
};
constexpr int PAIR_IDLE = 0, PAIR_NEW = 1, PAIR_RUN = 2;

// zero the two columns of every PAIR_NEW slot in the blocks P and C.  grid = (row blocks, panels)
__global__ void __launch_bounds__(COL_THREADS)
pair_zero_kernel(double* __restrict__ P, double* __restrict__ C, int64_t n, const int* __restrict__ flag) {
    __shared__ int fl[LPT];
    const int q = blockIdx.y, sub = threadIdx.x % LPT;
    if (threadIdx.x < LPT) fl[threadIdx.x] = flag[q * LPT + threadIdx.x];
    __syncthreads();
    if (fl[sub] != PAIR_NEW) return;
    const int64_t po = (int64_t)q * n * PW;
    const int64_t r0 = (int64_t)blockIdx.x * COL_ROWS_PER_CTA;
    const int64_t r1 = min(n, r0 + COL_ROWS_PER_CTA);
    const double2 z = make_double2(0.0, 0.0);
    for (int64_t r = r0 + (threadIdx.x / LPT); r < r1; r += COL_THREADS / LPT) {
        const int64_t o = po + r * PW + sub * 2;
        *reinterpret_cast<double2*>(P + o) = z;
        *reinterpret_cast<double2*>(C + o) = z;
    }
}

// fixed-order CTA sum of NV values per thread (256 threads); totals valid in thread 0
template <int NV>
__device__ __forceinline__ void seed_reduce(double (&v)[NV], double* smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = v[i];
        for (int off = 16; off; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
        v[i] = x;
    }
    if (lane == 0)
        for (int i = 0; i < NV; ++i) smem[warp * NV + i] = v[i];
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 0; i < NV; ++i) {
            double s = 0.0;
            for (int w = 0; w < COL_WARPS; ++w) s += smem[w * NV + i];
            v[i] = s;
        }
}

// Step 1 of a freshly assigned slot, straight from the CSR rows of its end points (one CTA per new slot):
//   P(:, slot) = [e_i e_j],  C(:, slot) = W1 = A(:, [i j]) with rows i, j zeroed  (= A*U - U*(U'AU), the result of
//   CGS2 at lanczos_krylov.m:86-88 - the second pass finds exactly zero coefficients), G3 = W1'W1, hc = U'AU.
// The columns must have been zeroed (pair_zero_kernel).  Column indices of a stored row are ascending.
__global__ void __launch_bounds__(COL_THREADS)
pair_seed_kernel(CsrDevView A, PairState st, double* __restrict__ P, double* __restrict__ C, int64_t n,
                 const int* __restrict__ new_slots) {
    __shared__ double red[COL_WARPS * 6];
    const int h = new_slots[blockIdx.x];
    const int i = st.ei[h], j = st.ej[h];
    const int si = A.row_pos[i], sj = A.row_pos[j];
    const int i0 = A.row_ptr[si], i1 = A.row_ptr[si + 1];
    const int j0 = A.row_ptr[sj], j1 = A.row_ptr[sj + 1];
    const int c0 = 2 * h, c1 = 2 * h + 1;
    double* Cp = C + (int64_t)(c0 / PW) * n * PW;
    double* Pp = P + (int64_t)(c0 / PW) * n * PW;
    const int o0 = c0 % PW, o1 = c1 % PW;
    // acc: g11, g12, g22, a_ii, a_ij, a_jj
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int p = i0 + (int)threadIdx.x; p < i1; p += COL_THREADS) {
        const int r = A.col[p];
        const double v = A.val ? A.val[p] : A.uval;
        if (r == i) { acc[3] += v; continue; }
        if (r == j) { acc[4] += v; continue; }
        Cp[(int64_t)r * PW + o0] = v;
        acc[0] += v * v;
        // partner entry A(r, j): binary search in the stored row of j
        int lo = j0, hi = j1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (A.col[mid] < r) lo = mid + 1; else hi = mid;
        }
        if (lo < j1 && A.col[lo] == r) acc[1] += v * (A.val ? A.val[lo] : A.uval);
    }
    for (int p = j0 + (int)threadIdx.x; p < j1; p += COL_THREADS) {
        const int r = A.col[p];
        const double v = A.val ? A.val[p] : A.uval;
        if (r == j) { acc[5] += v; continue; }
        if (r == i) continue;
        Cp[(int64_t)r * PW + o1] = v;
        acc[2] += v * v;
    }
    seed_reduce<6>(acc, red);
    if (threadIdx.x == 0) {
        // pending edge edits (kr_matrix_set_edges): A = stored CSR + delta entries.  The rows of i and j are merged
        // here, serially (a handful of entries): W1 and its Gram follow the EFFECTIVE columns of A.
        if (A.dl_count > 0) {
            __threadfence_block();
            for (int side = 0; side < 2; ++side) {
                const int pos = side == 0 ? si : sj, oc = side == 0 ? o0 : o1;
                int lo = 0, hi = A.dl_count;                      // first entry of stored row `pos`
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (A.dl_pos[mid] < pos) lo = mid + 1; else hi = mid; }
                for (int e = lo; e < A.dl_count && A.dl_pos[e] == pos; ++e) {
                    const int r = A.dl_col[e];
                    const double d = A.dl_val[e];
                    if (r == i || r == j) {                       // entries of U'AU
                        if (side == 0 && r == i) acc[3] += d;
                        else if (side == 1 && r == j) acc[5] += d;
                        else if (side == 0) acc[4] += d;          // a_ij (the (j, i) twin carries the same delta)
                        continue;
                    }
                    double* ci = Cp + (int64_t)r * PW + o0;
                    double* cj = Cp + (int64_t)r * PW + o1;
                    const double oi = *ci, oj = *cj;
                    (side == 0 ? *ci : *cj) += d;
                    const double ni = *ci, nj = *cj;
                    acc[0] += ni * ni - oi * oi;
                    acc[1] += ni * nj - oi * oj;
                    acc[2] += nj * nj - oj * oj;
                    (void)oc;
                }
            }
        }
        Pp[(int64_t)i * PW + o0] = 1.0;
        Pp[(int64_t)j * PW + o1] = 1.0;
        st.G3[h * 4 + 0] = acc[0];
        st.G3[h * 4 + 1] = acc[1];
        st.G3[h * 4 + 2] = acc[2];
        st.G3[h * 4 + 3] = 0.0;
        st.hc[h * 4 + 0] = acc[3]; st.hc[h * 4 + 1] = acc[4];
        st.hc[h * 4 + 2] = acc[4]; st.hc[h * 4 + 3] = acc[5];
        for (int k = 0; k < 4; ++k) {
            st.hp[h * 4 + k] = 0.0;
            st.Tp[h * 4 + k] = (k == 0 || k == 3) ? 1.0 : 0.0;
            st.Tc[h * 4 + k] = (k == 0 || k == 3) ? 1.0 : 0.0;
        }
        st.Xstop[h * 2] = st.Xstop[h * 2 + 1] = 0.0;
        st.step[h] = 0;
    }
}

// after pass A: h = T' G T (first CGS pass), coefficients of pass B.  g = {P'Y, C'Y} raw Grams (row-major 2x2 each),
// cf = {Ma, Mp, Mc}
__device__ __forceinline__ void pair_coef1_math(const double* g, const double* Tp, const double* Tc, double* cf, double* hp_out,
                                                double* hc_out) {
    double tmp[4], hp[4], hc[4], Mp[4], Mc[4];
    mm2(g + 4, Tc, tmp);       // (C'Y) Tc
    mtm2(Tc, tmp, hc);         // Tc' (C'Y) Tc
    mm2(Tc, hc, Mc);
    mm2(g, Tc, tmp);
    mtm2(Tp, tmp, hp);
    mm2(Tp, hp, Mp);
    for (int i = 0; i < 4; ++i) {
        cf[i] = Tc[i];
        cf[4 + i] = Mp[i];
        cf[8 + i] = Mc[i];
        hp_out[i] = hp[i];
        hc_out[i] = hc[i];
    }
}
// after pass B: h1 = T' G (W already carries T), h += h1, coefficients of pass C.  g = {P'W, C'W}
__device__ __forceinline__ void pair_coef2_math(const double* g, const double* Tp, const double* Tc, double* cf, double* hp_acc,
                                                double* hc_acc) {
    double hp[4], hc[4], Mp[4], Mc[4];
    mtm2(Tc, g + 4, hc);
    mm2(Tc, hc, Mc);
    mtm2(Tp, g, hp);
    mm2(Tp, hp, Mp);
    cf[0] = 1.0; cf[1] = 0.0; cf[2] = 0.0; cf[3] = 1.0;
    for (int i = 0; i < 4; ++i) {
        cf[4 + i] = Mp[i];
        cf[8 + i] = Mc[i];
        hp_acc[i] += hp[i];
        hc_acc[i] += hc[i];
    }
}

__global__ void pair_coef1_kernel(PairState st, const double* __restrict__ G) {
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= st.nslots) return;
    double* cf = st.coef + (int64_t)h * 12;
    if (st.flag[h] != PAIR_RUN) {
        for (int i = 0; i < 12; ++i) cf[i] = 0.0;       // idle slot: its columns stay finite (zero)
        return;
    }
    pair_coef1_math(G + (int64_t)h * 8, st.Tp + h * 4, st.Tc + h * 4, cf, st.hp + h * 4, st.hc + h * 4);
}

__global__ void pair_coef2_kernel(PairState st, const double* __restrict__ G) {
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= st.nslots) return;
    if (st.flag[h] != PAIR_RUN) return;               // coefficients of an idle slot stay zero
    pair_coef2_math(G + (int64_t)h * 8, st.Tp + h * 4, st.Tc + h * 4, st.coef + (int64_t)h * 12, st.hp + h * 4, st.hc + h * 4);
}

// Thin QR of an n x 2 block from its Gram matrix {g11, g12, g22} (ONE thread).  w1 / w2 point at element (0, column)
// of the orthogonalised, un-normalised block with row stride ws: only the LAPACK completion of exactly-zero columns
// touches the data.  Out: R (row-major 2x2, the sub-diagonal block of H) and T with Q = W * T.  Exactly-zero columns
// follow LAPACK's dgeqr2 / dorg2r (tau = 0 -> the completion is a coordinate vector), functions/lanczos_krylov.m:90.
__device__ inline void pair_qr_from_gram(double g11, double g12, double g22, double* w1, double* w2, int64_t ws, int64_t n,
                                         double* R, double* T) {
    R[0] = R[1] = R[2] = R[3] = 0.0;
    T[0] = 1.0; T[1] = 0.0; T[2] = 0.0; T[3] = 1.0;
    if (g11 == 0.0) {
        // H1 = I, R11 = 0, q1 = e_0
        const double b0 = w2[0], b1 = n > 1 ? w2[ws] : 0.0;
        w1[0] = 1.0;
        R[1] = b0;
        const double tail = g22 - b0 * b0 - b1 * b1;
        if (!(tail > 0.0)) {
            R[3] = b1;                       // tau2 = 0: q2 = e_1
            w2[0] = 0.0;
            if (n > 1) w2[ws] = 1.0;
        } else {
            const double beta2 = -copysign(sqrt(g22 - b0 * b0), b1);
            R[3] = beta2;
            w2[0] = 0.0;                     // q2 = [0; w2(2:n)] / beta2
            T[3] = 1.0 / beta2;
        }
    } else if (g22 == 0.0 && g12 == 0.0) {
        const double a0 = w1[0], a1 = n > 1 ? w1[ws] : 0.0;
        const double tail = g11 - a0 * a0;
        if (!(tail > 0.0)) {
            R[0] = a0;                       // w1 = a0 e_0: tau1 = 0, q1 = e_0, q2 = e_1
            w1[0] = 1.0;
            if (n > 1) w2[ws] = 1.0;
        } else {
            const double beta = -copysign(sqrt(g11), a0);
            const double kappa = a1 / (beta * (a0 - beta));
            R[0] = beta;
            T[0] = 1.0 / beta;
            T[1] = kappa;                    // q2 = kappa*w1 + (e_1 - kappa*beta*e_0)
            w2[0] = -kappa * beta;
            if (n > 1) w2[ws] = 1.0;
        }
    } else {
        const double r11 = sqrt(g11);
        const double r12 = g12 / r11;
        const double d = g22 - r12 * r12;
        R[0] = r11;
        R[1] = r12;
        T[0] = 1.0 / r11;
        if (d > 1e-28 * g22) {
            const double r22 = sqrt(d);
            R[3] = r22;
            T[1] = -r12 / (r11 * r22);
            T[3] = 1.0 / r22;
        } else {                             // numerically dependent column: deflate it
            R[3] = 0.0;
            T[1] = 0.0;
            T[3] = 0.0;
        }
    }
}

// Xm of step j from the block tridiagonal H (diagonal Hd, super-diagonal Hs, sub-diagonal Hr; [step][4] row-major
// 2x2 blocks): Gm = H(1:2j, 1:2j) symmetrised, tGm = Gm + Cm, two Jacobi eigen-solves and the trace formula
// (functions/trace_fun_update.m:72-89).  All NT threads of the CTA call; work = 2*nn*(nn|1) + 2*nn doubles
// (shared or global), nn = 2j.
template <int NT>
__device__ double pair_projected_trace(const double* Hd, const double* Hs, const double* Hr, int j, double b_off, int fun,
                                       double* work, JacobiShared* sh) {
    const int nn = 2 * j, lda = nn | 1;
    double* G = work;
    double* tG = G + nn * lda;
    double* d1 = tG + nn * lda;
    double* d2 = d1 + nn;
    for (int e = threadIdx.x; e < nn * nn; e += NT) {
        int r = e % nn, c = e / nn;
        int br = r >> 1, bc = c >> 1, ir = r & 1, ic = c & 1;
        // H(r, c): block (br, bc); column block bc is step bc+1
        auto Hval = [&](int rr, int cc, int irr, int icc) -> double {
            if (rr == cc) return Hd[cc * 4 + irr * 2 + icc];
            if (rr == cc - 1) return Hs[cc * 4 + irr * 2 + icc];
            if (rr == cc + 1) return Hr[cc * 4 + irr * 2 + icc];
            return 0.0;
        };
        double v = 0.5 * (Hval(br, bc, ir, ic) + Hval(bc, br, ic, ir));
        G[r + c * lda] = v;
        // Cm = B in the leading 2x2 block (V1 = U, so V1'U = I): B = b_off * [0 1; 1 0]
        double cm = (r < 2 && c < 2 && r != c) ? b_off : 0.0;
        tG[r + c * lda] = v + cm;
    }
    __syncthreads();
    if (nn <= MS_MAX_N) {
        // LAPACK's route (tridiagonalise + tridiagonal eigenvalues): two warps reduce one matrix each, then all threads
        // bracket all eigenvalues of both by multisection on Sturm counts (smalldense.cuh)
        __shared__ double ms_work[2][6 * MS_MAX_N];
        __shared__ int ms_cnt[NT];
        const int warp = threadIdx.x >> 5;
        if (warp == 0) warp_tridiag(tG, nn, lda, ms_work[0], ms_work[0] + MS_MAX_N, ms_work[0] + 2 * MS_MAX_N, ms_work[0] + 3 * MS_MAX_N);
        else if (warp == 1) warp_tridiag(G, nn, lda, ms_work[1], ms_work[1] + MS_MAX_N, ms_work[1] + 2 * MS_MAX_N, ms_work[1] + 3 * MS_MAX_N);
        __syncthreads();
        sturm_multisect2<NT>(ms_work, nn, d1, d2, ms_cnt);
    } else {
        block_jacobi<NT>(tG, nn, lda, nullptr, 0, sh);
        block_sorted_diag<NT>(tG, nn, lda, d1);
        block_jacobi<NT>(G, nn, lda, nullptr, 0, sh);
        block_sorted_diag<NT>(G, nn, lda, d2);
    }
    return block_trace_formula<NT>(fun, d1, d2, nn, sh->red);
}

// One CTA per slot in state `mode` (PAIR_NEW: finish step 1 after the seed; PAIR_RUN: finish step step+1 after
// pass C).  G3[slot][4] = {g11, g12, g22, -}; W is the panel-major block holding the orthogonalised
// (un-normalised) new block.  gscratch (may be null): per-slot global work space used instead of shared memory
// when the projected matrices outgrow it (2j > ~110).
__global__ void __launch_bounds__(JAC_THREADS)
pair_step_kernel(PairState st, const double* __restrict__ G3, double* __restrict__ W, int64_t n, int mode,
                 double* __restrict__ gscratch, int64_t gscratch_stride) {
    extern __shared__ double dyn[];
    __shared__ JacobiShared sh;
    __shared__ double Tn[4];
    __shared__ int s_lucky;
    const int h = blockIdx.x;
    if (st.flag[h] != mode) return;
    const int it = st.it;
    const int j = st.step[h] + 1;
    double* Hd = st.Hd + ((int64_t)h * it) * 4;
    double* Hs = st.Hs + ((int64_t)h * it) * 4;
    double* Hr = st.Hr + ((int64_t)h * it) * 4;
    if (threadIdx.x == 0) {
        const int c0 = 2 * h, c1 = 2 * h + 1;
        double* w1 = W + (int64_t)(c0 / PW) * n * PW + (c0 % PW);    // element (r, c0) at w1[r*PW]
        double* w2 = W + (int64_t)(c1 / PW) * n * PW + (c1 % PW);
        double R[4], T[4];
        pair_qr_from_gram(G3[h * 4 + 0], G3[h * 4 + 1], G3[h * 4 + 2], w1, w2, PW, n, R, T);
        for (int i = 0; i < 4; ++i) {
            Tn[i] = T[i];
            Hd[(j - 1) * 4 + i] = st.hc[h * 4 + i];
            Hs[(j - 1) * 4 + i] = st.hp[h * 4 + i];
            Hr[(j - 1) * 4 + i] = R[i];
        }
        s_lucky = sqrt(R[0] * R[0] + R[1] * R[1] + R[2] * R[2] + R[3] * R[3]) < 1e-8;   // lanczos_krylov.m:91
    }
    __syncthreads();
    double* work = gscratch ? gscratch + (int64_t)h * gscratch_stride : dyn;
    const double Xm = pair_projected_trace<JAC_THREADS>(Hd, Hs, Hr, j, st.b_off, st.fun, work, &sh);
    if (threadIdx.x == 0) {
        bool done = false;
        double* Xs = st.Xstop + h * 2;
        if (j <= 2) {
            Xs[j - 1] = Xm;
        } else {
            const double err = fabs(Xm - Xs[0]);
            if (err < st.tol) done = true;
            else { Xs[0] = Xs[1]; Xs[1] = Xm; }
        }
        if (!done && s_lucky) done = true;
        if (j == it) done = true;
        const long long cand = st.cand[h];
        st.res_Xm[cand] = Xm;
        st.res_iter[cand] = j;
        st.res_lucky[cand] = s_lucky;
        st.step[h] = j;
        if (done) {
            st.flag[h] = PAIR_IDLE;
            st.fin_slots[atomicAdd(st.fin_count, 1)] = h;
        } else {
            st.flag[h] = PAIR_RUN;
        }
        // rotate transforms: previous <- current, current <- new
        for (int i = 0; i < 4; ++i) {
            st.Tp[h * 4 + i] = st.Tc[h * 4 + i];
            st.Tc[h * 4 + i] = Tn[i];
        }
    }
}

// panel_active[q] = any slot of panel q still iterating (lets the SpMM and the update passes skip whole
// panels; only matters once the queue has run dry)
__global__ void pair_panel_active_kernel(const int* __restrict__ flag, int nslots, int* __restrict__ panel_active) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q * LPT >= nslots) return;
    int any = 0;
    for (int i = 0; i < LPT; ++i) any |= (flag[q * LPT + i] == PAIR_RUN);
    panel_active[q] = any;
}

// Scores the candidates (i_q, j_q), q < np (1-based end points, i != j, n > 130) and writes Xm / iter / lucky
// in candidate order.  max_slots bounds the three n x (2*slots) work blocks.
inline void pairs_run(kr_ctx* ctx, const kr_matrix* M, const int64_t* Ei, const int64_t* Ej, int64_t np, int64_t max_slots,
                      double b_off, double tol, int it, int fun, double* Xm_out, int64_t* iter_out, int* lucky_out) {
    if (np <= 0) return;
    const CsrDev& A = M->dev;
    const int64_t n = A.n;
    const int nslots_req = (int)std::min<int64_t>(np, std::max<int64_t>(LPT, max_slots));
    PanelBuf B0(ctx, n, 2 * nslots_req), B1(ctx, n, 2 * nslots_req), B2(ctx, n, 2 * nslots_req);
    const int panels = B0.panels;
    const int ns = panels * LPT;                      // slots padded to whole panels
    B0.buf.zero();
    B1.buf.zero();
    B2.buf.zero();
    const int rb = col_row_blocks(n);
    const int nparts = std::max(rb, A.ntiles);
    DevBuf<double> partial(ctx, (size_t)nparts * ns * 8), Gsum(ctx, (size_t)ns * 8);
    DevBuf<double> dstate(ctx, (size_t)ns * (4 + 4 + 4 + 4 + 12 + 2 + 4) + (size_t)ns * it * 12);
    DevBuf<int> istate(ctx, (size_t)ns * 6 + 1), pact(ctx, panels);
    DevBuf<long long> cand(ctx, ns), res_iter(ctx, np);
    DevBuf<double> res_x(ctx, np);
    DevBuf<int> res_lucky(ctx, np);
    dstate.zero();
    istate.zero();
    PairState st;
    st.nslots = ns; st.it = it; st.fun = fun; st.tol = tol; st.b_off = b_off;
    double* d = dstate.p;
    st.Tp = d; d += ns * 4;
    st.Tc = d; d += ns * 4;
    st.hp = d; d += ns * 4;
    st.hc = d; d += ns * 4;
    st.coef = d; d += ns * 12;
    st.Xstop = d; d += ns * 2;
    st.G3 = d; d += ns * 4;
    st.Hd = d; d += (size_t)ns * it * 4;
    st.Hs = d; d += (size_t)ns * it * 4;
    st.Hr = d;
    st.ei = istate.p;
    st.ej = istate.p + ns;
    st.step = istate.p + 2 * ns;
    st.flag = istate.p + 3 * ns;
    st.fin_slots = istate.p + 4 * ns;
    int* new_slots_dev = istate.p + 5 * ns;
    st.fin_count = istate.p + 6 * ns;
    st.cand = cand.p;
    st.res_Xm = res_x.p;
    st.res_iter = res_iter.p;
    st.res_lucky = res_lucky.p;

    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(pair_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JAC_SMEM_LIMIT));

    // host mirror of the slot table
    std::vector<long long> h_cand(ns, -1);
    std::vector<int> h_ei(ns, 0), h_ej(ns, 0), h_flag(ns, PAIR_IDLE), h_step(ns, 0), h_new, h_fin(ns);
    int64_t next = 0;
    int running = 0;
    double* P = B0.p();
    double* C = B1.p();
    double* Y = B2.p();
    const int cb = (int)ceil_div(ns, 128);
    dim3 ugrid((unsigned)rb, (unsigned)panels);
    DevBuf<double> gscratch;                           // only when the projections outgrow shared memory
    auto step_smem = [&](int jmax, int64_t* stride) -> size_t {
        const int nn = 2 * jmax;
        const size_t need = (size_t)(2 * nn * (nn | 1) + 2 * nn) * sizeof(double);
        if (need <= JAC_SMEM_LIMIT) { *stride = 0; return need; }
        const int nn_it = 2 * it;
        *stride = (int64_t)2 * nn_it * (nn_it | 1) + 2 * nn_it;
        if (!gscratch.p) gscratch.reset(ctx, (size_t)ns * (size_t)*stride);
        return 0;
    };
    auto launch_step = [&](double* W, int mode, int jmax) {
        int64_t stride = 0;
        const size_t smem = step_smem(jmax, &stride);
        KR_LAUNCH(ctx, pair_step_kernel, ns, JAC_THREADS, smem, st, st.G3, W, n, mode, stride ? gscratch.p : (double*)nullptr, stride);
    };
    std::vector<int> free_slots(ns);
    for (int h = 0; h < ns; ++h) free_slots[h] = ns - 1 - h;     // pop from the back: slot 0 first
    for (;;) {
        // ---- (re-)seed idle slots from the queue
        h_new.clear();
        while (next < np && !free_slots.empty()) {
            const int h = free_slots.back();
            free_slots.pop_back();
            h_cand[h] = next;
            h_ei[h] = (int)(Ei[next] - 1);
            h_ej[h] = (int)(Ej[next] - 1);
            h_flag[h] = PAIR_NEW;
            h_step[h] = 0;
            h_new.push_back(h);
            ++next;
        }
        if (!h_new.empty()) {
            // the slot tables are small: ship them whole (flags of running slots are unchanged on both sides)
            KR_CUDA(cudaMemcpyAsync(st.cand, h_cand.data(), ns * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
            KR_CUDA(cudaMemcpyAsync(st.ei, h_ei.data(), ns * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
            KR_CUDA(cudaMemcpyAsync(st.ej, h_ej.data(), ns * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
            KR_CUDA(cudaMemcpyAsync(st.flag, h_flag.data(), ns * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
            KR_CUDA(cudaMemcpyAsync(new_slots_dev, h_new.data(), h_new.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
            ctx->counters[3] += (int64_t)ns * 20;
            KR_LAUNCH(ctx, pair_zero_kernel, ugrid, COL_THREADS, 0, P, C, n, st.flag);
            KR_LAUNCH(ctx, pair_seed_kernel, (int)h_new.size(), COL_THREADS, 0, A.view(), st, P, C, n, new_slots_dev);
            launch_step(C, PAIR_NEW, 1);
            for (int h : h_new) { h_flag[h] = PAIR_RUN; h_step[h] = 1; }
            running += (int)h_new.size();
            // a seeded slot can finish at step 1 (it == 1 or a lucky breakdown): collect before the dense step
            int nfin = 0;
            KR_CUDA(cudaMemcpyAsync(&nfin, st.fin_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            KR_CUDA(cudaStreamSynchronize(ctx->stream));
            if (nfin > 0) {
                KR_CUDA(cudaMemcpyAsync(h_fin.data(), st.fin_slots, nfin * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
                KR_CUDA(cudaMemsetAsync(st.fin_count, 0, sizeof(int), ctx->stream));
                KR_CUDA(cudaStreamSynchronize(ctx->stream));
                for (int k = 0; k < nfin; ++k) {
                    const int h = h_fin[k];
                    h_flag[h] = PAIR_IDLE; h_cand[h] = -1;
                    free_slots.push_back(h);
                }
                running -= nfin;
                if (next < np) continue;               // re-seed those right away
            }
        }
        if (running == 0) break;
        // ---- one dense block-Lanczos step for every running slot
        int jmax = 0;
        for (int h = 0; h < ns; ++h)
            if (h_flag[h] == PAIR_RUN) jmax = std::max(jmax, h_step[h] + 1);
        KR_LAUNCH(ctx, pair_panel_active_kernel, (int)ceil_div(panels, 128), 128, 0, st.flag, ns, pact.p);
        EpiGram2 epi;
        epi.Y = Y; epi.P = P; epi.C = C; epi.partial = partial.p; epi.ncand = ns;
        launch_spmm(ctx, A, C, panels, epi, nullptr, 2 * running, pact.p);
        sum_partials(ctx, partial.p, A.ntiles, ns * 8, Gsum.p);
        KR_LAUNCH(ctx, pair_coef1_kernel, cb, 128, 0, st, Gsum.p);
        KR_LAUNCH(ctx, pair_update_kernel<0>, ugrid, COL_THREADS, 0, Y, P, C, n, st.coef, ns, partial.p, pact.p);
        sum_partials(ctx, partial.p, rb, ns * 8, Gsum.p);
        KR_LAUNCH(ctx, pair_coef2_kernel, cb, 128, 0, st, Gsum.p);
        KR_LAUNCH(ctx, pair_update_kernel<1>, ugrid, COL_THREADS, 0, Y, P, C, n, st.coef, ns, partial.p, pact.p);
        sum_partials(ctx, partial.p, rb, ns * 4, st.G3);
        launch_step(Y, PAIR_RUN, jmax);
        // rotate blocks: previous <- current, current <- W
        double* oldP = P;
        P = C;
        C = Y;
        Y = oldP;
        for (int h = 0; h < ns; ++h)
            if (h_flag[h] == PAIR_RUN) h_step[h] += 1;
        int nfin = 0;
        KR_CUDA(cudaMemcpyAsync(&nfin, st.fin_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        if (nfin > 0) {
            KR_CUDA(cudaMemcpyAsync(h_fin.data(), st.fin_slots, nfin * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            KR_CUDA(cudaMemsetAsync(st.fin_count, 0, sizeof(int), ctx->stream));
            KR_CUDA(cudaStreamSynchronize(ctx->stream));
            std::sort(h_fin.begin(), h_fin.begin() + nfin);      // the device appends in completion order
            for (int k = nfin - 1; k >= 0; --k) {
                const int h = h_fin[k];
                h_flag[h] = PAIR_IDLE; h_cand[h] = -1;
                free_slots.push_back(h);
            }
            running -= nfin;
        }
    }
    std::vector<double> xm(np);
    std::vector<long long> itv(np);
    std::vector<int> lk(np);
    KR_CUDA(cudaMemcpyAsync(xm.data(), st.res_Xm, np * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(itv.data(), st.res_iter, np * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(lk.data(), st.res_lucky, np * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->counters[4] += np * 20;
    for (int64_t q = 0; q < np; ++q) {
        Xm_out[q] = xm[q];
        iter_out[q] = itv[q];
        lucky_out[q] = lk[q];
    }
}

}  // namespace kr
