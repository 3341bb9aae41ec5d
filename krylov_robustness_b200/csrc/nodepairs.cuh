// nodepairs.cuh - a SCREEN for the greedy round of functions/krylov_miobi.m:76-124 when the candidate edges are
// dense in few nodes (config C5: the 10^5 candidates of find_top_missing_edges(...,'min') touch ~520 nodes).
//
// The reference scores every candidate (i, j) with its own block Lanczos process on U = [e_i e_j]
// (functions/trace_fun_update.m:60-125): per step j it needs the eigenvalues of Gm = V'AV and tGm = V'(A+UBU')V for
// an orthonormal basis V of the block Krylov space K_j(A, U) = K_j(A, e_i) + K_j(A, e_j).  Those eigenvalues do not
// depend on the basis, so the spaces can be SHARED: one single-vector Arnoldi run per distinct node x (all nodes
// advanced together by an n x d SpMM: entries.cuh::ArnoldiBatch) gives orthonormal Q_x = [q_x^0 .. q_x^L] with
// A Q_x^(s) = Q_x^(s+1) Hbar_x, and for a pair the Ritz values are the generalised eigenvalues of
//     K = Z'AZ,  M = Z'Z,   Z = [Q_i^(s) Q_j^(s)],
// built from Hbar_i, Hbar_j and the cross Grams S_ij = Q_i' Q_j - tall-skinny contractions over ALL node pairs at
// once (level-pair Grams V_a' V_b on the FP64 tensor cores, tsdense.cuh::ts_gram).  10^5 block Lanczos runs become
// 520 Lanczos runs + 15 DMMA Grams + 10^5 tiny eigenproblems.
//
// WHY IT IS ONLY A SCREEN.  Z is not orthonormal: eps-level rounding of the products and dot products is multiplied
// by cond(M) (40 - 200 for hub pairs, whose spaces all lean towards the dominant eigenvector), and the score is a
// difference ~1e-4 of the eigenvalue scale.  Against the oracle the screen reproduces the reference's values to
// 1e-9 .. 1e-8 relative with equal step counts - far inside the reference's own stopping tolerance (1e-6 e^||A||),
// outside the 1e-10 parity gate.  So kr_greedy_round uses it to DISCARD candidates: every candidate within a
// relative margin of 1e-6 of the approximate leader (100x the observed error), every ill-conditioned pair and every
// pair not converged within the shared steps is re-scored by the exact path (pairs.cuh), and the reference's
// first-wins selection runs on exact values.  The selected edge and its value are those of the exact round.
// The per-candidate flavour (WB = true, kr_greedy_round_w) reads B's off-diagonal value from bw[candidate].
#pragma once
#include "entries.cuh"
#include "pairs.cuh"
#include "tsdense.cuh"

namespace kr {

constexpr int NP_MAXL = 7;             // at most 7 shared steps (8 levels q^0 .. q^7)
constexpr int NP_THREADS = 64;
constexpr int NP_MAXNN = 2 * NP_MAXL;  // largest pair problem

struct NodePairArgs {
    // G[a*(NP_MAXL+1)+b] = V_a' V_b, column-major with leading dimension dpad.  Full mode: a <= b only, all dpad columns
    // (the transposed block serves a > b).  Restricted mode (jcol0 >= 0): every ordered (a, b), columns jcol0 .. dpad
    // only - the second end points of a rank's candidate shard are few, the first ones are not.
    const double* G[(NP_MAXL + 1) * (NP_MAXL + 1)];
    int jcol0;
    const double* Hc;                                 // ArnoldiBatch::Hc: [node][step][0..it1]
    int it1, dpad, L;                                 // L = shared steps available (levels 0..L)
    const int* ci;                                    // [np] node column of end point i
    const int* cj;
    int np, it, fun, s0;                              // s0: first step to evaluate (state is kept across calls)
    double tol, b_off, piv_min;
    double* Xstop;                                    // [np][2] lag-2 buffer
    double* approx;                                   // [np]
    int* steps;                                       // [np]
    int* status;                                      // [np] 0 running, 1 converged, 2 ill-conditioned -> exact path
};

// The per-candidate flavour's arguments (pairs.cuh: PairStateW)
struct NodePairArgsW : NodePairArgs {
    const double* bw;                                 // [np] off-diagonal value of B per candidate
};
template <bool WB> using NodePairArgsOf = std::conditional_t<WB, NodePairArgsW, NodePairArgs>;

// B's off-diagonal value of candidate c (read where it is used: the scalar flavour compiles as before the flavours)
template <bool WB>
__device__ __forceinline__ double node_pair_b(const NodePairArgsOf<WB>& a, int c) {
    if constexpr (WB) return a.bw[c];
    else return a.b_off;
}

// One CTA per candidate: steps s0 .. L of the pair recurrence in node coordinates.
template <bool WB>
__global__ void __launch_bounds__(NP_THREADS)
node_pair_kernel(NodePairArgsOf<WB> a) {
    __shared__ double S[(NP_MAXL + 1) * (NP_MAXL + 1)];          // S[p][q] = q_i^p . q_j^q
    __shared__ double Hi[(NP_MAXL + 1) * NP_MAXL], Hj[(NP_MAXL + 1) * NP_MAXL];   // Hbar (r, c) at [r * NP_MAXL + c]
    __shared__ double Mm[NP_MAXNN * NP_MAXNN], Lc[NP_MAXNN * NP_MAXNN];
    __shared__ double Kk[2][NP_MAXNN * (NP_MAXNN | 1)];          // [0] tK, [1] K; overwritten by L^-1 . L^-T
    __shared__ double Xw[2][NP_MAXNN * NP_MAXNN];
    __shared__ double d1[NP_MAXNN], d2[NP_MAXNN];
    __shared__ double ms_work[2][6 * MS_MAX_N];
    __shared__ int ms_cnt[NP_THREADS];
    __shared__ double red[8];
    __shared__ int s_state;
    __shared__ double s_piv;
    const int c = blockIdx.x, tid = threadIdx.x;
    if (a.status[c] != 0) return;
    const int ni = a.ci[c], nj = a.cj[c];
    const int L1 = a.L + 1, W = NP_MAXL + 1;
    for (int e = tid; e < L1 * L1; e += NP_THREADS) {
        const int p = e / L1, q = e % L1;
        if (a.jcol0 >= 0) S[p * W + q] = a.G[p * W + q][ni + (size_t)(nj - a.jcol0) * a.dpad];
        else S[p * W + q] = p <= q ? a.G[p * W + q][ni + (size_t)nj * a.dpad] : a.G[q * W + p][nj + (size_t)ni * a.dpad];
    }
    for (int e = tid; e < L1 * a.L; e += NP_THREADS) {
        const int r = e / a.L, col = e % a.L;                    // Hbar(r, col), nonzero for r <= col + 1
        const size_t oi = ((size_t)ni * a.it1 + col) * (a.it1 + 1) + r, oj = ((size_t)nj * a.it1 + col) * (a.it1 + 1) + r;
        Hi[r * NP_MAXL + col] = r <= col + 1 ? a.Hc[oi] : 0.0;
        Hj[r * NP_MAXL + col] = r <= col + 1 ? a.Hc[oj] : 0.0;
    }
    __syncthreads();
    for (int s = a.s0; s <= a.L; ++s) {
        const int nn = 2 * s, lda = nn | 1;
        // ---- M = [I S; S' I], K = Z'AZ (symmetrised), tK = K + b (u1 u2' + u2 u1')
        for (int e = tid; e < nn * nn; e += NP_THREADS) {
            const int p = e % nn, q = e / nn;
            const int bp = p >= s, bq = q >= s, pp = p - bp * s, qq = q - bq * s;
            double m, k;
            if (bp == bq) {
                m = p == q ? 1.0 : 0.0;
                const double* H = bp ? Hj : Hi;
                k = 0.5 * (H[pp * NP_MAXL + qq] + H[qq * NP_MAXL + pp]);
            } else {
                const int x = bp ? qq : pp, y = bp ? pp : qq;    // (x, y): row in the i block, column in the j block
                m = S[x * W + y];
                double k1 = 0.0, k2 = 0.0;                       // Q_i' (A Q_j) = S(:, 0:s+1) Hbar_j ; (A Q_i)' Q_j = Hbar_i' S
                for (int l = 0; l <= s; ++l) {
                    k1 += S[x * W + l] * Hj[l * NP_MAXL + y];
                    k2 += Hi[l * NP_MAXL + x] * S[l * W + y];
                }
                k = 0.5 * (k1 + k2);
            }
            // u1 = Z'e_i = [e_0 ; S(0, 0:s)'],  u2 = Z'e_j = [S(0:s, 0) ; e_0]
            const double u1p = bp ? S[0 * W + pp] : (pp == 0 ? 1.0 : 0.0), u2p = bp ? (pp == 0 ? 1.0 : 0.0) : S[pp * W + 0];
            const double u1q = bq ? S[0 * W + qq] : (qq == 0 ? 1.0 : 0.0), u2q = bq ? (qq == 0 ? 1.0 : 0.0) : S[qq * W + 0];
            Mm[p + q * nn] = m;
            Kk[1][p + q * lda] = k;
            Kk[0][p + q * lda] = k + node_pair_b<WB>(a, c) * (u1p * u2q + u2p * u1q);
        }
        __syncthreads();
        // ---- Cholesky M = Lc Lc' (serial: nn <= 14) with the smallest pivot as the conditioning signal
        if (tid == 0) {
            double pmin = 1.0;
            for (int k = 0; k < nn; ++k) {
                double dk = Mm[k + k * nn];
                for (int l = 0; l < k; ++l) dk -= Lc[k + l * nn] * Lc[k + l * nn];
                pmin = fmin(pmin, dk);
                const double lk = dk > 0.0 ? sqrt(dk) : 1.0;
                Lc[k + k * nn] = lk;
                for (int i = k + 1; i < nn; ++i) {
                    double v = Mm[i + k * nn];
                    for (int l = 0; l < k; ++l) v -= Lc[i + l * nn] * Lc[k + l * nn];
                    Lc[i + k * nn] = v / lk;
                }
            }
            s_piv = pmin;
        }
        __syncthreads();
        if (!(s_piv > a.piv_min)) {                              // the two node spaces (nearly) intersect: exact path
            if (tid == 0) a.status[c] = 2;
            return;
        }
        // ---- C = Lc^-1 X Lc^-T for X = tK, K: columns first (thread t: column t of matrix t / 32), then rows
        {
            const int mtx = tid >> 5, t = tid & 31;
            if (t < nn) {
                for (int i = 0; i < nn; ++i) {                   // solve Lc x = X(:, t)
                    double v = Kk[mtx][i + t * lda];
                    for (int l = 0; l < i; ++l) v -= Lc[i + l * nn] * Xw[mtx][l + t * nn];
                    Xw[mtx][i + t * nn] = v / Lc[i + i * nn];
                }
            }
            __syncthreads();
            if (t < nn) {
                for (int i = 0; i < nn; ++i) {                   // row t: solve Lc y = Xw(t, :)'
                    double v = Xw[mtx][t + i * nn];
                    for (int l = 0; l < i; ++l) v -= Lc[i + l * nn] * Kk[mtx][t + l * lda];
                    Kk[mtx][t + i * lda] = v / Lc[i + i * nn];
                }
            }
            __syncthreads();
            for (int e = tid; e < nn * nn; e += NP_THREADS) {    // symmetrise both
                const int p = e % nn, q = e / nn;
                if (p < q) {
                    for (int m2 = 0; m2 < 2; ++m2) {
                        const double v = 0.5 * (Kk[m2][p + q * lda] + Kk[m2][q + p * lda]);
                        Kk[m2][p + q * lda] = v;
                        Kk[m2][q + p * lda] = v;
                    }
                }
            }
            __syncthreads();
        }
        // ---- eigenvalues (ascending) and the trace formula of trace_fun_update.m:83-89
        {
            const int warp = tid >> 5;
            warp_tridiag(Kk[warp], nn, lda, ms_work[warp], ms_work[warp] + MS_MAX_N, ms_work[warp] + 2 * MS_MAX_N, ms_work[warp] + 3 * MS_MAX_N);
            __syncthreads();
            sturm_multisect2<NP_THREADS>(ms_work, nn, d1, d2, ms_cnt);
        }
        const double Xm = block_trace_formula<NP_THREADS>(a.fun, d1, d2, nn, red);
        if (tid == 0) {
            int state = 0;
            double* Xs = a.Xstop + (size_t)c * 2;
            if (s <= 2) {
                Xs[s - 1] = Xm;
            } else {
                if (fabs(Xm - Xs[0]) < a.tol) state = 1;         // trace_fun_update.m:104-118
                else { Xs[0] = Xs[1]; Xs[1] = Xm; }
            }
            if (s == a.it) state = 1;
            a.approx[c] = Xm;
            a.steps[c] = s;
            if (state) a.status[c] = state;
            s_state = state;
        }
        __syncthreads();
        if (s_state) return;
    }
}

// Grams against level 0 without a pass over n: level 0 holds the unit vectors e_{node}, so
//   G_0q(i, j) = V_q(node_i, j)   (transposed == 0)        G_p0(i, j) = V_p(node_j, i)   (transposed != 0)
// for the columns j = jcol0 .. dpad (5 of the 15 Grams of a 4-step screen).  grid = (dpad / 16, cols / 16), 256 threads.
__global__ void __launch_bounds__(256)
node_gram0_kernel(const double* __restrict__ Vx, int64_t n, const int64_t* __restrict__ nodes, int d, int dpad, int jcol0,
                  int transposed, double* __restrict__ G) {
    const int i = blockIdx.x * 16 + threadIdx.x / 16, jj = blockIdx.y * 16 + threadIdx.x % 16, j = jcol0 + jj;
    double v = 0.0;
    if (i < d && j < d) {
        const int row = transposed ? j : i, col = transposed ? i : j;
        v = Vx[(int64_t)(col / PW) * n * PW + (nodes[row] - 1) * PW + (col % PW)];
    }
    G[i + (size_t)jj * dpad] = v;
}

struct NodeScreenOut {
    std::vector<double> approx;
    std::vector<int> steps, status;    // status: 1 converged (approx usable), anything else -> exact path
    int distinct_nodes = 0, levels = 0;
    bool restricted = false;           // Grams restricted to the column window of the "j" end points
};

// can the screen be used at all for this candidate list?
inline bool node_screen_applicable(const kr_matrix* M, int64_t np, int64_t distinct, int64_t it) {
    const int64_t n = M->dev.n;
    if (n <= 130 || it < 3) return false;
    if (distinct > TS_MAXP * PW || np < 8 * distinct) return false;                 // dense in few nodes only
    const int64_t dpad = ceil_div(distinct, (int64_t)PW) * PW;
    return n * dpad * 8 * (NP_MAXL + 2) <= ((int64_t)96 << 30);                      // the shared bases must fit
}

// E: np pairs (1-based, i != j).  Fills approximate scores for the candidates the node bases could settle.  bw (device,
// [np], may be null): the off-diagonal value of B per candidate, replacing b_off.
inline NodeScreenOut node_screen_run(kr_ctx* ctx, const kr_matrix* M, const int64_t* Ei, const int64_t* Ej, int64_t np,
                                     double b_off, double tol, int it, int fun, const double* bw = nullptr) {
    NodeScreenOut out;
    const CsrDev& A = M->dev;
    const int64_t n = A.n;
    // Orientation: the side with fewer distinct end points becomes "j" (the score is symmetric in the end points);
    // node columns: nodes that only occur as "i" first, the "j" nodes last, so that the j side is a column window.
    std::vector<int64_t> si(Ei, Ei + np), sj(Ej, Ej + np);
    std::sort(si.begin(), si.end());
    si.erase(std::unique(si.begin(), si.end()), si.end());
    std::sort(sj.begin(), sj.end());
    sj.erase(std::unique(sj.begin(), sj.end()), sj.end());
    const bool swap_sides = si.size() < sj.size();
    if (swap_sides) std::swap(si, sj);
    std::vector<int64_t> nodes;                        // column order
    for (int64_t v : si)
        if (!std::binary_search(sj.begin(), sj.end(), v)) nodes.push_back(v);
    const int jstart = (int)nodes.size();
    nodes.insert(nodes.end(), sj.begin(), sj.end());
    const int d = (int)nodes.size();
    out.distinct_nodes = d;
    auto col_of = [&](int64_t v) -> int {
        auto jt = std::lower_bound(sj.begin(), sj.end(), v);
        if (jt != sj.end() && *jt == v) return jstart + (int)(jt - sj.begin());
        return (int)(std::lower_bound(nodes.begin(), nodes.begin() + jstart, v) - nodes.begin());
    };
    std::vector<int> ci((size_t)np), cj((size_t)np);
    for (int64_t q = 0; q < np; ++q) {
        ci[(size_t)q] = col_of(swap_sides ? Ej[q] : Ei[q]);
        cj[(size_t)q] = col_of(swap_sides ? Ei[q] : Ej[q]);
    }
    const int Lmax = std::min(it, NP_MAXL);
    ArnoldiBatch B(ctx, A, nodes, Lmax);
    const int dpad = B.tc;
    DevBuf<int> dci(ctx, (size_t)np), dcj(ctx, (size_t)np), dsteps(ctx, (size_t)np), dstatus(ctx, (size_t)np);
    DevBuf<double> dX(ctx, (size_t)np * 2), dapprox(ctx, (size_t)np), gscratch;
    dci.upload(ci.data(), (size_t)np);
    dcj.upload(cj.data(), (size_t)np);
    dsteps.zero(); dstatus.zero(); dX.zero(); dapprox.zero();
    std::vector<DevBuf<double>> G((size_t)(NP_MAXL + 1) * (NP_MAXL + 1));
    NodePairArgsW aw;
    NodePairArgs& a = aw;
    aw.bw = bw;
    for (auto& g : a.G) g = nullptr;
    a.Hc = B.Hc.p; a.it1 = B.it1; a.dpad = dpad;
    a.ci = dci.p; a.cj = dcj.p; a.np = (int)np; a.it = it; a.fun = fun;
    a.tol = tol; a.b_off = b_off; a.piv_min = 1e-3;
    a.Xstop = dX.p; a.approx = dapprox.p; a.steps = dsteps.p; a.status = dstatus.p;
    DevBuf<int64_t> dnodes(ctx, (size_t)d);
    dnodes.upload(nodes.data(), (size_t)d);
    // restricted mode pays (L+1)^2 Grams of dpad x jcols instead of (L+1)(L+2)/2 of dpad x dpad
    const int jpanel0 = jstart / PW, jcols = dpad - jpanel0 * PW;
    bool restricted = jcols * 20 <= dpad * 11;
    if (const char* e = getenv("KR_SCREEN_RESTRICT")) restricted = atoi(e) != 0;
    a.jcol0 = restricted ? jpanel0 * PW : -1;
    out.restricted = restricted;
    const int gcol0 = restricted ? jpanel0 * PW : 0, gcols = restricted ? jcols : dpad;
    auto gram = [&](int p, int q) {                               // G_pq = V_p' V_q(:, gcol0 ..)
        DevBuf<double>& g = G[(size_t)p * (NP_MAXL + 1) + q];
        g.reset(ctx, (size_t)dpad * gcols);
        a.G[p * (NP_MAXL + 1) + q] = g.p;
        if (p == 0 || q == 0) {                                   // rows of a level at the nodes: no contraction needed
            KR_LAUNCH(ctx, node_gram0_kernel, dim3((unsigned)(dpad / 16), (unsigned)(gcols / 16)), 256, 0,
                      B.V[(size_t)(p == 0 ? q : p)]->p(), n, dnodes.p, d, dpad, gcol0, p == 0 ? 0 : 1, g.p);
            return;
        }
        PanelList Vp, Vq;
        Vp.add(*B.V[(size_t)p]);
        const PanelBuf& bq = *B.V[(size_t)q];
        for (int pq = gcol0 / PW; pq < bq.panels; ++pq) Vq.p[Vq.count++] = bq.p() + (int64_t)pq * n * PW;
        ts_gram(ctx, Vp, Vq, n, g.p, gscratch);
    };
    gram(0, 0);
    int L = 0, evaluated = 0;
    // shared steps: 4 first (the usual count at the reference's tolerance), then one at a time while enough candidates
    // are still running to pay for another level
    while (L < Lmax) {
        const int target = L == 0 ? std::min(4, Lmax) : L + 1;
        for (; L < target; ++L) {
            B.step(L);
            for (int p = 0; p <= L + 1; ++p) gram(p, L + 1);
            if (restricted)
                for (int q = 0; q <= L; ++q) gram(L + 1, q);
        }
        a.L = L;
        a.s0 = evaluated + 1;
        if (bw) KR_LAUNCH(ctx, node_pair_kernel<true>, (int)np, NP_THREADS, 0, aw);
        else KR_LAUNCH(ctx, node_pair_kernel<false>, (int)np, NP_THREADS, 0, a);
        evaluated = L;
        out.status = dstatus.to_host();
        int64_t running = 0;
        for (int v : out.status) running += (v == 0);
        if (running * 20 < np) break;                            // < 5 % left: the exact path takes them
    }
    out.levels = L + 1;
    out.status = dstatus.to_host();
    out.steps = dsteps.to_host();
    out.approx = dapprox.to_host();
    return out;
}

}  // namespace kr
