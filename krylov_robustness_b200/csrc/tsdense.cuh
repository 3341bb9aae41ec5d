// tsdense.cuh - tall-skinny dense kernels of the general-width block Krylov step on PANEL-MAJOR blocks:
//   ts_gram     G = V' W          (CGS2 coefficients h = V'w, functions/lanczos_krylov.m:110-112,
//                                  functions/arnoldi_krylov.m:104,120-122; also W'W, Q'X of mc_trace.m:46-49)
//   ts_update   W -= V h          (functions/lanczos_krylov.m:111,113)
//   hqr         thin Householder QR of an n x bs block in place (qr(w,0), functions/lanczos_krylov.m:48,90):
//               LAPACK's dgeqr2 / dorg2r operation for operation (tau = 0 for an exactly zero column, so the
//               completed basis vector is a coordinate vector exactly as in the reference), one launch per
//               column with the trailing update fused with the next column's dot products.
// A "block" is a PanelBuf (spmm.cuh layout: panels of PW = 16 columns, each a contiguous row-major n x 16
// array); the SpMM reads and writes the same storage, so a block step never transposes anything.  Columns
// beyond the logical width of a block's last panel are kept at ZERO by every kernel.
//
// The two contractions run on the FP64 tensor cores (mma.sync.m8n8k4.f64 = SASS DMMA; tcgen05 has no fp64
// kind), operands staged through shared memory with cp.async double buffering, split-K over row chunks with
// partials in a fixed layout summed in a fixed order (bit-reproducible).
#pragma once
#include "dense.cuh"

namespace kr {

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

constexpr int TS_MAXP = 64;          // panels in one list (64 * 16 = 1024 columns)
struct PanelList {                   // panel q: n x PW row-major at p[q]
    const double* p[TS_MAXP];
    int count = 0;
    void add(const PanelBuf& b) {
        for (int q = 0; q < b.panels; ++q) {
            if (count >= TS_MAXP) fail(KR_ERR_UNSUPPORTED, "block Krylov basis wider than %d columns", TS_MAXP * PW);
            p[count++] = b.p() + (int64_t)q * b.n * PW;
        }
    }
};

// ------------------------------------------------------------------------------------ Gram
// partial[chunk][col-major (cp*16) x (bp*16)] += V(chunk rows)' W(chunk rows).
// grid = (chunks, ceil(cp/8), ceil(bp/4)); CTA tile 128 x 64 of G, 8 warps as 4 (m) x 2 (n), warp tile 32 x 32.
constexpr int TSG_VP = 8, TSG_WP = 4, TSG_ROWS = 32;
constexpr int TSG_VS = TSG_VP * PW + 4, TSG_WS = TSG_WP * PW + 4;          // padded shared-memory row strides (doubles)
constexpr size_t TSG_SMEM = (size_t)2 * TSG_ROWS * (TSG_VS + TSG_WS) * sizeof(double);

__global__ void __launch_bounds__(256)
ts_gram_kernel(PanelList V, PanelList W, int64_t n, int rows_per_cta, double* __restrict__ partial) {
    extern __shared__ __align__(16) double ts_smem[];
    double* Vs[2] = {ts_smem, ts_smem + TSG_ROWS * TSG_VS};
    double* Ws[2] = {ts_smem + 2 * TSG_ROWS * TSG_VS, ts_smem + 2 * TSG_ROWS * TSG_VS + TSG_ROWS * TSG_WS};
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kk = lane & 3, idx = lane >> 2;
    const int vp0 = blockIdx.y * TSG_VP, wp0 = blockIdx.z * TSG_WP;
    const int nvp = min(TSG_VP, V.count - vp0), nwp = min(TSG_WP, W.count - wp0);
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta, r1 = min(n, r0 + (int64_t)rows_per_cta);
    const int wm = warp >> 1, wn = warp & 1;          // warp tile: G rows [32 wm, +32), G cols [32 wn, +32)
    double acc[4][4][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

    auto stage = [&](int buf, int64_t row0) {
        // 16-byte chunks: V: 32 rows x nvp panels x 8; W: 32 rows x nwp panels x 8
        for (int c = threadIdx.x; c < TSG_ROWS * TSG_VP * 8; c += 256) {
            const int r = c / (TSG_VP * 8), q = (c / 8) % TSG_VP, e = c % 8;
            double* dst = Vs[buf] + r * TSG_VS + q * PW + e * 2;
            if (q < nvp && row0 + r < r1) cp_async16(dst, V.p[vp0 + q] + (row0 + r) * PW + e * 2);
            else { dst[0] = 0.0; dst[1] = 0.0; }
        }
        for (int c = threadIdx.x; c < TSG_ROWS * TSG_WP * 8; c += 256) {
            const int r = c / (TSG_WP * 8), q = (c / 8) % TSG_WP, e = c % 8;
            double* dst = Ws[buf] + r * TSG_WS + q * PW + e * 2;
            if (q < nwp && row0 + r < r1) cp_async16(dst, W.p[wp0 + q] + (row0 + r) * PW + e * 2);
            else { dst[0] = 0.0; dst[1] = 0.0; }
        }
        cp_async_commit();
    };
    const bool active_m = wm * 2 < nvp;               // warp-uniform: its 32 G rows hold real V columns
    const bool active_n = wn * 2 < nwp;
    int buf = 0;
    if (r0 < r1) stage(0, r0);
    for (int64_t row0 = r0; row0 < r1; row0 += TSG_ROWS) {
        if (row0 + TSG_ROWS < r1) { stage(buf ^ 1, row0 + TSG_ROWS); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
        if (active_m && active_n) {
            const double* vs = Vs[buf] + wm * 32 + idx;
            const double* ws = Ws[buf] + wn * 32 + idx;
#pragma unroll
            for (int k0 = 0; k0 < TSG_ROWS; k0 += 4) {
                double a[4], b[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    a[t] = vs[(k0 + kk) * TSG_VS + t * 8];
                    b[t] = ws[(k0 + kk) * TSG_WS + t * 8];
                }
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 4; ++nt) dmma884(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
            }
        }
        __syncthreads();
        buf ^= 1;
    }
    // C fragment: lane holds C[idx][2*kk], C[idx][2*kk+1] of each 8x8 tile
    const int ldg = V.count * PW;
    double* out = partial + (int64_t)blockIdx.x * ldg * (W.count * PW);
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            const int m = vp0 * PW + wm * 32 + mt * 8 + idx;
            const int c = wp0 * PW + wn * 32 + nt * 8 + 2 * kk;
            if (wm * 32 + mt * 8 < nvp * PW && wn * 32 + nt * 8 < nwp * PW) {
                out[m + (int64_t)c * ldg] = acc[mt][nt][0];
                out[m + (int64_t)(c + 1) * ldg] = acc[mt][nt][1];
            }
        }
}

inline int ts_rows_per_cta(kr_ctx* ctx, int64_t n) {
    // ~2 CTAs per SM worth of row chunks, whole slabs, at least 256 rows
    int64_t r = ceil_div(n, (int64_t)ctx->num_sms * 2);
    r = ceil_div(std::max<int64_t>(r, 256), TSG_ROWS) * TSG_ROWS;
    return (int)std::min<int64_t>(r, 4096);
}

// G (column-major (V.count*16) x (W.count*16), device) = V' W
inline void ts_gram(kr_ctx* ctx, const PanelList& V, const PanelList& W, int64_t n, double* G, DevBuf<double>& scratch) {
    if (V.count == 0 || W.count == 0) return;
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(ts_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TSG_SMEM));
    const int rows = ts_rows_per_cta(ctx, n);
    const int chunks = (int)std::max<int64_t>(1, ceil_div(n, rows));
    const size_t gsz = (size_t)V.count * PW * W.count * PW;
    if (scratch.count < (size_t)chunks * gsz) scratch.reset(ctx, (size_t)chunks * gsz);
    dim3 grid((unsigned)chunks, (unsigned)ceil_div(V.count, TSG_VP), (unsigned)ceil_div(W.count, TSG_WP));
    KR_LAUNCH(ctx, ts_gram_kernel, grid, 256, TSG_SMEM, V, W, n, rows, scratch.p);
    sum_partials(ctx, scratch.p, chunks, (int)gsz, G);
}

// ------------------------------------------------------------------------------------ update
// W -= V h   (h: column-major (V.count*16) x (W.count*16), device).  grid = (row chunks, ceil(bp/4)); the CTA
// walks the V panels in groups of 8: h group (128 x 64, negated) in shared memory, V slab 32 x 128 staged per
// group, the 32 x 64 tile of W lives in the DMMA accumulator fragments.
constexpr int TSU_HS = TSG_WP * PW + 4;
constexpr size_t TSU_SMEM = (size_t)(TSG_VP * PW * TSU_HS + TSG_ROWS * TSG_VS) * sizeof(double);

// OVERWRITE: W = V h instead (the right-multiplication of CholQR, V and W must be DIFFERENT blocks and V at most 128
// columns wide so that there is a single V group); `skip` (may be null): do nothing if *skip != 0.
template <bool OVERWRITE>
__global__ void __launch_bounds__(256)
ts_update_kernel(PanelList V, PanelList Wl, int64_t n, int rows_per_cta, const double* __restrict__ h,
                 const int* __restrict__ skip) {
    if (skip && *skip) return;
    extern __shared__ __align__(16) double ts_smem[];
    double* hs = ts_smem;                                   // [128][TSU_HS]: -h(group rows, this CTA's 64 columns)
    double* vs = ts_smem + TSG_VP * PW * TSU_HS;            // [32][TSG_VS]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kk = lane & 3, idx = lane >> 2;
    const int wp0 = blockIdx.y * TSG_WP;
    const int nwp = min(TSG_WP, Wl.count - wp0);
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta, r1 = min(n, r0 + (int64_t)rows_per_cta);
    const int ldh = V.count * PW;
    // warp tile of the 32 x 64 output slab: rows [8 (warp&3), +8), columns [32 (warp>>2), +32)
    const int mrow = (warp & 3) * 8, ncol = (warp >> 2) * 32;
    for (int vg = 0; vg < V.count; vg += TSG_VP) {
        const int nvp = min(TSG_VP, V.count - vg);
        __syncthreads();
        for (int e = threadIdx.x; e < TSG_VP * PW * TSG_WP * PW; e += 256) {
            const int k = e % (TSG_VP * PW), c = e / (TSG_VP * PW);
            double v = 0.0;
            if (k < nvp * PW && c < nwp * PW) v = (OVERWRITE ? 1.0 : -1.0) * h[(vg * PW + k) + (int64_t)(wp0 * PW + c) * ldh];
            hs[k * TSU_HS + c] = v;
        }
        for (int64_t row0 = r0; row0 < r1; row0 += TSG_ROWS) {
            __syncthreads();
            for (int c = threadIdx.x; c < TSG_ROWS * TSG_VP * 8; c += 256) {
                const int r = c / (TSG_VP * 8), q = (c / 8) % TSG_VP, e = c % 8;
                double* dst = vs + r * TSG_VS + q * PW + e * 2;
                if (q < nvp && row0 + r < r1) cp_async16(dst, V.p[vg + q] + (row0 + r) * PW + e * 2);
                else { dst[0] = 0.0; dst[1] = 0.0; }
            }
            cp_async_commit();
            // C fragments: W(row0 + mrow + idx, ncol + 8 t + 2 kk (+1))
            double c0[4], c1[4];
            const int64_t row = row0 + mrow + idx;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int col = ncol + t * 8 + 2 * kk;                 // column inside the CTA's 64
                c0[t] = c1[t] = 0.0;
                if (!OVERWRITE && row < r1 && col < nwp * PW) {
                    const double2 w = *reinterpret_cast<const double2*>(Wl.p[wp0 + col / PW] + row * PW + col % PW);
                    c0[t] = w.x; c1[t] = w.y;
                }
            }
            cp_async_wait<0>();
            __syncthreads();
            const double* va = vs + (mrow + idx) * TSG_VS + kk;
            const double* hb = hs + kk * TSU_HS + ncol + idx;
            for (int k0 = 0; k0 < nvp * PW; k0 += 4) {
                const double a = va[k0];
#pragma unroll
                for (int t = 0; t < 4; ++t) dmma884(c0[t], c1[t], a, hb[k0 * TSU_HS + t * 8]);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int col = ncol + t * 8 + 2 * kk;
                if (row < r1 && col < nwp * PW)
                    *reinterpret_cast<double2*>(const_cast<double*>(Wl.p[wp0 + col / PW]) + row * PW + col % PW) = make_double2(c0[t], c1[t]);
            }
        }
    }
}

inline void ts_update(kr_ctx* ctx, const PanelList& V, const PanelList& W, int64_t n, const double* h) {
    if (V.count == 0 || W.count == 0) return;
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(ts_update_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TSU_SMEM));
    const int rows = ts_rows_per_cta(ctx, n);
    dim3 grid((unsigned)std::max<int64_t>(1, ceil_div(n, rows)), (unsigned)ceil_div(W.count, TSG_WP));
    KR_LAUNCH(ctx, ts_update_kernel<false>, grid, 256, TSU_SMEM, V, W, n, rows, h, (const int*)nullptr);
}

// W = V m   (m: column-major (V.count*16) x (W.count*16), device); V and W distinct, V.count <= 8
inline void ts_rightmul(kr_ctx* ctx, const PanelList& V, const PanelList& W, int64_t n, const double* m, const int* skip) {
    if (V.count == 0 || W.count == 0) return;
    if (V.count > TSG_VP) fail(KR_ERR_UNSUPPORTED, "ts_rightmul: block wider than %d columns", TSG_VP * PW);
    static bool attr_set[64] = {};
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(ts_update_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TSU_SMEM));
    const int rows = ts_rows_per_cta(ctx, n);
    dim3 grid((unsigned)std::max<int64_t>(1, ceil_div(n, rows)), (unsigned)ceil_div(W.count, TSG_WP));
    KR_LAUNCH(ctx, ts_update_kernel<true>, grid, 256, TSU_SMEM, V, W, n, rows, m, skip);
}

// ------------------------------------------------------------------------------------ Householder QR
// State of one factorisation (device): R (bs x bs column-major, upper triangular), tau[bs], and per-pass
// partial dot products.  Pass k of the factor phase (k = 0 .. bs):
//   - finish reflector k-1 from the dots of the previous pass (every CTA recomputes the same scalars from the
//     partials in a fixed order), apply it to the trailing columns of the CTA's rows, store v in column k-1,
//   - accumulate, over the rows below the NEW diagonal row k, dots[j] = sum_r W(r,k) W(r,j), j = k .. bs-1.
// Pass k of the form-Q phase (dorg2r, k = bs-1 .. 0, plus one leading dots-only pass) works the same way with
// the reflectors read back from the strictly lower part of W.
constexpr int HQR_MAXB = 128;        // widest block of the default instantiation
constexpr int HQR_WIDEB = 256;       // widest block at all: the second instantiation, for the edge sets of the budget
                                     // scripts (Tests/test_unweighted_break_budget.m:89-90,119-120: up to 100 edges,
                                     // i.e. up to 200 selector columns); half the threads keep its shared memory static
constexpr int HQR_THREADS = 1024;    // 32 warps, one row per warp at a time: the passes are latency-bound (a row's
constexpr int HQR_ROWS = 128;        // reflector entry is a dependent load), so few rows per warp = 4; larger n: see HqrWork::prepare

struct HqrState {
    double* R;          // [bs*bs]
    double* tau;        // [bs]
    double* beta;       // [bs] diagonal of R
    double* partial;    // [2][nctas][MAXB] ping-pong (MAXB = HQR_MAXB or HQR_WIDEB, the kernels' template argument)
    double* pivot;      // [2][MAXB] row k of the trailing matrix (written by the CTA that owns row k)
};

// element (r, c) of a block given as a panel list
__device__ __forceinline__ double* hqr_at(const PanelList& W, int64_t r, int c) {
    return const_cast<double*>(W.p[c / PW]) + r * PW + (c % PW);
}

// Factor pass k (0 <= k <= bs).  Reflector k-1 is defined by: alpha = pivot value W(k-1,k-1) (pass k-1 saved the
// pivot row), xnorm^2 = dots[k-1], and for j >= k: d_j = dots[j] (over rows below k-1), W(k-1, j) = pivot[j].
template <int MAXB, int THREADS>
__global__ void __launch_bounds__(THREADS)
hqr_factor_pass_kernel(PanelList W, int64_t n, int bs, int k, HqrState st, int nctas, int rows_per_cta) {
    __shared__ double coef[MAXB];      // tau * s_j for the trailing columns of reflector k-1
    __shared__ double sdots[MAXB];
    __shared__ double wred[THREADS / 32][MAXB];
    __shared__ double s_scale, s_tau;
    const int tid = threadIdx.x;
    const int pp = k & 1;                                  // this pass writes partial/pivot set pp, reads pp^1
    const double* pin = st.partial + (size_t)(pp ^ 1) * nctas * MAXB;
    double* pout = st.partial + (size_t)pp * nctas * MAXB;
    const double* pivin = st.pivot + (pp ^ 1) * MAXB;
    double* pivout = st.pivot + pp * MAXB;
    if (k > 0) {
        // dots of pass k-1, summed in CTA order
        for (int j = tid; j < bs; j += THREADS) {
            double s = 0.0;
            if (j >= k - 1)
                for (int c = 0; c < nctas; ++c) s += pin[(size_t)c * MAXB + j];
            sdots[j] = s;
        }
        __syncthreads();
        if (tid == 0) {
            const double alpha = pivin[k - 1];
            const double xn2 = sdots[k - 1];
            double beta, tau, scale;
            if (xn2 == 0.0) {                              // dlarfg: H = I
                tau = 0.0; beta = alpha; scale = 0.0;
            } else {
                beta = -copysign(sqrt(alpha * alpha + xn2), alpha);
                tau = (beta - alpha) / beta;
                scale = 1.0 / (alpha - beta);
            }
            s_tau = tau; s_scale = scale;
            if (blockIdx.x == 0) {
                st.tau[k - 1] = tau;
                st.beta[k - 1] = beta;
                st.R[(k - 1) + (size_t)(k - 1) * bs] = beta;
            }
        }
        __syncthreads();
        const double tau = s_tau, scale = s_scale;
        for (int j = tid; j < bs; j += THREADS) {
            double cf = 0.0;
            if (j >= k) {
                const double sj = pivin[j] + scale * sdots[j];     // v' W(:, j), v(1) = 1
                cf = tau * sj;
                if (blockIdx.x == 0) st.R[(k - 1) + (size_t)j * bs] = pivin[j] - cf;   // row k-1 of R
            }
            coef[j] = cf;
        }
        __syncthreads();
    }
    // rows of this CTA
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta, r1 = min(n, r0 + (int64_t)rows_per_cta);
    const int warp = tid >> 5, lane = tid & 31;
    double acc[MAXB / 32];
#pragma unroll
    for (int t = 0; t < MAXB / 32; ++t) acc[t] = 0.0;
    const double scale = k > 0 ? s_scale : 0.0;
    for (int64_t r = r0 + warp; r < r1; r += THREADS / 32) {
        double v = 0.0;
        if (k > 0 && r > k - 1) {
            double* pv = hqr_at(W, r, k - 1);
            v = *pv * scale;                               // all lanes read the same address
            __syncwarp();
            if (lane == 0) *pv = v;                        // store the reflector (v(1) = 1 implicit)
        }
        if (r < k) continue;                               // rows above the new diagonal are finished
        double xk = 0.0;
        if (k < bs) {
            xk = *hqr_at(W, r, k);
            if (k > 0 && r > k - 1) xk -= coef[k] * v;
        }
#pragma unroll
        for (int t = 0; t < MAXB / 32; ++t) {
            const int j = lane + 32 * t;
            if (j >= k && j < bs) {
                double* pw = hqr_at(W, r, j);
                double w = *pw;
                if (k > 0 && r > k - 1) {                  // r >= k here, so always below row k-1
                    w -= coef[j] * v;
                    *pw = w;
                }
                if (r == k) pivout[j] = w;                 // the new pivot row
                else acc[t] += xk * w;                     // rows strictly below the diagonal
            }
        }
    }
    if (k >= bs) return;
    // CTA partial dots in warp order
#pragma unroll
    for (int t = 0; t < MAXB / 32; ++t) wred[warp][lane + 32 * t] = acc[t];
    __syncthreads();
    for (int j = tid; j < MAXB; j += THREADS) {
        double s = 0.0;
        for (int w = 0; w < THREADS / 32; ++w) s += wred[w][j];
        pout[(size_t)blockIdx.x * MAXB + j] = s;
    }
}

// Form-Q pass for reflector k (k = bs-1 .. 0), LAPACK dorg2r: on entry the columns k+1 .. bs-1 of W hold
// Q(:, k+1:) restricted to rows >= k+1 ... in place.  dots[j] = v_k' Q(k:, j) for j > k were accumulated by the
// previous pass (pass k+1, or the leading dots-only pass when k = bs-1 has none to apply to).
//   Q(k:, j) -= tau_k v_k dots[j]  (j > k);  Q(k,k) = 1 - tau_k;  Q(k+1:, k) = -tau_k v_k;  Q(0:k-1, k) = 0
// and the pass accumulates dots'[j] = v_{k-1}' Q(k-1:, j) for j >= k for the next one.
template <int MAXB, int THREADS>
__global__ void __launch_bounds__(THREADS)
hqr_formq_pass_kernel(PanelList W, int64_t n, int bs, int k, HqrState st, int nctas, int rows_per_cta) {
    __shared__ double coef[MAXB];
    __shared__ double wred[THREADS / 32][MAXB];
    const int tid = threadIdx.x;
    const int pp = k & 1;
    const double* pin = st.partial + (size_t)(pp ^ 1) * nctas * MAXB;
    double* pout = st.partial + (size_t)pp * nctas * MAXB;
    const double tau = st.tau[k];
    for (int j = tid; j < bs; j += THREADS) {
        double s = 0.0;
        if (j > k)
            for (int c = 0; c < nctas; ++c) s += pin[(size_t)c * MAXB + j];
        coef[j] = tau * s;
    }
    __syncthreads();
    const double tau_prev = k > 0 ? st.tau[k - 1] : 0.0;
    (void)tau_prev;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta, r1 = min(n, r0 + (int64_t)rows_per_cta);
    const int warp = tid >> 5, lane = tid & 31;
    double acc[MAXB / 32];
#pragma unroll
    for (int t = 0; t < MAXB / 32; ++t) acc[t] = 0.0;
    for (int64_t r = r0 + warp; r < r1; r += THREADS / 32) {
        // v_k(r): 0 above row k, 1 at row k, stored value below
        const double vk = r < k ? 0.0 : (r == k ? 1.0 : *hqr_at(W, r, k));
        // v_{k-1}(r) for the next pass' dots
        double vp = 0.0;
        if (k > 0) vp = r < k - 1 ? 0.0 : (r == k - 1 ? 1.0 : *hqr_at(W, r, k - 1));
        __syncwarp();
#pragma unroll
        for (int t = 0; t < MAXB / 32; ++t) {
            const int j = lane + 32 * t;
            if (j >= k && j < bs) {
                double* pq = hqr_at(W, r, j);
                double q;
                if (j == k) q = r < k ? 0.0 : (r == k ? 1.0 - tau : -tau * vk);
                else {
                    q = *pq;
                    if (r >= k) q -= coef[j] * vk;
                }
                *pq = q;
                acc[t] += vp * q;
            }
        }
    }
    if (k == 0) return;
#pragma unroll
    for (int t = 0; t < MAXB / 32; ++t) wred[warp][lane + 32 * t] = acc[t];
    __syncthreads();
    for (int j = tid; j < MAXB; j += THREADS) {
        double s = 0.0;
        for (int w = 0; w < THREADS / 32; ++w) s += wred[w][j];
        pout[(size_t)blockIdx.x * MAXB + j] = s;
    }
}

__global__ void hqr_clear_kernel(double* p, size_t count) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) p[i] = 0.0;
}

struct HqrWork {
    DevBuf<double> buf;
    HqrState st;
    int nctas = 0, bs = 0, rows_per_cta = HQR_ROWS, maxb = HQR_MAXB;
    void prepare(kr_ctx* ctx, int64_t n, int bs_) {
        bs = bs_;
        maxb = bs <= HQR_MAXB ? HQR_MAXB : HQR_WIDEB;
        // every CTA of a pass first sums the previous pass' per-CTA partial dots (nctas x bs loads): keep nctas at two
        // waves of resident CTAs instead of n / 128 (n = 200 k: 1 563 CTAs, 0.4 ms per pass, most of it that prologue)
        rows_per_cta = (int)std::max<int64_t>(HQR_ROWS, ceil_div(ceil_div(n, (int64_t)2 * ctx->num_sms), 32) * 32);
        nctas = (int)std::max<int64_t>(1, ceil_div(n, rows_per_cta));
        const size_t need = (size_t)bs * bs + 2 * (size_t)bs + 2 * (size_t)nctas * maxb + 2 * (size_t)maxb;
        if (buf.count < need) buf.reset(ctx, need);
        double* d = buf.p;
        st.R = d; d += (size_t)bs * bs;
        st.tau = d; d += bs;
        st.beta = d; d += bs;
        st.partial = d; d += 2 * (size_t)nctas * maxb;
        st.pivot = d;
    }
};

// W (n x bs, panel list, padded columns zero) <- Q of the thin Householder QR; work.st.R holds R afterwards.
template <int MAXB, int THREADS>
inline void hqr_thin_impl(kr_ctx* ctx, const PanelList& W, int64_t n, int bs, HqrWork& work) {
    KR_LAUNCH(ctx, hqr_clear_kernel, 8, 256, 0, work.buf.p, work.buf.count);
    for (int k = 0; k <= bs; ++k)
        KR_LAUNCH(ctx, (hqr_factor_pass_kernel<MAXB, THREADS>), work.nctas, THREADS, 0, W, n, bs, k, work.st, work.nctas, work.rows_per_cta);
    // dorg2r: a leading pass that only accumulates v_{bs-1}' Q(:, j) is unnecessary (no columns to the right of
    // bs-1), but the partial set read by pass bs-1 must be zero: pass k reads set (k&1)^1
    KR_LAUNCH(ctx, hqr_clear_kernel, 8, 256, 0, work.st.partial, 2 * (size_t)work.nctas * MAXB);
    for (int k = bs - 1; k >= 0; --k)
        KR_LAUNCH(ctx, (hqr_formq_pass_kernel<MAXB, THREADS>), work.nctas, THREADS, 0, W, n, bs, k, work.st, work.nctas, work.rows_per_cta);
}

inline void hqr_thin(kr_ctx* ctx, const PanelList& W, int64_t n, int bs, HqrWork& work) {
    if (bs > HQR_WIDEB) fail(KR_ERR_UNSUPPORTED, "thin QR: block width %d exceeds %d", bs, HQR_WIDEB);
    if (n < bs) fail(KR_ERR_UNSUPPORTED, "thin QR needs n >= block size");
    work.prepare(ctx, n, bs);
    if (work.maxb == HQR_MAXB) hqr_thin_impl<HQR_MAXB, HQR_THREADS>(ctx, W, n, bs, work);
    else hqr_thin_impl<HQR_WIDEB, HQR_THREADS / 2>(ctx, W, n, bs, work);
}

// ------------------------------------------------------------------------------------ CholQR2 + Householder signs
// The passes of hqr_thin above cost 2*bs + 1 launches per factorisation: on the reference's graphs (launch-bound)
// and on large ones (latency-bound row loops) they were 97 % of a block Krylov step (profiles/
// r02l_launches_arnoldi_bs64.csv).  For a block of full numerical rank the SAME factors come from two rounds of
// Cholesky QR (Gram on the tensor cores, bs x bs Cholesky in one CTA, right-multiplication on the tensor cores):
//   W = Q+ R+ with diag(R+) > 0 is unique, and LAPACK's Householder factors are Q = Q+ S, R = S R+ with the signs
//   s_k = -sgn(alpha_k) of dlarfg, which the elimination of "Reconstructing Householder vectors from tall-skinny
//   QR" (Ballard et al., 2014) recovers from the TOP bs x bs block of Q+ alone (checked against LAPACK on 300
//   random and badly scaled blocks: factors equal to 1e-12, all signs equal).
// A block whose Cholesky pivot falls below 1e-10 of its diagonal (condition number beyond ~1e5), an exactly zero
// column included, is left untouched and goes through hqr_thin: the reference's dgeqr2/dorg2r semantics for rank
// deficient blocks (tau = 0, coordinate-vector completion) are kept to the letter.
constexpr int CQ_THREADS = 256;
constexpr int CQ_MAXB = 80;          // three bs x (bs+1) matrices in shared memory: 155 KB at 80; wider blocks take hqr_thin

// pass 1: G -> R1 (to Rkeep), R1^{-1} (to Minv);  pass 2: G -> R2, signs from top(S) R2^{-1}, Minv = R2^{-1} D,
// Rout = D R2 R1.  All matrices column-major with leading dimension ld (>= bs; padding kept zero).  flag: set to 1
// on breakdown (never cleared here).  Single CTA; dynamic shared memory: 3 * bs * (bs + 1) doubles.
__global__ void __launch_bounds__(CQ_THREADS)
cholqr_factor_kernel(const double* __restrict__ G, int bs, int ld, int pass, double* __restrict__ Rkeep,
                     double* __restrict__ Minv, double* __restrict__ Rout, PanelList S, int* __restrict__ flag) {
    extern __shared__ double cq[];
    __shared__ double s_sign[HQR_MAXB];
    const int tid = threadIdx.x, ls = bs + 1;
    double* R = cq;                    // upper triangular factor
    double* Ri = R + bs * ls;          // its inverse
    double* T = Ri + bs * ls;          // scratch: top(S) * Ri, or R2 * R1
    if (*flag) return;
    for (int e = tid; e < bs * bs; e += CQ_THREADS) {
        const int i = e % bs, j = e / bs;
        R[i + j * ls] = i <= j ? G[i + (size_t)j * ld] : 0.0;
        Ri[i + j * ls] = 0.0;
    }
    __syncthreads();
    // right-looking Cholesky, upper: row k of R, then the trailing update
    for (int k = 0; k < bs; ++k) {
        const double gkk = G[k + (size_t)k * ld];
        const double d = R[k + k * ls];
        if (!(d > 1e-10 * gkk) || !(gkk > 0.0)) {      // uniform: every thread reads the same values
            if (tid == 0) *flag = 1;
            return;
        }
        const double rkk = sqrt(d);
        __syncthreads();
        for (int j = k + tid; j < bs; j += CQ_THREADS) R[k + j * ls] = j == k ? rkk : R[k + j * ls] / rkk;
        __syncthreads();
        for (int e = tid; e < (bs - k - 1) * (bs - k - 1); e += CQ_THREADS) {
            const int i = k + 1 + e % (bs - k - 1), j = k + 1 + e / (bs - k - 1);
            if (i <= j) R[i + j * ls] -= R[k + i * ls] * R[k + j * ls];
        }
        __syncthreads();
    }
    // inverse of the upper triangular R, column by column (thread per column, back substitution)
    for (int j = tid; j < bs; j += CQ_THREADS) {
        for (int i = j; i >= 0; --i) {
            double acc = i == j ? 1.0 : 0.0;
            for (int l = i + 1; l <= j; ++l) acc -= R[i + l * ls] * Ri[l + j * ls];
            Ri[i + j * ls] = acc / R[i + i * ls];
        }
    }
    __syncthreads();
    if (pass == 1) {
        for (int e = tid; e < bs * bs; e += CQ_THREADS) {
            const int i = e % bs, j = e / bs;
            Rkeep[i + (size_t)j * ld] = R[i + j * ls];
            Minv[i + (size_t)j * ld] = Ri[i + j * ls];
        }
        return;
    }
    // ---- pass 2: signs of LAPACK's Householder factors from the top block of Q+ = S * Ri
    for (int e = tid; e < bs * bs; e += CQ_THREADS) {
        const int i = e % bs, j = e / bs;          // T(i, j) = sum_l S(i, l) Ri(l, j), l <= j
        double acc = 0.0;
        for (int l = 0; l <= j; ++l) acc += S.p[l / PW][(int64_t)i * PW + l % PW] * Ri[l + j * ls];
        T[i + j * ls] = acc;
    }
    __syncthreads();
    for (int k = 0; k < bs; ++k) {
        if (tid == 0) {
            const double t = T[k + k * ls];
            const double sg = t >= 0.0 ? -1.0 : 1.0;   // s_k = -sgn(alpha_k), sgn(0) = +1 (copysign in dlarfg)
            s_sign[k] = sg;
            T[k + k * ls] = t - sg;
        }
        __syncthreads();
        const double piv = T[k + k * ls];              // |piv| >= 1
        for (int e = tid; e < (bs - k - 1) * (bs - k - 1); e += CQ_THREADS) {
            const int i = k + 1 + e % (bs - k - 1), j = k + 1 + e / (bs - k - 1);
            T[i + j * ls] -= (T[i + k * ls] / piv) * T[k + j * ls];
        }
        __syncthreads();
    }
    // Minv = Ri * D;  Rout = D * (R2 * R1)
    for (int e = tid; e < bs * bs; e += CQ_THREADS) {
        const int i = e % bs, j = e / bs;
        Minv[i + (size_t)j * ld] = Ri[i + j * ls] * s_sign[j];
        double acc = 0.0;
        if (i <= j)
            for (int l = i; l <= j; ++l) acc += R[i + l * ls] * Rkeep[l + (size_t)j * ld];
        T[i + j * ls] = acc * s_sign[i];
    }
    __syncthreads();
    for (int e = tid; e < bs * bs; e += CQ_THREADS) {
        const int i = e % bs, j = e / bs;
        Rout[i + (size_t)j * bs] = T[i + j * ls];      // HqrState::R is bs x bs, leading dimension bs
    }
}

struct ThinQrWork {
    HqrWork hqr;                       // the fall-back, and the owner of R (hqr.st.R: bs x bs column-major)
    DevBuf<double> G, R1, Minv, gscratch;
    DevBuf<int> flag;
    std::unique_ptr<PanelBuf> S;       // the intermediate block of the two-round scheme
    int64_t fallbacks = 0, calls = 0;
};

// W (n x bs block given as one PanelBuf) <- Q of qr(W, 0) with LAPACK's sign conventions; work.hqr.st.R <- R.
// Synchronises once (the breakdown flag decides between the two routes on the host).
inline void thin_qr(kr_ctx* ctx, PanelBuf& Wb, int bs, ThinQrWork& work) {
    const int64_t n = Wb.n;
    PanelList W;
    W.add(Wb);
    work.calls += 1;
    if (n < bs || bs > CQ_MAXB) {
        hqr_thin(ctx, W, n, bs, work.hqr);
        return;
    }
    work.hqr.prepare(ctx, n, bs);                      // bs <= CQ_MAXB here
    const int ld = Wb.panels * PW;
    const size_t msz = (size_t)ld * ld;
    if (work.G.count < msz) { work.G.reset(ctx, msz); work.R1.reset(ctx, msz); work.Minv.reset(ctx, msz); }
    if (!work.flag.p) work.flag.reset(ctx, 1);
    if (!work.S || work.S->n != n || work.S->cols != Wb.cols) work.S.reset(new PanelBuf(ctx, n, Wb.cols));
    PanelList S;
    S.add(*work.S);
    static bool attr_set[64] = {};
    const size_t smem = (size_t)3 * bs * (bs + 1) * sizeof(double);
    if (first_use_on_device(attr_set, ctx->device))
        KR_CUDA(cudaFuncSetAttribute(cholqr_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)((size_t)3 * CQ_MAXB * (CQ_MAXB + 1) * sizeof(double))));
    KR_CUDA(cudaMemsetAsync(work.flag.p, 0, sizeof(int), ctx->stream));
    KR_CUDA(cudaMemsetAsync(work.Minv.p, 0, msz * sizeof(double), ctx->stream));
    KR_CUDA(cudaMemsetAsync(work.R1.p, 0, msz * sizeof(double), ctx->stream));
    ts_gram(ctx, W, W, n, work.G.p, work.gscratch);
    KR_LAUNCH(ctx, cholqr_factor_kernel, 1, CQ_THREADS, smem, work.G.p, bs, ld, 1, work.R1.p, work.Minv.p, work.hqr.st.R, S, work.flag.p);
    ts_rightmul(ctx, W, S, n, work.Minv.p, work.flag.p);
    ts_gram(ctx, S, S, n, work.G.p, work.gscratch);
    KR_LAUNCH(ctx, cholqr_factor_kernel, 1, CQ_THREADS, smem, work.G.p, bs, ld, 2, work.R1.p, work.Minv.p, work.hqr.st.R, S, work.flag.p);
    ts_rightmul(ctx, S, W, n, work.Minv.p, work.flag.p);
    int bad = 0;
    KR_CUDA(cudaMemcpyAsync(&bad, work.flag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    if (bad) {                          // rank deficient or ill conditioned: W is untouched
        work.fallbacks += 1;
        hqr_thin(ctx, W, n, bs, work.hqr);
    }
}

}  // namespace kr
