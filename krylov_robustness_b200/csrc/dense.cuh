// dense.cuh - panel-major dense blocks: layout conversion, per-column fused updates/reductions,
// and the batched tridiagonal quadrature  e1' f(T) e1  used by the stochastic-Lanczos path.
//
// All reductions are two-stage (per-CTA partials in a fixed layout, then a fixed-order sum), never
// float atomics, so alpha/beta and every stopping decision are bit-reproducible (SURVEY.md 7.2.2).
#pragma once
#include <type_traits>
#include "spmm.cuh"

namespace kr {

struct PanelBuf {                  // owning panel-major block
    DevBuf<double> buf;
    int64_t n = 0;
    int cols = 0, panels = 0;
    PanelBuf() = default;
    PanelBuf(kr_ctx* ctx, int64_t n_, int cols_) { reset(ctx, n_, cols_); }
    void reset(kr_ctx* ctx, int64_t n_, int cols_) {
        n = n_;
        cols = cols_;
        panels = (cols_ + PW - 1) / PW;
        buf.reset(ctx, (size_t)n * panels * PW);
    }
    double* p() const { return buf.p; }
    int64_t elems() const { return n * panels * PW; }
};

// ------------------------------------------------------------------ layout conversion
// column-major (ld) -> panel-major.  grid = (ceil(n/64), panels), 256 threads.
__global__ void __launch_bounds__(256)
cm_to_panel_kernel(const double* __restrict__ src, int64_t ld, int64_t n, int cols,
                   double* __restrict__ dst) {
    __shared__ double t[PW][65];
    const int q = blockIdx.y;
    const int64_t r0 = (int64_t)blockIdx.x * 64;
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int c = e / 64, i = e % 64;
        int64_t r = r0 + i;
        int col = q * PW + c;
        t[c][i] = (r < n && col < cols) ? src[r + (int64_t)col * ld] : 0.0;
    }
    __syncthreads();
    double* d = dst + (int64_t)q * n * PW + r0 * PW;
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int i = e / PW, c = e % PW;
        if (r0 + i < n) d[e] = t[c][i];
    }
}

__global__ void __launch_bounds__(256)
panel_to_cm_kernel(const double* __restrict__ src, int64_t n, int cols, double* __restrict__ dst,
                   int64_t ld) {
    __shared__ double t[PW][65];
    const int q = blockIdx.y;
    const int64_t r0 = (int64_t)blockIdx.x * 64;
    const double* s = src + (int64_t)q * n * PW + r0 * PW;
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int i = e / PW, c = e % PW;
        t[c][i] = (r0 + i < n) ? s[e] : 0.0;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int c = e / 64, i = e % 64;
        int64_t r = r0 + i;
        int col = q * PW + c;
        if (r < n && col < cols) dst[r + (int64_t)col * ld] = t[c][i];
    }
}

// column-major int8 signs (+1 / -1, anything else is taken by its sign, 0 stays 0) -> int8 sign panel (the
// panel-major layout with one byte per entry, padded columns 0): Rademacher probes carry one bit per entry, so
// the host -> device copy of kr_slq_trace_sign moves 1/8 of the bytes of the fp64 entry point, and the SLQ pass
// reads the probes as signs (slq.cuh) without an fp64 copy.
__global__ void __launch_bounds__(256)
cm_i8_to_panel_kernel(const signed char* __restrict__ src, int64_t ld, int64_t n, int cols,
                      signed char* __restrict__ dst) {
    __shared__ signed char t[PW][64 + 4];
    const int q = blockIdx.y;
    const int64_t r0 = (int64_t)blockIdx.x * 64;
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int c = e / 64, i = e % 64;
        int64_t r = r0 + i;
        int col = q * PW + c;
        t[c][i] = (r < n && col < cols) ? src[r + (int64_t)col * ld] : (signed char)0;
    }
    __syncthreads();
    signed char* d = dst + (int64_t)q * n * PW + r0 * PW;
    for (int e = threadIdx.x; e < PW * 64; e += 256) {
        int i = e / PW, c = e % PW;
        const int v = t[c][i];
        if (r0 + i < n) d[e] = (signed char)(v > 0 ? 1 : (v < 0 ? -1 : 0));
    }
}
// n x cols column-major (ld) -> panel-major block of the same element type
inline void cm_to_panel(kr_ctx* ctx, const signed char* src_dev, int64_t ld, int64_t n, int cols, signed char* dst,
                        cudaStream_t stream) {
    const int panels = (cols + PW - 1) / PW;
    if (n == 0 || panels == 0) return;
    dim3 grid((unsigned)ceil_div(n, 64), (unsigned)panels);
    cm_i8_to_panel_kernel<<<grid, 256, 0, stream>>>(src_dev, ld, n, cols, dst);
    check_launch(ctx, "cm_i8_to_panel_kernel");
}
inline void cm_to_panel(kr_ctx* ctx, const double* src_dev, int64_t ld, int64_t n, int cols, double* dst,
                        cudaStream_t stream) {
    const int panels = (cols + PW - 1) / PW;
    if (n == 0 || panels == 0) return;
    dim3 grid((unsigned)ceil_div(n, 64), (unsigned)panels);
    cm_to_panel_kernel<<<grid, 256, 0, stream>>>(src_dev, ld, n, cols, dst);
    check_launch(ctx, "cm_to_panel_kernel");
}
inline void cm_to_panel(kr_ctx* ctx, const double* src_dev, int64_t ld, PanelBuf& dst) {
    cm_to_panel(ctx, src_dev, ld, dst.n, dst.cols, dst.p(), ctx->stream);
}
inline void panel_to_cm(kr_ctx* ctx, const PanelBuf& src, double* dst_dev, int64_t ld) {
    if (src.n == 0 || src.panels == 0) return;
    dim3 grid((unsigned)ceil_div(src.n, 64), (unsigned)src.panels);
    KR_LAUNCH(ctx, panel_to_cm_kernel, grid, 256, 0, src.p(), src.n, src.cols, dst_dev, ld);
}

// counter-based Rademacher stream: entry (i, j) = +-1 from splitmix64(seed ^ (j << 32 | i)).  sgn (may be null):
// the same entries as an int8 sign panel.
__host__ __device__ inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__global__ void rademacher_kernel(double* __restrict__ dst, signed char* __restrict__ sgn, int64_t n, int cols,
                                  int panels, uint64_t seed, int64_t col_offset) {
    const int64_t total = n * panels * PW;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (int64_t)gridDim.x * blockDim.x) {
        int64_t q = e / (n * PW), rem = e % (n * PW);
        int64_t i = rem / PW;
        int c = (int)(q * PW + rem % PW);
        double v = 0.0;
        if (c < cols) {
            uint64_t h = splitmix64(seed ^ (((uint64_t)(c + col_offset) << 32) | (uint64_t)i));
            v = (h >> 63) ? -1.0 : 1.0;
        }
        dst[e] = v;
        if (sgn) sgn[e] = (signed char)v;
    }
}

// ------------------------------------------------------------------ per-column reductions
constexpr int COL_THREADS = 256;
constexpr int COL_ROWS_PER_CTA = 2048;   // rows of one panel handled by one CTA

inline int col_row_blocks(int64_t n) { return (int)ceil_div(n, COL_ROWS_PER_CTA); }

// deterministic CTA reduction of NV values per (threadIdx.x % LPT) class -> lanes 0..LPT-1 of warp 0
template <int NV>
__device__ __forceinline__ void col_cta_reduce(double (&v)[NV], double* smem) {
    cta_reduce_by_sub<NV>(v, smem);      // 8 warps (COL_THREADS = 256)
}

// two adjacent entries of a panel-major block, fp64 or int8 signs
__device__ __forceinline__ double2 ld_pair(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ double2 ld_pair(const signed char* p) {
    const char2 s = *reinterpret_cast<const char2*>(p);
    return make_double2((double)(signed char)s.x, (double)(signed char)s.y);
}

// partial[rb][col] = sum over the CTA's rows of X(r,col)^2.  grid = (row_blocks, panels)
template <class XT>
__global__ void __launch_bounds__(COL_THREADS)
colnorm2_kernel(const XT* __restrict__ X, int64_t n, double* __restrict__ partial, int total_cols) {
    __shared__ double smem[COL_WARPS * LPT * 2];
    const int q = blockIdx.y, sub = threadIdx.x % LPT;
    const XT* Xp = X + (int64_t)q * n * PW;
    const int64_t r0 = (int64_t)blockIdx.x * COL_ROWS_PER_CTA;
    const int64_t r1 = min(n, r0 + COL_ROWS_PER_CTA);
    double acc[2] = {0.0, 0.0};
    for (int64_t r = r0 + (threadIdx.x / LPT); r < r1; r += COL_THREADS / LPT) {
        double2 x = ld_pair(Xp + r * PW + sub * 2);
        acc[0] += x.x * x.x;
        acc[1] += x.y * x.y;
    }
    col_cta_reduce<2>(acc, smem);
    if (threadIdx.x < LPT) {
        double* o = partial + (int64_t)blockIdx.x * total_cols + q * PW + threadIdx.x * 2;
        o[0] = acc[0];
        o[1] = acc[1];
    }
}

// W = c0[col]*Y + c1[col]*U1 + c2[col]*U0 (W may alias U0), partial[rb][col] = sum W^2.
// The Lanczos three-term recurrence with per-probe coefficients (SLQ path).  U1 and U0 are fp64 or int8 sign
// panels (T1, T0 = signed char: the probes of steps 0 and 1).  T0 = void: step 0, whose U0 is zero; the term is
// kept as c2 * 0.0 so that the rounding is that of the three-term form.  STORE = false: the last step, where only
// beta is needed.
template <class T1, class T0, bool STORE = true>
__global__ void __launch_bounds__(COL_THREADS)
combine3_norm_kernel(const double* __restrict__ Y, const T1* __restrict__ U1,
                     const T0* U0, double* W, int64_t n, const double* __restrict__ coef,
                     int total_cols, double* __restrict__ partial) {
    __shared__ double smem[COL_WARPS * LPT * 2];
    const int q = blockIdx.y, sub = threadIdx.x % LPT;
    const int64_t po = (int64_t)q * n * PW;
    const int col = q * PW + sub * 2;
    const double c0x = coef[col], c0y = coef[col + 1];
    const double c1x = coef[total_cols + col], c1y = coef[total_cols + col + 1];
    const double c2x = coef[2 * total_cols + col], c2y = coef[2 * total_cols + col + 1];
    const int64_t r0 = (int64_t)blockIdx.x * COL_ROWS_PER_CTA;
    const int64_t r1 = min(n, r0 + COL_ROWS_PER_CTA);
    double acc[2] = {0.0, 0.0};
    for (int64_t r = r0 + (threadIdx.x / LPT); r < r1; r += COL_THREADS / LPT) {
        const int64_t o = po + r * PW + sub * 2;
        double2 y = __ldcs(reinterpret_cast<const double2*>(Y + o));
        double2 u1 = ld_pair(U1 + o);
        double2 u0;
        if constexpr (std::is_void<T0>::value) u0 = make_double2(0.0, 0.0);
        else u0 = ld_pair(U0 + o);
        double2 w;
        w.x = c0x * y.x + c1x * u1.x + c2x * u0.x;
        w.y = c0y * y.y + c1y * u1.y + c2y * u0.y;
        if (STORE) *reinterpret_cast<double2*>(W + o) = w;
        acc[0] += w.x * w.x;
        acc[1] += w.y * w.y;
    }
    col_cta_reduce<2>(acc, smem);
    if (threadIdx.x < LPT) {
        double* o = partial + (int64_t)blockIdx.x * total_cols + q * PW + threadIdx.x * 2;
        o[0] = acc[0];
        o[1] = acc[1];
    }
}

// out[col] = sum_b partial[b][col] in a fixed order: 32 columns x 8 row-groups per CTA, every thread
// sums a strided slice, the 8 slices meet in shared memory in index order (deterministic).
__global__ void __launch_bounds__(256)
sum_partials_kernel(const double* __restrict__ partial, int nblocks, int total_cols,
                    double* __restrict__ out) {
    __shared__ double sm[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    double s = 0.0;
    if (c < total_cols)
        for (int b = ty; b < nblocks; b += 8) s += partial[(int64_t)b * total_cols + c];
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < total_cols) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += sm[k][tx];
        out[c] = t;
    }
}

inline void sum_partials(kr_ctx* ctx, const double* partial, int nblocks, int total_cols, double* out) {
    KR_LAUNCH(ctx, sum_partials_kernel, (int)ceil_div(total_cols, 32), 256, 0, partial, nblocks, total_cols, out);
}

// ------------------------------------------------------------------ SLQ scalar recurrences
// state per column: s1 (scale of U1: v_j = s1*U1), s0 (scale of U0), beta_prev, nrm2 (||z||^2)
struct SlqState {
    double* s1;
    double* s0;
    double* beta_prev;
    double* coef;      // [3][total_cols]
    double* alpha;     // [m][total_cols]
    double* beta;      // [m][total_cols]
};

// after the SpMM of step j: alpha_j = s1^2 * (U1 . A U1); coefficients of the three-term update
__global__ void slq_alpha_kernel(const double* __restrict__ sums, int total_cols, SlqState st, int j) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= total_cols) return;
    const double d = sums[c];
    const double s1 = st.s1[c];
    const double a = s1 * s1 * d;
    st.alpha[(int64_t)j * total_cols + c] = a;
    st.coef[c] = s1;
    st.coef[total_cols + c] = -a * s1;
    st.coef[2 * total_cols + c] = -st.beta_prev[c] * st.s0[c];
}

// after the update of step j: beta_j = ||w||; rotate scales
__global__ void slq_beta_kernel(const double* __restrict__ sums, int total_cols, SlqState st, int j) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= total_cols) return;
    const double d = sums[c];
    const double b = sqrt(d);
    st.beta[(int64_t)j * total_cols + c] = b;
    st.s0[c] = st.s1[c];
    st.s1[c] = (b > 0.0) ? 1.0 / b : 0.0;
    st.beta_prev[c] = b;
}

__global__ void slq_init_kernel(const double* __restrict__ sums, int total_cols, SlqState st,
                                double* __restrict__ nrm2) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= total_cols) return;
    const double d = sums[c];
    nrm2[c] = d;
    st.s1[c] = d > 0.0 ? 1.0 / sqrt(d) : 0.0;
    st.s0[c] = 0.0;
    st.beta_prev[c] = 0.0;
}

__device__ __forceinline__ double apply_fun(int fun, double x) {
    return fun == KR_FUN_EXP ? exp(x) : fun == KR_FUN_SINH ? sinh(x) : cosh(x);
}

// Batched tridiagonal quadrature: one thread per probe.  Implicit QL on T (d, e) carrying only the
// first row of the eigenvector matrix; val = nrm2 * sum_i z_i^2 f(lambda_i).
constexpr int SLQ_MAX_M = 128;
__global__ void slq_quadrature_kernel(const double* __restrict__ alpha, const double* __restrict__ beta,
                                      const double* __restrict__ nrm2, int m, int cols, int total_cols,
                                      int fun, double* __restrict__ vals) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    double d[SLQ_MAX_M], e[SLQ_MAX_M], z[SLQ_MAX_M];
    int n = m;
    for (int i = 0; i < m; ++i) {
        d[i] = alpha[(int64_t)i * total_cols + c];
        e[i] = beta[(int64_t)i * total_cols + c];
        z[i] = 0.0;
        if (n == m && !(e[i] > 0.0)) n = i + 1;   // breakdown: T is n x n
    }
    e[n - 1] = 0.0;
    z[0] = 1.0;
    for (int l = 0; l < n; ++l) {
        int iter = 0, mm;
        do {
            for (mm = l; mm < n - 1; ++mm) {
                double dd = fabs(d[mm]) + fabs(d[mm + 1]);
                if (fabs(e[mm]) <= 2.220446049250313e-16 * dd) break;
            }
            if (mm != l) {
                if (iter++ == 100) break;
                double g = (d[l + 1] - d[l]) / (2.0 * e[l]);
                double r = hypot(g, 1.0);
                g = d[mm] - d[l] + e[l] / (g + copysign(r, g));
                double s = 1.0, cc = 1.0, p = 0.0;
                int i;
                for (i = mm - 1; i >= l; --i) {
                    double f = s * e[i], b = cc * e[i];
                    r = hypot(f, g);
                    e[i + 1] = r;
                    if (r == 0.0) {
                        d[i + 1] -= p;
                        e[mm] = 0.0;
                        break;
                    }
                    s = f / r;
                    cc = g / r;
                    g = d[i + 1] - p;
                    r = (d[i] - g) * s + 2.0 * cc * b;
                    p = s * r;
                    d[i + 1] = g + p;
                    g = cc * r - b;
                    f = z[i + 1];
                    z[i + 1] = s * z[i] + cc * f;
                    z[i] = cc * z[i] - s * f;
                }
                if (r == 0.0 && i >= l) continue;
                d[l] -= p;
                e[l] = g;
                e[mm] = 0.0;
            }
        } while (mm != l);
    }
    // sum in ascending eigenvalue magnitude of the weights' contribution is unnecessary: all terms
    // are non-negative for exp/cosh; use a fixed index order.
    double acc = 0.0;
    for (int i = 0; i < n; ++i) acc += z[i] * z[i] * apply_fun(fun, d[i]);
    vals[c] = nrm2[c] * acc;
}

}  // namespace kr
