// blockkrylov.cuh - general-width block Lanczos / Arnoldi (functions/lanczos_krylov.m,
// functions/arnoldi_krylov.m) and the evaluators built on them with one wide block:
// trace_fun_update (rk > 2), fun_update, fun_and_grad_krylov_*, normest.
//
// Everything runs in hand-written kernels on PANEL-MAJOR blocks (the SpMM's own layout, no transposes):
//   one add_inf_pole step = SpMM -> Gram V'W (DMMA) -> W -= V h -> Gram -> W -= V h1 -> Householder QR
//   (dgeqr2/dorg2r semantics, tsdense.cuh) [-> Arnoldi's third pass], with h, h1, R written straight into the
//   device-resident block storage of H.  The projected matrices Gm / tGm are assembled on the device, f(Gm) is a
//   GEMM-based scaling-and-squaring Taylor evaluation (smallgemm.cuh), the stopping quantities are reduced on
//   the device; per Krylov step the host reads back a handful of scalars (one synchronisation).
// No cuBLAS / cuSOLVER anywhere (round 1 used dgemm / geqrf / orgqr / syevd here).
#pragma once
#include <memory>

#include "dense.cuh"
#include "smalldense.cuh"
#include "smallgemm.cuh"
#include "vecops.cuh"

namespace kr {

struct HostMat {                     // small column-major host matrix
    int64_t rows = 0, cols = 0;
    std::vector<double> a;
    HostMat() = default;
    HostMat(int64_t r, int64_t c) : rows(r), cols(c), a((size_t)(r * c), 0.0) {}
    double& operator()(int64_t i, int64_t j) { return a[(size_t)(i + j * rows)]; }
    double operator()(int64_t i, int64_t j) const { return a[(size_t)(i + j * rows)]; }
};

// host column-major (ld) -> panel-major device block (synchronises: the caller's buffer may go away)
inline void upload_cm_block(kr_ctx* ctx, const double* host, int64_t ld, PanelBuf& dst) {
    const int64_t n = dst.n;
    const int k = dst.cols;
    if (ld < n) fail(KR_ERR_ARG, "leading dimension smaller than the number of rows");
    DevBuf<double> stage(ctx, (size_t)std::max<int64_t>(n * k, 1));
    if (n > 0 && k > 0) {
        KR_CUDA(cudaMemcpy2DAsync(stage.p, n * sizeof(double), host, ld * sizeof(double), n * sizeof(double), k,
                                  cudaMemcpyHostToDevice, ctx->stream));
        ctx->counters[3] += n * k * (int64_t)sizeof(double);
    }
    cm_to_panel(ctx, stage.p, n, dst);
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
}
// panel-major device block -> host column-major, columns [0, cols)
inline void download_cm_block(kr_ctx* ctx, const PanelBuf& src, double* host, int64_t ld, int cols = -1) {
    const int64_t n = src.n;
    const int k = cols < 0 ? src.cols : std::min(cols, src.cols);
    if (ld < n) fail(KR_ERR_ARG, "leading dimension smaller than the number of rows");
    DevBuf<double> stage(ctx, (size_t)std::max<int64_t>(n * src.cols, 1));
    panel_to_cm(ctx, src, stage.p, n);
    if (n > 0 && k > 0) {
        KR_CUDA(cudaMemcpy2DAsync(host, ld * sizeof(double), stage.p, n * sizeof(double), n * sizeof(double), k,
                                  cudaMemcpyDeviceToHost, ctx->stream));
        ctx->counters[4] += n * k * (int64_t)sizeof(double);
    }
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
}

inline bool is_symmetric(const HostMat& B) {
    for (int64_t i = 0; i < B.rows; ++i)
        for (int64_t j = 0; j < i; ++j)
            if (B(i, j) != B(j, i)) return false;
    return B.rows == B.cols;
}

// ------------------------------------------------------------------------------------ small device kernels
__global__ void add_inplace_kernel(double* __restrict__ a, const double* __restrict__ b, int64_t total) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) a[e] += b[e];
}

// R (bs x bs, unpadded) -> padded bpad x bpad block (upper triangle; the rest zero) and the lucky-breakdown test:
// Lanczos ||R||_F < 1e-8 (lanczos_krylov.m:74,91); Arnoldi ||R||_2 < 1e-12 (arnoldi_krylov.m:79,100), decided by the
// Frobenius norm where it can be (||R||_F / sqrt(bs) <= ||R||_2 <= ||R||_F) and by a power iteration on R'R otherwise.
__global__ void __launch_bounds__(256)
hsub_lucky_kernel(const double* __restrict__ R, int bs, int bpad, double* __restrict__ Rp, int arnoldi, int* __restrict__ lucky) {
    __shared__ double red[256];
    __shared__ double x[HQR_WIDEB], y[HQR_WIDEB];
    double s = 0.0;
    for (int e = threadIdx.x; e < bpad * bpad; e += 256) {
        const int i = e % bpad, j = e / bpad;
        double v = 0.0;
        if (i < bs && j < bs && i <= j) v = R[i + (size_t)j * bs];
        Rp[e] = v;
        s += v * v;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
        __syncthreads();
    }
    const double fro = sqrt(red[0]);
    int lk;
    if (!arnoldi) lk = fro < 1e-8;
    else if (bs == 1) lk = fabs(R[0]) < 1e-12;
    else if (fro / sqrt((double)bs) >= 1e-12) lk = 0;
    else if (fro < 1e-12) lk = 1;
    else {
        // ||R||_2 by power iteration on R'R (bs <= HQR_WIDEB; a rare path, right at a breakdown)
        for (int i = threadIdx.x; i < bs; i += 256) x[i] = 1.0;
        __syncthreads();
        double lam = 0.0;
        for (int itn = 0; itn < 200; ++itn) {
            for (int i = threadIdx.x; i < bs; i += 256) {          // y = R x
                double t = 0.0;
                for (int j = i; j < bs; ++j) t += R[i + (size_t)j * bs] * x[j];
                y[i] = t;
            }
            __syncthreads();
            for (int j = threadIdx.x; j < bs; j += 256) {          // x = R' y
                double t = 0.0;
                for (int i = 0; i <= j; ++i) t += R[i + (size_t)j * bs] * y[i];
                x[j] = t;
            }
            __syncthreads();
            double nn2 = 0.0;
            for (int j = 0; j < bs; ++j) nn2 += x[j] * x[j];       // every thread the same serial sum
            const double nrm = sqrt(nn2);
            lam = nrm;
            __syncthreads();
            if (nrm == 0.0) break;
            for (int j = threadIdx.x; j < bs; j += 256) x[j] /= nrm;
            __syncthreads();
        }
        lk = sqrt(lam) < 1e-12;
    }
    if (threadIdx.x == 0) *lucky = lk;
}

// Assemble [tGm; Gm] (two nn x nn column-major matrices, tGm first) from the device-resident blocks of H:
//   Gm = sym(H(1:nn, 1:nn)),  tGm = Gm + CmS (rk x rk, leading block)   (trace_fun_update.m:72-81, fun_update.m:93-104)
struct HBlocks {
    const double* const* hcol;   // [steps] (rows_s * bpad) x bpad
    const double* const* hsub;   // [steps] bpad x bpad
    int arnoldi, bs, bpad;
};
__device__ __forceinline__ double hblock_at(const HBlocks& H, int a, int b) {
    const int lb = b / H.bs, ib = b % H.bs, la = a / H.bs, ia = a % H.bs;
    if (la == lb + 1) return H.hsub[lb][ia + (size_t)ib * H.bpad];
    if (la > lb) return 0.0;
    int local, rows;
    if (H.arnoldi) { local = la; rows = lb + 1; }
    else {
        const int first = lb > 0 ? lb - 1 : 0;
        if (la < first) return 0.0;
        local = la - first;
        rows = lb > 0 ? 2 : 1;
    }
    return H.hcol[lb][(size_t)(local * H.bpad + ia) + (size_t)ib * rows * H.bpad];
}
__global__ void assemble_proj_kernel(HBlocks H, int nn, const double* __restrict__ CmS, int rk, double* __restrict__ out) {
    const int64_t total = (int64_t)nn * nn;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int a = (int)(e % nn), b = (int)(e / nn);
        const double g = 0.5 * (hblock_at(H, a, b) + hblock_at(H, b, a));
        const double cm = (a < rk && b < rk) ? CmS[a + (size_t)b * rk] : 0.0;
        out[e] = g + cm;
        out[total + e] = g;
    }
}

// D = sym(X - pad(Xold)) (nn x nn; Xold is no x no in the leading corner), partial[b] = sum of squares
__global__ void __launch_bounds__(256)
diff_sym_kernel(const double* __restrict__ X, int nn, const double* __restrict__ Xold, int no, double* __restrict__ D,
                double* __restrict__ partial) {
    __shared__ double red[256];
    const int64_t total = (int64_t)nn * nn;
    double s = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
        const int a = (int)(e % nn), b = (int)(e / nn);
        double v = 0.5 * (X[a + (size_t)b * nn] + X[b + (size_t)a * nn]);
        if (a < no && b < no) v -= 0.5 * (Xold[a + (size_t)b * no] + Xold[b + (size_t)a * no]);
        D[e] = v;
        s += v * v;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}
// info[0] = ||D||_F, need = Frobenius norm does not decide ||D||_2 < tol
__global__ void stop_band_kernel(const double* __restrict__ partial, int count, int nn, double tol, double* __restrict__ info,
                                 int* __restrict__ need) {
    double s = 0.0;
    for (int i = 0; i < count; ++i) s += partial[i];
    const double fro = sqrt(s);
    info[0] = fro;
    info[1] = -1.0;
    *need = (fro >= tol) && (fro / sqrt((double)nn) < tol);
}

// rows of the basis at the given nodes: Ra (k x dim, column-major) with Ra(a, blk*bs + c) = Um_blk(node_a, c)
struct BlockPtrs { const double* p[TS_MAXP]; };      // one pointer per BLOCK (panel 0 of the block)
__global__ void gather_basis_rows_kernel(BlockPtrs B, int nblocks, int bs, int64_t n, const int64_t* __restrict__ nodes, int k,
                                         int dim, double* __restrict__ Ra) {
    const int64_t total = (int64_t)k * dim;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int a = (int)(e % k), col = (int)(e / k);
        const int blk = col / bs, c = col % bs;
        double v = 0.0;
        if (blk < nblocks) v = B.p[blk][(int64_t)(c / PW) * n * PW + (nodes[a] - 1) * PW + (c % PW)];
        Ra[e] = v;
    }
}
// s[q] = sum_b T(i1[q], b) * Ra(i2[q], b)      (one warp per q)
__global__ void bilinear_rows_kernel(const double* __restrict__ T, const double* __restrict__ Ra, int k, int dim,
                                     const int* __restrict__ i1, const int* __restrict__ i2, int nq, double* __restrict__ s) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;
    double acc = 0.0;
    for (int b = lane; b < dim; b += 32) acc += T[i1[q] + (size_t)b * k] * Ra[i2[q] + (size_t)b * k];
    for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) s[q] = acc;
}
// out[q] = X(i1[q], i2[q]) of an n x n column-major matrix
__global__ void gather_entries_kernel(const double* __restrict__ X, int64_t n, const int64_t* __restrict__ i1,
                                      const int64_t* __restrict__ i2, int nq, double* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq) out[q] = X[(i1[q] - 1) + (i2[q] - 1) * n];
}

}  // namespace kr

// ------------------------------------------------------------------------------------------------
// params + V + H (+K) of the reference, device-resident behind a handle
struct kr_krylov {
    kr_ctx* ctx = nullptr;
    const kr_matrix* A = nullptr;
    bool arnoldi = false;
    int64_t n = 0, bs = 0, steps = 0;
    int bp = 0, bpad = 0;                                   // panels per block, padded block width
    std::vector<std::unique_ptr<kr::PanelBuf>> V;           // Lanczos: the last <= 2 blocks; Arnoldi: all blocks
    std::vector<kr::DevBuf<double>> hcol, hsub;             // per step: CGS2 coefficients vs the retained blocks; R
    std::vector<int> hrows;                                 // blocks in hcol[s]
    kr::DevBuf<int> lucky_dev;
    kr::DevBuf<const double*> hcol_ptr, hsub_ptr;           // device copies of the block pointers (grown as needed)
    std::vector<const double*> hcol_host, hsub_host;        // their host staging (must outlive the async copies)
    kr::ThinQrWork qr;
    kr::DevBuf<double> scratch, h1;
    bool lucky = false;                                     // valid after sync_lucky()
    int64_t vcols() const { return (int64_t)V.size() * bs; }
    kr::HBlocks hblocks() const {
        kr::HBlocks H;
        H.hcol = hcol_ptr.p; H.hsub = hsub_ptr.p; H.arnoldi = arnoldi; H.bs = (int)bs; H.bpad = bpad;
        return H;
    }
};

namespace kr {

inline PanelList list_of(const std::vector<std::unique_ptr<PanelBuf>>& V) {
    PanelList l;
    for (auto& b : V) l.add(*b);
    return l;
}
inline PanelList list_of(const PanelBuf& b) {
    PanelList l;
    l.add(b);
    return l;
}

inline void krylov_publish_pointers(kr_krylov* st) {
    kr_ctx* ctx = st->ctx;
    const size_t s = st->hcol.size();
    if (st->hcol_ptr.count < s) {
        const size_t cap = std::max<size_t>(16, 2 * s);
        st->hcol_ptr.reset(ctx, cap);
        st->hsub_ptr.reset(ctx, cap);
    }
    std::vector<const double*>& a = st->hcol_host;
    std::vector<const double*>& b = st->hsub_host;
    a.reserve(256);                                   // no reallocation while earlier copies may be in flight
    b.reserve(256);
    if (s > a.capacity()) KR_CUDA(cudaStreamSynchronize(ctx->stream));
    a.resize(s);
    b.resize(s);
    for (size_t i = 0; i < s; ++i) { a[i] = st->hcol[i].p; b[i] = st->hsub[i].p; }
    KR_CUDA(cudaMemcpyAsync(st->hcol_ptr.p, a.data(), s * sizeof(double*), cudaMemcpyHostToDevice, ctx->stream));
    KR_CUDA(cudaMemcpyAsync(st->hsub_ptr.p, b.data(), s * sizeof(double*), cudaMemcpyHostToDevice, ctx->stream));
}

// one add_inf_pole step (lanczos_krylov.m:73-101 / arnoldi_krylov.m:78-111); the continuation
// block params.last is always the last block of V.  Enqueues only; lucky is read back by sync_lucky().
inline void krylov_step(kr_krylov* st) {
    kr_ctx* ctx = st->ctx;
    const int64_t n = st->n;
    const int bs = (int)st->bs, bpad = st->bpad;
    std::unique_ptr<PanelBuf> W(new PanelBuf(ctx, n, bs));
    const PanelBuf& last = *st->V.back();
    EpiPlain epi{W->p(), last.p(), 1.0, 0.0};
    launch_spmm(ctx, st->A->dev, last.p(), last.panels, epi, nullptr, bs);
    const PanelList Vl = list_of(st->V), Wl = list_of(*W);
    const int cblocks = (int)st->V.size();
    const size_t hsz = (size_t)cblocks * bpad * bpad;
    st->hcol.emplace_back(ctx, hsz);
    st->hsub.emplace_back(ctx, (size_t)bpad * bpad);
    st->hrows.push_back(cblocks);
    double* h = st->hcol.back().p;
    if (st->h1.count < hsz) st->h1.reset(ctx, hsz);
    const int eg = ew_grid(ctx, (int64_t)hsz);
    // CGS2 against the retained blocks (lanczos_krylov.m:109-115, arnoldi_krylov.m:119-125)
    ts_gram(ctx, Vl, Wl, n, h, st->scratch);
    ts_update(ctx, Vl, Wl, n, h);
    ts_gram(ctx, Vl, Wl, n, st->h1.p, st->scratch);
    ts_update(ctx, Vl, Wl, n, st->h1.p);
    KR_LAUNCH(ctx, add_inplace_kernel, eg, 256, 0, h, st->h1.p, (int64_t)hsz);
    // [w, R] = qr(w, 0)
    thin_qr(ctx, *W, bs, st->qr);
    if (!st->lucky_dev.p) st->lucky_dev.reset(ctx, 1);
    KR_LAUNCH(ctx, hsub_lucky_kernel, 1, 256, 0, st->qr.hqr.st.R, bs, bpad, st->hsub.back().p, (int)st->arnoldi, st->lucky_dev.p);
    if (st->arnoldi) {
        // third reorthogonalisation (arnoldi_krylov.m:104-106): hh = V'w; w -= V hh; H(1:end-bs, last) += hh R
        ts_gram(ctx, Vl, Wl, n, st->h1.p, st->scratch);
        ts_update(ctx, Vl, Wl, n, st->h1.p);
        const int cpad = cblocks * bpad;
        sgemm(ctx, cpad, bpad, bpad, 1.0, st->h1.p, cpad, 0, st->hsub.back().p, bpad, 0, 1.0, h, cpad, 0, 1);
        st->V.push_back(std::move(W));
    } else {
        st->V.push_back(std::move(W));
        if (st->V.size() > 2) st->V.erase(st->V.begin());                     // lanczos_krylov.m:94-99
    }
    st->steps += 1;
    krylov_publish_pointers(st);
}

inline void sync_lucky(kr_krylov* st) {
    int lk = 0;
    KR_CUDA(cudaMemcpyAsync(&lk, st->lucky_dev.p, sizeof(int), cudaMemcpyDeviceToHost, st->ctx->stream));
    KR_CUDA(cudaStreamSynchronize(st->ctx->stream));
    st->lucky = lk != 0;
}

// start: V1 = qr(b, 0), one step    (lanczos_krylov.m:30-58, arnoldi_krylov.m:32-62); b is consumed
inline std::unique_ptr<kr_krylov> krylov_start(kr_ctx* ctx, const kr_matrix* A, bool arnoldi, int64_t bs,
                                               std::unique_ptr<PanelBuf> b) {
    const int64_t n = A->dev.n;
    if (b->n != n) fail(KR_ERR_ARG, "The block vector b has wrong number of rows");
    if (bs < 1) fail(KR_ERR_ARG, "empty starting block");
    if (bs > HQR_WIDEB) fail(KR_ERR_UNSUPPORTED, "block width %lld exceeds %d", (long long)bs, HQR_WIDEB);
    std::unique_ptr<kr_krylov> st(new kr_krylov());
    st->ctx = ctx; st->A = A; st->arnoldi = arnoldi; st->n = n; st->bs = bs;
    st->bp = b->panels;
    st->bpad = b->panels * PW;
    thin_qr(ctx, *b, (int)bs, st->qr);
    st->V.push_back(std::move(b));
    krylov_step(st.get());
    return st;
}

// dense symmetric copy of A for the small-n branches (host assembly)
inline HostMat dense_of(const kr_matrix* M) {
    const CsrHost& H = M->host;
    HostMat D(H.n, H.n);
    for (int64_t i = 0; i < H.n; ++i)
        for (int64_t p = H.row_ptr[i]; p < H.row_ptr[i + 1]; ++p) D(i, H.col[p]) += H.val[p];
    return D;
}
// fAt = sym(fA + U B U')
inline HostMat dense_updated(const HostMat& fA, int64_t rk, const double* U, int64_t ldu, const HostMat& B, bool symmetrise) {
    const int64_t n = fA.rows;
    HostMat fAt = fA;
    std::vector<double> UB((size_t)n * rk, 0.0);
    for (int64_t a = 0; a < n; ++a)
        for (int64_t q = 0; q < rk; ++q) {
            double s = 0;
            for (int64_t p = 0; p < rk; ++p) s += U[a + p * ldu] * B(p, q);
            UB[(size_t)(a + q * n)] = s;
        }
    for (int64_t b = 0; b < n; ++b)
        for (int64_t q = 0; q < rk; ++q) {
            const double u = U[b + q * ldu];
            if (u == 0.0) continue;
            for (int64_t a = 0; a < n; ++a) fAt(a, b) += UB[(size_t)(a + q * n)] * u;
        }
    if (symmetrise) {
        HostMat S(n, n);
        for (int64_t i = 0; i < n; ++i)
            for (int64_t j = 0; j < n; ++j) S(i, j) = 0.5 * (fAt(i, j) + fAt(j, i));
        return S;
    }
    return fAt;
}
inline double host_norm1(const HostMat& S) {
    double m = 0;
    for (int64_t j = 0; j < S.cols; ++j) {
        double s = 0;
        for (int64_t i = 0; i < S.rows; ++i) s += std::abs(S(i, j));
        m = std::max(m, s);
    }
    return m;
}

// Shared front end of trace_fun_update / fun_update: U on the device, Krylov start, CmS = sym((V1'U) B (V1'U)')
struct WideSetup {
    std::unique_ptr<kr_krylov> st;
    DevBuf<double> CmS;            // rk x rk
    double norm_bound = 0;         // >= ||tGm||_2, ||Gm||_2
};
inline WideSetup wide_setup(kr_ctx* ctx, const kr_matrix* M, int64_t rk, const double* U, int64_t ldu, const HostMat& B,
                            bool arnoldi) {
    const int64_t n = M->dev.n;
    WideSetup ws;
    PanelBuf Ud(ctx, n, (int)rk);
    upload_cm_block(ctx, U, ldu, Ud);
    std::unique_ptr<PanelBuf> b0(new PanelBuf(ctx, n, (int)rk));
    KR_CUDA(cudaMemcpyAsync(b0->p(), Ud.p(), (size_t)Ud.elems() * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    ws.st = krylov_start(ctx, M, arnoldi, rk, std::move(b0));
    kr_krylov* st = ws.st.get();
    // Cm = (V1' U) B (V1' U)'   (trace_fun_update.m:65-66): V1 is the first retained block right after the start
    const int bpad = st->bpad;
    DevBuf<double> dC(ctx, (size_t)bpad * bpad);
    ts_gram(ctx, list_of(*st->V.front()), list_of(Ud), n, dC.p, st->scratch);
    std::vector<double> c = dC.to_host();            // one synchronisation per call
    HostMat T(rk, rk), Cm(rk, rk);
    for (int64_t i = 0; i < rk; ++i)
        for (int64_t j = 0; j < rk; ++j) {
            double s = 0;
            for (int64_t k = 0; k < rk; ++k) s += c[(size_t)(i + k * bpad)] * B(k, j);
            T(i, j) = s;
        }
    for (int64_t i = 0; i < rk; ++i)
        for (int64_t j = 0; j < rk; ++j) {
            double s = 0;
            for (int64_t k = 0; k < rk; ++k) s += T(i, k) * c[(size_t)(j + k * bpad)];
            Cm(i, j) = s;
        }
    std::vector<double> cs((size_t)rk * rk);
    double fro = 0;
    for (int64_t i = 0; i < rk; ++i)
        for (int64_t j = 0; j < rk; ++j) {
            const double v = 0.5 * (Cm(i, j) + Cm(j, i));
            cs[(size_t)(i + j * rk)] = v;
            fro += v * v;
        }
    ws.CmS.reset(ctx, (size_t)rk * rk);
    ws.CmS.upload(cs.data(), cs.size());
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    ws.norm_bound = M->norm1 + std::sqrt(fro);        // ||Gm||_2 <= ||A||_2 <= ||A||_1 (A symmetric)
    return ws;
}

struct TfuResult { double Xm = 0; int64_t iter = 0; int lucky = 0; };

// trace_fun_update with one wide block (any rk)      (trace_fun_update.m:21-130)
inline TfuResult trace_fun_update_general(kr_ctx* ctx, const kr_matrix* M, int64_t rk, const double* U, int64_t ldu,
                                          const HostMat& B, double tol, int64_t it, int fun) {
    const int64_t n = M->dev.n;
    TfuResult out;
    if (!is_symmetric(B)) fail(KR_ERR_UNSUPPORTED, "trace_fun_update: the device path needs a symmetric (Hermitian) B");
    ExpmWork ew;
    DevBuf<double> xm(ctx, 1);
    // A block as wide as the space (rk >= n: U = selector of every node, the literal "all edges" call of config C2):
    // V = qr(U) spans everything, W = AV - V(V'AV) is zero, the reference stops at j = 1 on a lucky breakdown with
    // Gm = V'AV, i.e. with the dense quantity below (trace_fun_update.m:62-87,119-124).
    const bool whole_space = rk >= n && n > 130;
    if (n <= 130 || whole_space) {                            // :37-51 dense branch
        if (whole_space) { out.iter = 1; out.lucky = 1; }
        const HostMat fA = dense_of(M);
        const HostMat S = dense_updated(fA, rk, U, ldu, B, true);
        std::vector<double> both((size_t)2 * n * n);
        std::copy(S.a.begin(), S.a.end(), both.begin());
        for (int64_t i = 0; i < n; ++i)
            for (int64_t j = 0; j < n; ++j) both[(size_t)(n * n + i + j * n)] = 0.5 * (fA(i, j) + fA(j, i));
        DevBuf<double> dS(ctx, both.size()), dF(ctx, both.size());
        dS.upload(both.data(), both.size());
        symfun_batched(ctx, dS.p, (int)n, 2, fun, std::max(host_norm1(S), host_norm1(fA)), dF.p, ew);
        KR_LAUNCH(ctx, trace_diff_kernel, 1, 256, 0, dF.p, dF.p + n * n, (int)n, xm.p);
        xm.download(&out.Xm, 1);
        return out;
    }
    WideSetup ws = wide_setup(ctx, M, rk, U, ldu, B, false);
    kr_krylov* st = ws.st.get();
    double Xstop[2] = {0, 0};
    int64_t j = 0;
    DevBuf<double> SG, F;
    for (j = 1; j <= it; ++j) {
        if (j > 1) krylov_step(st);
        const int nn = (int)(j * rk);
        const size_t sz = (size_t)2 * nn * nn;
        if (SG.count < sz) { SG.reset(ctx, sz); F.reset(ctx, sz); }
        KR_LAUNCH(ctx, assemble_proj_kernel, ew_grid(ctx, (int64_t)nn * nn), 256, 0, st->hblocks(), nn, ws.CmS.p, (int)rk, SG.p);
        for (int attempt = 0; attempt < 2; ++attempt) {
            ew.begin(ctx, attempt == 1);
            symfun_batched(ctx, SG.p, nn, 2, fun, ws.norm_bound, F.p, ew);
            KR_LAUNCH(ctx, trace_diff_kernel, 1, 256, 0, F.p, F.p + (size_t)nn * nn, nn, xm.p);
            KR_CUDA(cudaMemcpyAsync(&out.Xm, xm.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            ew.enqueue_readback(ctx);
            sync_lucky(st);                                   // the step's only synchronisation
            if (ew.accept()) break;
        }
        out.lucky = st->lucky;
        bool done = false;
        if (j <= 2) Xstop[j - 1] = out.Xm;
        else {
            if (std::abs(out.Xm - Xstop[0]) < tol) done = true;
            else { Xstop[0] = Xstop[1]; Xstop[1] = out.Xm; }
        }
        if (done || st->lucky) break;
    }
    out.iter = std::min(j, it);
    return out;
}

}  // namespace kr

// result of the last fun_update kept on the device until fetched
struct FunUpdateResult {
    kr::DevBuf<double> Xm;                                  // dim x dim column-major
    std::vector<std::unique_ptr<kr::PanelBuf>> Um;          // basis blocks (bs columns each)
    int64_t n = 0, dim = 0, bs = 0;
    bool identity_basis = false;
    bool has_basis = false;
};

namespace kr {

struct FuInfo { int64_t dim = 0, iter = 0; int lucky = 0; int dense_fallback = 0; };

// fun_update     (fun_update.m:20-137)
inline FuInfo fun_update_general(kr_ctx* ctx, const kr_matrix* M, int64_t rk, const double* U, int64_t ldu,
                                 const HostMat& B, int fun, double tol, int64_t it, bool want_basis,
                                 FunUpdateResult& res) {
    const int64_t n = M->dev.n;
    FuInfo info;
    if (!is_symmetric(B)) fail(KR_ERR_UNSUPPORTED, "fun_update: the device path needs a symmetric (Hermitian) B");
    ExpmWork ew;
    auto dense_fallback = [&](int64_t j, int lucky) {          // :85-90: f(A + U B U') - f(A) in dense arithmetic, Um = I
        const HostMat fA = dense_of(M);
        const HostMat fAt = dense_updated(fA, rk, U, ldu, B, false);
        std::vector<double> both((size_t)2 * n * n);
        std::copy(fAt.a.begin(), fAt.a.end(), both.begin());
        std::copy(fA.a.begin(), fA.a.end(), both.begin() + (size_t)n * n);
        DevBuf<double> dS(ctx, both.size()), dF(ctx, both.size());
        dS.upload(both.data(), both.size());
        symfun_batched(ctx, dS.p, (int)n, 2, fun, std::max(host_norm1(fAt), host_norm1(fA)), dF.p, ew);
        res.Xm.reset(ctx, (size_t)n * n);
        KR_LAUNCH(ctx, axpby_kernel, ew_grid(ctx, n * n), 256, 0, res.Xm.p, 1.0, dF.p, -1.0, dF.p + (size_t)n * n, n * n);
        KR_CUDA(cudaStreamSynchronize(ctx->stream));
        res.n = n; res.dim = n; res.bs = rk; res.identity_basis = true; res.has_basis = true;
        info.dim = n; info.iter = j; info.lucky = lucky; info.dense_fallback = 1;
    };
    // A block wider than the QR kernels take (HQR_WIDEB) whose first Arnoldi step already saturates the space
    // (2 * 2rk >= n): the reference leaves through its dense branch at j = 1 whatever the step produced, so the step
    // is not needed.  lucky is what the step would report for a connected graph: W vanishes only when the block
    // spans everything.
    if (want_basis && rk > HQR_WIDEB && 4 * rk >= n) {
        dense_fallback(1, rk >= n ? 1 : 0);
        return info;
    }
    WideSetup ws = wide_setup(ctx, M, rk, U, ldu, B, want_basis);
    kr_krylov* st = ws.st.get();
    std::vector<DevBuf<double>> Xs;                            // Xm of every step (the lag-2 test needs j-2)
    std::vector<int> Xdim;
    DevBuf<double> SG, F, D, part(ctx, 256), info_dev(ctx, 2), Q;
    DevBuf<int> need(ctx, 1);
    int64_t j = 0;
    for (j = 1; j <= it; ++j) {
        if (j > 1) krylov_step(st);
        if (want_basis && 2 * st->vcols() >= n) {               // :85-90 dense fallback
            sync_lucky(st);
            dense_fallback(j, st->lucky);
            return info;
        }
        const int nn = (int)(j * rk);
        const size_t sz = (size_t)nn * nn;
        if (SG.count < 2 * sz) { SG.reset(ctx, 2 * sz); F.reset(ctx, 2 * sz); D.reset(ctx, sz); }
        KR_LAUNCH(ctx, assemble_proj_kernel, ew_grid(ctx, (int64_t)sz), 256, 0, st->hblocks(), nn, ws.CmS.p, (int)rk, SG.p);
        Xs.emplace_back(ctx, sz);
        Xdim.push_back(nn);
        double hinfo[2] = {0, 0};
        int hneed = 0;
        for (int attempt = 0; attempt < 2; ++attempt) {
            ew.begin(ctx, attempt == 1);
            symfun_batched(ctx, SG.p, nn, 2, fun, ws.norm_bound, F.p, ew);
            KR_LAUNCH(ctx, axpby_kernel, ew_grid(ctx, (int64_t)sz), 256, 0, Xs.back().p, 1.0, F.p, -1.0, F.p + sz, (int64_t)sz);   // :106
            if (j > 2) {
                // || Xm - pad(Xm(j-2)) ||_2 < tol   (:112-114): Frobenius norm first, Lanczos only inside the band
                const int ctas = (int)std::min<int64_t>(256, std::max<int64_t>(1, ceil_div((int64_t)sz, 256)));
                KR_LAUNCH(ctx, diff_sym_kernel, ctas, 256, 0, Xs.back().p, nn, Xs[Xs.size() - 3].p, Xdim[Xdim.size() - 3], D.p, part.p);
                KR_LAUNCH(ctx, stop_band_kernel, 1, 1, 0, part.p, ctas, nn, tol, info_dev.p, need.p);
                if (Q.count < (size_t)nn * (NRM2_STEPS + 1)) Q.reset(ctx, (size_t)nn * (NRM2_STEPS + 1));
                KR_LAUNCH(ctx, sym_norm2_kernel, 1, 256, 0, D.p, nn, Q.p, need.p, tol, info_dev.p + 1);
                KR_CUDA(cudaMemcpyAsync(hinfo, info_dev.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
                KR_CUDA(cudaMemcpyAsync(&hneed, need.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            }
            ew.enqueue_readback(ctx);
            sync_lucky(st);                                   // the step's only synchronisation
            if (ew.accept()) break;
        }
        info.lucky = st->lucky;
        bool done = false;
        if (j > 2) {
            const double err = hneed ? hinfo[1] : hinfo[0];      // inside the band the 2-norm, else the Frobenius bound decides
            done = hneed ? (err < tol) : (hinfo[0] < tol);
        }
        if (done || st->lucky) break;
        if (Xs.size() > 3) { Xs.erase(Xs.begin()); Xdim.erase(Xdim.begin()); }
    }
    info.iter = std::min(j, it);
    info.dim = Xdim.back();
    res.Xm = std::move(Xs.back());
    res.n = n;
    res.dim = Xdim.back();
    res.bs = rk;
    res.identity_basis = false;
    res.has_basis = true;
    // Um(:, 1:size(Xm,1))  (:137) - for Lanczos this is the 2-block window, as in the reference
    res.Um = std::move(st->V);
    KR_CUDA(cudaStreamSynchronize(ctx->stream));
    return info;
}

// ------------------------------------------------------------------------------------ normest
// One CTA runs MATLAB's normest(S, tol) entirely on the device when the matrix is small (the reference's graphs):
// power iteration on S'S from the column abs-sums, data-dependent stopping test included - one launch, no host
// round trip per iteration.  S = A (symmetric) or general with the transpose supplied.
__global__ void __launch_bounds__(1024)
normest_small_kernel(CsrDevView A, CsrDevView At, double tol, double* __restrict__ x, double* __restrict__ sx,
                     double* __restrict__ out /* e, cnt */) {
    __shared__ double red[32];
    __shared__ double s_val;
    const int n = A.n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto bsum = [&](double v) -> double {
        for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        __syncthreads();
        if (lane == 0) red[warp] = v;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int w = 0; w < 32; ++w) s += red[w];
            s_val = s;
        }
        __syncthreads();
        return s_val;
    };
    const int splitA = cta_spmv_split(A), splitT = cta_spmv_split(At);
    auto spmv_cta = [&](const CsrDevView& S, const double* in, double* o) {
        cta_spmv<1024>(S, in, o, nullptr, &S == &A ? splitA : splitT);
    };
    // x = sum(abs(S), 1)' = abs-sums of the columns of S = row abs-sums of S'
    for (int g = warp; g < n; g += 32) {
        const int p0 = At.row_ptr[g], p1 = At.row_ptr[g + 1];
        double s = 0.0;
        for (int p = p0 + lane; p < p1; p += 32) s += fabs(At.val ? At.val[p] : At.uval);
        for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) x[At.row_order[g]] = s;
    }
    __syncthreads();
    double a = 0.0;
    for (int i = tid; i < n; i += 1024) a += x[i] * x[i];
    double e = sqrt(bsum(a));
    double cnt = 0.0;
    if (e == 0.0) {
        if (tid == 0) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; }
        return;
    }
    for (int i = tid; i < n; i += 1024) x[i] /= e;
    __syncthreads();
    double e0 = 0.0;
    int failed = 0;
    while (fabs(e - e0) > tol * e) {
        e0 = e;
        spmv_cta(A, x, sx);
        a = 0.0;
        for (int i = tid; i < n; i += 1024) a += sx[i] * sx[i];
        const double nsx = sqrt(bsum(a));
        if (nsx == 0.0) { failed = 1; break; }
        spmv_cta(At, sx, x);
        a = 0.0;
        for (int i = tid; i < n; i += 1024) a += x[i] * x[i];
        const double nx = sqrt(bsum(a));
        e = nx / nsx;
        const double inv = 1.0 / nx;
        for (int i = tid; i < n; i += 1024) x[i] *= inv;
        __syncthreads();
        cnt += 1.0;
        if (cnt > 100.0) break;
    }
    if (tid == 0) { out[0] = e; out[1] = cnt; out[2] = (double)failed; }
}

__global__ void colabs_rowsum_kernel(CsrDevView At, double* __restrict__ x) {
    const int g = (blockIdx.x * 256 + threadIdx.x) >> 3, sub = threadIdx.x & 7;
    if (g >= At.n) return;
    double s = 0.0;
    for (int p = At.row_ptr[g] + sub; p < At.row_ptr[g + 1]; p += 8) s += fabs(At.val ? At.val[p] : At.uval);
    const unsigned m = __activemask();
    s += __shfl_xor_sync(m, s, 1);
    s += __shfl_xor_sync(m, s, 2);
    s += __shfl_xor_sync(m, s, 4);
    if (sub == 0) x[At.row_order[g]] = s;
}
__global__ void vec_scale_kernel(double* __restrict__ x, int64_t n, double f) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= f;
}

// Leading eigenvector by power iteration, whole loop in ONE CTA (small graphs: launch-bound otherwise).
//   mode 0 ('eig', functions/compute_centrality.m:15-17): y = A (A x) / ||.||  - two products per test so that a
//           bipartite-like oscillation does not fool the stopping rule;
//   mode 1 ('pr', :20-26): y = alpha A D x + (1 - alpha) sum(x) / n, D = diag(1 ./ sum(A)), alpha = 0.85.
// Stops when || y/||y|| - x ||_2 < tol.  out = {iterations, converged}.
__global__ void __launch_bounds__(1024)
power_iteration_small_kernel(CsrDevView A, int mode, double tol, int maxit, double* __restrict__ x, double* __restrict__ y,
                             double* __restrict__ dinv, double* __restrict__ out) {
    __shared__ double red[32];
    __shared__ double s_val;
    const int n = A.n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    auto bsum = [&](double v) -> double {
        for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        __syncthreads();
        if (lane == 0) red[warp] = v;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int w = 0; w < 32; ++w) s += red[w];
            s_val = s;
        }
        __syncthreads();
        return s_val;
    };
    const int split = cta_spmv_split(A);
    auto spmv_cta = [&](const double* in, double* o, const double* scale) { cta_spmv<1024>(A, in, o, scale, split); };
    if (mode == 1) {        // dinv = 1 ./ sum(A) (column sums = row sums of the symmetric A)
        for (int g = warp; g < n; g += 32) {
            double s = 0.0;
            for (int p = A.row_ptr[g] + lane; p < A.row_ptr[g + 1]; p += 32) s += A.val ? A.val[p] : A.uval;
            for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
            if (lane == 0) dinv[A.row_order[g]] = 1.0 / s;
        }
    }
    const double x0 = 1.0 / sqrt((double)n);
    for (int i = tid; i < n; i += 1024) x[i] = x0;
    __syncthreads();
    int it = 0, conv = 0;
    while (it < maxit) {
        if (mode == 0) {
            spmv_cta(x, y, nullptr);
            // x is still needed for the test: the second product lands in a third vector = dinv (unused in mode 0)
            spmv_cta(y, dinv, nullptr);
        } else {
            double sx = 0.0;
            for (int i = tid; i < n; i += 1024) sx += x[i];
            sx = bsum(sx);
            spmv_cta(x, y, dinv);
            const double add = (1.0 - 0.85) * sx / (double)n;
            for (int i = tid; i < n; i += 1024) y[i] = 0.85 * y[i] + add;
            __syncthreads();
        }
        double* z = mode == 0 ? dinv : y;
        double a = 0.0;
        for (int i = tid; i < n; i += 1024) a += z[i] * z[i];
        const double nrm = sqrt(bsum(a));
        if (!(nrm > 0.0)) break;
        double d = 0.0;
        for (int i = tid; i < n; i += 1024) {
            const double v = z[i] / nrm;
            const double e = v - x[i];
            d += e * e;
            z[i] = v;
        }
        d = sqrt(bsum(d));
        for (int i = tid; i < n; i += 1024) x[i] = z[i];
        __syncthreads();
        ++it;
        if (d < tol) { conv = 1; break; }
    }
    if (tid == 0) { out[0] = (double)it; out[1] = (double)conv; }
}

// one step of the same iteration with grid-wide kernels (large graphs); the host reads the distance every few steps
__global__ void pr_combine_kernel(double* __restrict__ y, int64_t n, const double* __restrict__ sumx) {
    const double add = (1.0 - 0.85) * sumx[0] / (double)n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y[i] = 0.85 * y[i] + add;
}
__global__ void vec_mul_kernel(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ o, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) o[i] = a[i] * b[i];
}
__global__ void vec_recip_kernel(double* __restrict__ a, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) a[i] = 1.0 / a[i];
}
// z <- z / sqrt(*n2); partial[b] = sum (z - x)^2; x <- z
__global__ void __launch_bounds__(256)
normalize_diff_kernel(double* __restrict__ z, double* __restrict__ x, int64_t n, const double* __restrict__ n2,
                      double* __restrict__ partial) {
    __shared__ double red[8];
    const double nrm = sqrt(n2[0]);
    const double f = nrm > 0.0 ? 1.0 / nrm : 0.0;
    double d = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const double v = z[i] * f, e = v - x[i];
        d += e * e;
        x[i] = v;
    }
    for (int off = 16; off; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) d += red[w];
        partial[blockIdx.x] = d;
    }
}

struct CentralityInfo { int64_t iters = 0; int converged = 0; };
// c = |leading eigenvector| (unit 2-norm), mode 0 'eig' / mode 1 'pr'
inline CentralityInfo leading_vector_dev(kr_ctx* ctx, const kr_matrix* M, int mode, double tol, int64_t maxit, double* c_host) {
    const int64_t n = M->dev.n;
    CentralityInfo info;
    if (n == 0) return info;
    if (mode == 1 && !M->symmetric) fail(KR_ERR_UNSUPPORTED, "compute_centrality 'pr': the device path expects a symmetric A");
    DevBuf<double> x(ctx, n), y(ctx, n), z(ctx, n), sc(ctx, 4), part(ctx, VEC_RED_CTAS);
    if (M->dev.nnz <= CSR_L2_RESIDENT_NNZ) {
        KR_LAUNCH(ctx, power_iteration_small_kernel, 1, 1024, 0, M->dev.view(), mode, tol, (int)std::min<int64_t>(maxit, 1 << 30), x.p, y.p, z.p, sc.p);
        double h[2];
        sc.download(h, 2);
        info.iters = (int64_t)h[0];
        info.converged = (int)h[1];
    } else {
        const int eg = ew_grid(ctx, n);
        const int ctas = (int)std::min<int64_t>(VEC_RED_CTAS, std::max<int64_t>(1, ceil_div(n, 256)));
        KR_LAUNCH(ctx, fill_kernel, eg, 256, 0, x.p, n, 1.0 / std::sqrt((double)n));
        DevBuf<double> dinv;
        if (mode == 1) {
            dinv.reset(ctx, n);
            KR_LAUNCH(ctx, colabs_rowsum_kernel, (int)ceil_div(n * 8, 256), 256, 0, M->dev.view(), dinv.p);
            KR_LAUNCH(ctx, vec_recip_kernel, eg, 256, 0, dinv.p, n);
        }
        while (info.iters < maxit && !info.converged) {
            double* out = z.p;
            if (mode == 0) {
                spmv(ctx, M->dev, x.p, y.p);
                spmv(ctx, M->dev, y.p, z.p);
            } else {
                vec_reduce<2>(ctx, x.p, x.p, n, part.p, sc.p + 2);           // sum(x): x >= 0 throughout
                KR_LAUNCH(ctx, vec_mul_kernel, eg, 256, 0, x.p, dinv.p, y.p, n);
                spmv(ctx, M->dev, y.p, z.p);
                KR_LAUNCH(ctx, pr_combine_kernel, eg, 256, 0, z.p, n, sc.p + 2);
            }
            vec_reduce<0>(ctx, out, out, n, part.p, sc.p);
            KR_LAUNCH(ctx, normalize_diff_kernel, ctas, 256, 0, out, x.p, n, sc.p, part.p);
            KR_LAUNCH(ctx, vec_reduce_finish_kernel<0>, 1, 1, 0, part.p, ctas, sc.p + 1);
            info.iters += 1;
            double dist = 0;                                             // one scalar per iteration (large graphs only)
            KR_CUDA(cudaMemcpyAsync(&dist, sc.p + 1, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            KR_CUDA(cudaStreamSynchronize(ctx->stream));
            if (std::sqrt(dist) < tol) info.converged = 1;
        }
    }
    std::vector<double> h = x.to_host();
    for (int64_t i = 0; i < n; ++i) c_host[i] = std::abs(h[(size_t)i]);
    return info;
}

// MATLAB normest(S, tol): power iteration on S'S from the column abs-sums
inline void normest_dev(kr_ctx* ctx, const kr_matrix* M, double tol, double* est, int64_t* count) {
    const int64_t n = M->dev.n;
    if (n == 0) { *est = 0; *count = 0; return; }
    DevBuf<double> x(ctx, n), sx(ctx, n), part(ctx, VEC_RED_CTAS), sc(ctx, 4);
    if (M->dev.nnz <= CSR_L2_RESIDENT_NNZ) {
        KR_LAUNCH(ctx, normest_small_kernel, 1, 1024, 0, M->dev.view(), M->T().view(), tol, x.p, sx.p, sc.p);
        double h[3];
        sc.download(h, 3);
        if (h[2] != 0.0) fail(KR_ERR_UNSUPPORTED, "normest: S*x vanished");
        *est = h[0];
        *count = (int64_t)h[1];
        return;
    }
    KR_LAUNCH(ctx, colabs_rowsum_kernel, (int)ceil_div(n * 8, 256), 256, 0, M->T().view(), x.p);
    double h = 0;
    vec_reduce<0>(ctx, x.p, x.p, n, part.p, sc.p);
    sc.download(&h, 1);
    double e = std::sqrt(h);
    int64_t cnt = 0;
    if (e == 0) { *est = 0; *count = 0; return; }
    const int eg = ew_grid(ctx, n);
    KR_LAUNCH(ctx, vec_scale_kernel, eg, 256, 0, x.p, n, 1.0 / e);
    double e0 = 0;
    while (std::abs(e - e0) > tol * e) {
        e0 = e;
        spmv(ctx, M->dev, x.p, sx.p);                                // Sx = S*x
        vec_reduce<0>(ctx, sx.p, sx.p, n, part.p, sc.p);
        spmv(ctx, M->T(), sx.p, x.p);                                // x = S'*Sx
        vec_reduce<0>(ctx, x.p, x.p, n, part.p, sc.p + 1);
        double hh[2];
        sc.download(hh, 2);                                          // one synchronisation per iteration
        if (hh[0] == 0) fail(KR_ERR_UNSUPPORTED, "normest: S*x vanished");
        const double nx = std::sqrt(hh[1]);
        e = nx / std::sqrt(hh[0]);
        KR_LAUNCH(ctx, vec_scale_kernel, eg, 256, 0, x.p, n, 1.0 / nx);
        cnt += 1;
        if (cnt > 100) break;
    }
    *est = e;
    *count = cnt;
}

}  // namespace kr
