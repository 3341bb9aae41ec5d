// slq.cuh - throughput-mode trace estimator (SURVEY.md 8d, config C3): all probes at once,
// single-vector Lanczos per probe column, no reorthogonalisation, Gauss quadrature at the end.
//
// Per step and per probe the dense traffic is 48 B per row: the SpMM writes y and re-reads u_j for
// the fused alpha dot (16 B), the three-term update reads y, u_j, u_{j-1} and writes w (32 B).
// Basis vectors are never normalised in memory: v_j = s_j * u_j with the scale folded into the
// per-probe coefficients of the next update, which removes a full read+write pass per step.
#pragma once
#include "dense.cuh"

namespace kr {

struct SlqResult {
    double tr = 0.0;
    std::vector<double> vals, alpha, beta;   // alpha/beta: [m][cols] row-major
};

// One SLQ job on a panel-major probe block: enqueue() launches every kernel of the m Lanczos steps and the
// quadrature without touching the host; collect() brings the per-probe values back.  Splitting the two
// lets a caller overlap the host->device copy of the next column chunk with this chunk's compute.
//
// The probes Z are only read: they are the U1 of step 0 and the U0 of step 1.  Z is an fp64 block or an int8
// sign panel (XT = signed char: +-1 probes at 1/8 of the bytes, the same numbers); either way every value the
// job returns is the same to the bit.  Two work blocks P, Q and Y hold the rest: step 0 writes its W into P,
// step 1 gathers P and writes into Q, and from step 2 on W overwrites U0.  Dropped as dead work: the U0 = 0
// term of step 0 (its coefficient is -0 * 0), and at the last step the update and the store of Y when alpha /
// beta are not asked for (the quadrature never reads beta_{m-1}); with them, the last update only sums |w|^2.
struct SlqJob {
    kr_ctx* ctx;
    int m, cols, tc;
    bool want_ab;
    PanelBuf P, Q, Y;
    DevBuf<double> partial, sums, scal, alpha, beta, vals;

    template <class XT>
    SlqJob(kr_ctx* c, const kr_matrix* M, int64_t zn, int zcols, const XT* Z, int m_, int fun, bool want_ab_)
        : ctx(c), m(m_), want_ab(want_ab_) {
        if (m < 1 || m > SLQ_MAX_M) fail(KR_ERR_ARG, "slq: m must be in 1..%d", SLQ_MAX_M);
        const CsrDev& A = M->dev;
        const int64_t n = A.n;
        if (zn != n) fail(KR_ERR_ARG, "The block vector b has wrong number of rows");
        cols = zcols;
        const int panels = (cols + PW - 1) / PW;
        tc = panels * PW;
        P.reset(ctx, n, cols);
        if (m > 2) Q.reset(ctx, n, cols);
        Y.reset(ctx, n, cols);
        const int rb = col_row_blocks(n);
        const int nparts = std::max(rb, A.ntiles);
        partial.reset(ctx, (size_t)nparts * tc);
        sums.reset(ctx, tc);
        scal.reset(ctx, (size_t)tc * 7);               // s1, s0, beta_prev, coef[3], nrm2
        alpha.reset(ctx, (size_t)m * tc);
        beta.reset(ctx, (size_t)m * tc);
        vals.reset(ctx, tc);
        scal.zero();
        SlqState st;
        st.s1 = scal.p;
        st.s0 = scal.p + tc;
        st.beta_prev = scal.p + 2 * tc;
        st.coef = scal.p + 3 * tc;
        double* nrm2 = scal.p + 6 * tc;
        st.alpha = alpha.p;
        st.beta = beta.p;
        const int sb = (int)ceil_div(tc, 128);
        const dim3 cgrid((unsigned)rb, (unsigned)panels);
        KR_LAUNCH(ctx, colnorm2_kernel, cgrid, COL_THREADS, 0, Z, n, partial.p, tc);
        sum_partials(ctx, partial.p, rb, tc, sums.p);
        KR_LAUNCH(ctx, slq_init_kernel, sb, 128, 0, sums.p, tc, st, nrm2);
        double* U1 = P.p();
        double* U0 = Q.p();
        for (int j = 0; j < m; ++j) {
            const bool last = j == m - 1;
            const bool store = !last || want_ab;       // Y is read by this step's update
            if (j == 0) spmm_dot(A, Z, panels, store);
            else spmm_dot(A, (const double*)U1, panels, store);
            sum_partials(ctx, partial.p, A.ntiles, tc, sums.p);
            KR_LAUNCH(ctx, slq_alpha_kernel, sb, 128, 0, sums.p, tc, st, j);
            if (!store) break;
            if (j == 0) update(cgrid, n, Z, (const void*)nullptr, P.p(), !last);
            else if (j == 1) update(cgrid, n, (const double*)P.p(), Z, Q.p(), !last);
            else update(cgrid, n, (const double*)U1, (const double*)U0, U0, !last);
            sum_partials(ctx, partial.p, rb, tc, sums.p);
            KR_LAUNCH(ctx, slq_beta_kernel, sb, 128, 0, sums.p, tc, st, j);
            if (j >= 1) std::swap(U0, U1);             // after step 1: U1 = Q, U0 = P
        }
        KR_LAUNCH(ctx, slq_quadrature_kernel, (int)ceil_div(cols, 64), 64, 0, alpha.p, beta.p, nrm2, m, cols, tc, fun, vals.p);
    }

    // Y = A * X with the fused alpha dot; the row operand of the dot is X itself
    template <class XT>
    void spmm_dot(const CsrDev& A, const XT* X, int panels, bool store) {
        if (store) launch_spmm(ctx, A, X, panels, EpiDotT<XT, true>{Y.p(), X, partial.p, tc}, nullptr, cols);
        else launch_spmm(ctx, A, X, panels, EpiDotT<XT, false>{Y.p(), X, partial.p, tc}, nullptr, cols);
    }
    template <class T1, class T0>
    void update(dim3 cgrid, int64_t n, const T1* U1, const T0* U0, double* W, bool store) {
        if (store)
            combine3_norm_kernel<T1, T0, true><<<cgrid, COL_THREADS, 0, ctx->stream>>>(Y.p(), U1, U0, W, n, scal.p + 3 * tc, tc, partial.p);
        else
            combine3_norm_kernel<T1, T0, false><<<cgrid, COL_THREADS, 0, ctx->stream>>>(Y.p(), U1, U0, W, n, scal.p + 3 * tc, tc, partial.p);
        check_launch(ctx, "combine3_norm_kernel");
    }

    // non-blocking completion marker: lets a caller enqueue the next job before waiting for this one
    cudaEvent_t finished = nullptr;
    void mark() {
        KR_CUDA(cudaEventCreateWithFlags(&finished, cudaEventDisableTiming));
        KR_CUDA(cudaEventRecord(finished, ctx->stream));
    }
    ~SlqJob() { if (finished) cudaEventDestroy(finished); }

    SlqResult collect() {
        SlqResult R;
        std::vector<double> v(vals.count);
        if (finished) {
            // wait for THIS job only (later jobs may already be queued behind it), then copy on the copy stream
            KR_CUDA(cudaEventSynchronize(finished));
            cudaStream_t cs = ctx->copy_stream ? ctx->copy_stream : ctx->stream;
            KR_CUDA(cudaMemcpyAsync(v.data(), vals.p, v.size() * sizeof(double), cudaMemcpyDeviceToHost, cs));
            KR_CUDA(cudaStreamSynchronize(cs));
            ctx->counters[4] += (int64_t)(v.size() * sizeof(double));
        } else {
            v = vals.to_host();
        }
        R.vals.assign(v.begin(), v.begin() + cols);
        double s = 0.0;
        for (int c = 0; c < cols; ++c) s += R.vals[c];
        R.tr = cols ? s / cols : 0.0;
        if (want_ab) {
            if (finished) KR_CUDA(cudaStreamSynchronize(ctx->stream));
            std::vector<double> a = alpha.to_host(), b = beta.to_host();
            R.alpha.resize((size_t)m * cols);
            R.beta.resize((size_t)m * cols);
            for (int j = 0; j < m; ++j)
                for (int c = 0; c < cols; ++c) {
                    R.alpha[(size_t)j * cols + c] = a[(size_t)j * tc + c];
                    R.beta[(size_t)j * cols + c] = b[(size_t)j * tc + c];
                }
        }
        return R;
    }
};


}  // namespace kr
