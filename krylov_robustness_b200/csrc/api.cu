// api.cu - extern "C" entry points of libkrylov_b200.so (see include/krylov_b200.h).
// Single translation unit: all kernels live in the .cuh files included below.
#include <memory>
#include <thread>
#include "common.cuh"
#include "csr.cuh"
#include "spmm.cuh"
#include "dense.cuh"
#include "slq.cuh"
#include "theta_table.h"
#include "smalldense.cuh"
#include "pairs.cuh"
#include "pairs_small.cuh"
#include "expmv.cuh"
#include "tsdense.cuh"
#include "smallgemm.cuh"
#include "vecops.cuh"
#include "blockkrylov.cuh"
#include "entries.cuh"
#include "entries_local.cuh"
#include "frechet.cuh"
#include "mctrace.cuh"
#include "nodepairs.cuh"
#include "nodes.cuh"
#include "sparse_update.cuh"
#include "hessp_local.cuh"

using namespace kr;

static void destroy_fun_update_result(kr_ctx* c);

struct kr_dense {
    kr_ctx* ctx;
    PanelBuf buf;
};

extern "C" {

const char* kr_last_error(void) { return tls_error().c_str(); }
const char* kr_version(void) { return "krylov_b200 0.1 (sm_100a)"; }

// ----------------------------------------------------------------------------- context
int kr_ctx_create(int device, kr_ctx** out) {
    return guarded([&] {
        if (!out) fail(KR_ERR_ARG, "kr_ctx_create: null output");
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) {
            cudaGetLastError();
            fail(KR_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                 e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        }
        if (device < 0 || device >= count) fail(KR_ERR_ARG, "device %d out of range (0..%d)", device, count - 1);
        KR_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        KR_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            fail(KR_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                 prop.major, prop.minor);
        kr_ctx* c = new kr_ctx();
        c->device = device;
        c->num_sms = prop.multiProcessorCount;
        c->l2_bytes = (size_t)prop.l2CacheSize;
        KR_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        *out = c;
    });
}

void kr_ctx_destroy(kr_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    destroy_fun_update_result(c);
    for (auto& ev : c->spmm_events) {
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    for (auto ev : c->free_events) cudaEventDestroy(ev);
    c->trim();
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int kr_ctx_sync(kr_ctx* c) {
    return guarded([&] {
        KR_CUDA(cudaSetDevice(c->device));
        KR_CUDA(cudaStreamSynchronize(c->stream));
    });
}

int kr_ctx_counters(kr_ctx* c, int64_t out[5]) {
    return guarded([&] {
        for (int i = 0; i < 5; ++i) out[i] = c->counters[i];
    });
}

int kr_ctx_set_timing(kr_ctx* c, int on) {
    return guarded([&] { c->timing = on != 0; });
}

int kr_ctx_spmm_time(kr_ctx* c, int reset, double* ms, int64_t* launches) {
    return guarded([&] {
        KR_CUDA(cudaStreamSynchronize(c->stream));
        for (auto& ev : c->spmm_events) {
            float t = 0.f;
            KR_CUDA(cudaEventElapsedTime(&t, ev.first, ev.second));
            c->spmm_ms += t;
            c->spmm_timed += 1;
            c->free_events.push_back(ev.first);
            c->free_events.push_back(ev.second);
        }
        c->spmm_events.clear();
        if (ms) *ms = c->spmm_ms;
        if (launches) *launches = c->spmm_timed;
        if (reset) {
            c->spmm_ms = 0.0;
            c->spmm_timed = 0;
        }
    });
}

void* kr_ctx_stream(kr_ctx* c) { return c ? (void*)c->stream : nullptr; }

// ----------------------------------------------------------------------------- matrix
int kr_matrix_create(kr_ctx* ctx, int64_t n, int64_t nnz, const int64_t* row_ptr, const int64_t* col_idx,
                     const double* val, kr_matrix** out) {
    return guarded([&] {
        if (!ctx || !out || !row_ptr || (nnz > 0 && (!col_idx || !val)))
            fail(KR_ERR_ARG, "kr_matrix_create: null argument");
        if (n < 0 || nnz < 0 || row_ptr[0] != 0 || row_ptr[n] != nnz)
            fail(KR_ERR_ARG, "kr_matrix_create: inconsistent row_ptr (the matrix A should be square, CSR, 0-based)");
        KR_CUDA(cudaSetDevice(ctx->device));
        std::unique_ptr<kr_matrix> M(new kr_matrix());
        M->ctx = ctx;
        M->host.n = n;
        M->host.row_ptr.assign(row_ptr, row_ptr + n + 1);
        M->host.col.resize(nnz);
        M->host.val.resize(nnz);
        for (int64_t i = 0; i < n; ++i)
            if (row_ptr[i + 1] < row_ptr[i]) fail(KR_ERR_ARG, "kr_matrix_create: row_ptr not monotone");
        int bad = 0;
#pragma omp parallel for reduction(|| : bad) schedule(static)
        for (int64_t p = 0; p < nnz; ++p) {
            bad = bad || col_idx[p] < 0 || col_idx[p] >= n;
            M->host.col[p] = (int32_t)col_idx[p];
            M->host.val[p] = val[p];
        }
        if (bad) fail(KR_ERR_ARG, "kr_matrix_create: column index out of range (The matrix A should be square)");
        analyse_and_upload(M.get());
        *out = M.release();
        // KR_GPUS=N: every matrix is replicated on N GPUs of this process, so callers that know nothing about devices
        // (the MATLAB wrappers: Tests/*.m unchanged) shard their candidate edges / probe columns across them
        if (const char* e = getenv("KR_GPUS")) {
            const int want = atoi(e);
            if (want > 1 && kr_matrix_replicate(*out, want, nullptr) != 0) {
                const std::string m = kr_last_error();
                kr_matrix_destroy(*out);
                *out = nullptr;
                fail(KR_ERR_CUDA, "KR_GPUS=%d: %s", want, m.c_str());
            }
        }
    });
}

void kr_matrix_destroy(kr_matrix* A) {
    if (!A) return;
    for (kr_matrix* P : A->peers) {              // replicas own their context
        kr_ctx* pc = P->ctx;
        cudaSetDevice(pc->device);
        delete P;
        kr_ctx_destroy(pc);
    }
    A->peers.clear();
    cudaSetDevice(A->ctx->device);
    delete A;
}

int kr_matrix_replicate(kr_matrix* A, int ndev, const int* devices) {
    return guarded([&] {
        if (!A || A->is_peer) fail(KR_ERR_ARG, "kr_matrix_replicate: null matrix or a replica");
        if (!A->peers.empty()) fail(KR_ERR_ARG, "kr_matrix_replicate: the matrix already has replicas");
        int count = 0;
        KR_CUDA(cudaGetDeviceCount(&count));
        std::vector<int> devs;
        if (ndev <= 0 || !devices) {
            const int want = ndev <= 0 ? count : std::min(ndev, count);
            for (int d = 0; d < count && (int)devs.size() < want - 1; ++d)
                if (d != A->ctx->device) devs.push_back(d);
        } else {
            for (int k = 0; k < ndev; ++k) {
                if (devices[k] < 0 || devices[k] >= count) fail(KR_ERR_ARG, "kr_matrix_replicate: device %d out of range", devices[k]);
                if (devices[k] != A->ctx->device) devs.push_back(devices[k]);
            }
        }
        materialize(A);                              // replicas start from the current matrix
        const CsrHost& H = A->host;
        std::vector<int> status(devs.size(), 0);
        std::vector<std::string> msg(devs.size());
        std::vector<kr_matrix*> made(devs.size(), nullptr);
        std::vector<std::thread> th;
        for (size_t k = 0; k < devs.size(); ++k)
            th.emplace_back([&, k] {
                status[k] = guarded([&] {
                    kr_ctx* pc = nullptr;
                    if (kr_ctx_create(devs[k], &pc) != 0) fail(KR_ERR_CUDA, "%s", kr_last_error());
                    std::unique_ptr<kr_matrix> M(new kr_matrix());
                    M->ctx = pc;
                    M->host = H;
                    M->is_peer = true;
                    try { analyse_and_upload(M.get()); } catch (...) { M.reset(); kr_ctx_destroy(pc); throw; }
                    made[k] = M.release();
                });
                if (status[k]) msg[k] = kr_last_error();
            });
        for (auto& t : th) t.join();
        for (size_t k = 0; k < devs.size(); ++k)
            if (status[k]) {
                for (kr_matrix* P : made)
                    if (P) { kr_ctx* pc = P->ctx; cudaSetDevice(pc->device); delete P; kr_ctx_destroy(pc); }
                fail(status[k], "%s", msg[k].c_str());
            }
        A->peers = made;
        KR_CUDA(cudaSetDevice(A->ctx->device));
    });
}

int kr_matrix_replicas(const kr_matrix* A) { return A ? 1 + (int)A->peers.size() : 0; }

int kr_matrix_info(const kr_matrix* A, int64_t* n, int64_t* nnz, int* symmetric, int* pattern_only,
                   int* nonnegative) {
    return guarded([&] {
        if (!A) fail(KR_ERR_ARG, "null matrix");
        // A = stored CSR + pending edits (kr_matrix_set_edges).  Describe the edited matrix without folding the edits
        // in, so that asking does not change which kernels the next call runs: every pending entry creates, keeps or
        // removes one stored entry, and only an edit that clears a stored negative value needs a rescan.
        const CsrHost& H = A->host;
        int64_t count = A->dev.nnz;
        bool neg_edit = false, neg_cleared = false;
        for (const auto& kv : A->pending) {
            const int64_t i = kv.first.first, j = kv.first.second;
            const int32_t* b = H.col.data() + H.row_ptr[i];
            const int32_t* e = H.col.data() + H.row_ptr[i + 1];
            const int32_t* q = std::lower_bound(b, e, (int32_t)j);
            const bool stored = q != e && *q == (int32_t)j;
            const double old = stored ? H.val[(size_t)(q - H.col.data())] : 0.0;
            const double now = old + kv.second;              // the value flush_pending stores
            count += (int64_t)(now != 0.0) - (int64_t)stored;
            neg_edit = neg_edit || now < 0;
            neg_cleared = neg_cleared || (old < 0 && !(now < 0));
        }
        bool nonneg = A->nonnegative && !neg_edit;
        if (!A->nonnegative && !neg_edit && neg_cleared) {   // is any stored negative left that no edit overrides?
            nonneg = true;
            for (int64_t i = 0; i < H.n && nonneg; ++i)
                for (int64_t p = H.row_ptr[i]; p < H.row_ptr[i + 1]; ++p)
                    if (H.val[(size_t)p] < 0 && !A->pending.count({i, (int64_t)H.col[(size_t)p]})) { nonneg = false; break; }
        }
        if (n) *n = A->dev.n;
        if (nnz) *nnz = count;
        if (symmetric) *symmetric = A->symmetric;
        if (pattern_only) *pattern_only = A->dev.pattern_only;
        if (nonnegative) *nonnegative = nonneg;
    });
}

int kr_matrix_set_edges(kr_matrix* A, int64_t count, const int64_t* ii, const int64_t* jj, const double* v) {
    return guarded([&] {
        if (!A) fail(KR_ERR_ARG, "null matrix");
        KR_CUDA(cudaSetDevice(A->ctx->device));
        const CsrHost& H = A->host;
        const int64_t n = H.n;
        for (int64_t e = 0; e < count; ++e) {
            const int64_t i = ii[e] - 1, j = jj[e] - 1;
            if (i < 0 || i >= n || j < 0 || j >= n) fail(KR_ERR_ARG, "kr_matrix_set_edges: index out of range");
            // both triangles (functions/krylov_miobi.m:129-135); recorded as (new value - stored value)
            A->pending[{i, j}] = v[e] - host_entry(H, i, j);
            A->pending[{j, i}] = v[e] - host_entry(H, j, i);
        }
        for (auto it = A->pending.begin(); it != A->pending.end();)
            it = (it->second == 0.0) ? A->pending.erase(it) : std::next(it);
        // The device keeps the stored CSR untouched and applies the few pending entries on the fly in the SpMM and
        // in the candidate-seed kernel (the greedy loop's only consumers): no host rebuild, no re-upload of A per
        // round.  Unsymmetric matrices (a transposed copy exists) and very long edit lists take the rebuild.
        if (!A->symmetric || A->pending.size() > KR_MAX_PENDING) flush_pending(A);
        else upload_pending(A);
        for (kr_matrix* P : A->peers)                // the same edit on every replica (a few hundred bytes each)
            if (kr_matrix_set_edges(P, count, ii, jj, v) != 0) fail(KR_ERR_CUDA, "replica on device %d: %s", P->ctx->device, kr_last_error());
        KR_CUDA(cudaSetDevice(A->ctx->device));
    });
}

// ----------------------------------------------------------------------------- dense blocks
int kr_dense_create(kr_ctx* ctx, int64_t n, int64_t k, kr_dense** out) {
    return guarded([&] {
        if (!ctx || !out || n < 0 || k < 0 || k > (1 << 20)) fail(KR_ERR_ARG, "kr_dense_create: bad argument");
        KR_CUDA(cudaSetDevice(ctx->device));
        std::unique_ptr<kr_dense> d(new kr_dense());
        d->ctx = ctx;
        d->buf.reset(ctx, n, (int)k);
        *out = d.release();
    });
}

void kr_dense_destroy(kr_dense* d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    delete d;
}

static void upload_cm(kr_ctx* ctx, const double* host, int64_t ld, PanelBuf& dst) { upload_cm_block(ctx, host, ld, dst); }
static void download_cm(kr_ctx* ctx, const PanelBuf& src, double* host, int64_t ld) { download_cm_block(ctx, src, host, ld); }

int kr_dense_upload(kr_dense* d, const double* host, int64_t ld) {
    return guarded([&] {
        if (!d || !host) fail(KR_ERR_ARG, "kr_dense_upload: null argument");
        KR_CUDA(cudaSetDevice(d->ctx->device));
        upload_cm(d->ctx, host, ld, d->buf);
    });
}

int kr_dense_download(const kr_dense* d, double* host, int64_t ld) {
    return guarded([&] {
        if (!d || !host) fail(KR_ERR_ARG, "kr_dense_download: null argument");
        KR_CUDA(cudaSetDevice(d->ctx->device));
        download_cm(d->ctx, d->buf, host, ld);
    });
}

int kr_dense_fill_rademacher(kr_dense* d, uint64_t seed, int64_t col_offset) {
    return guarded([&] {
        if (!d) fail(KR_ERR_ARG, "null block");
        KR_CUDA(cudaSetDevice(d->ctx->device));
        if (d->buf.elems() == 0) return;
        KR_LAUNCH(d->ctx, rademacher_kernel, d->ctx->num_sms * 8, 256, 0, d->buf.p(), d->buf.n, d->buf.cols,
                  d->buf.panels, seed, col_offset);
    });
}

// ----------------------------------------------------------------------------- SpMM
int kr_spmm_dev(kr_ctx* ctx, const kr_matrix* A, const kr_dense* X, kr_dense* Y) {
    return guarded([&] {
        if (!ctx || !A || !X || !Y) fail(KR_ERR_ARG, "kr_spmm_dev: null argument");
        if (X->buf.n != A->dev.n) fail(KR_ERR_ARG, "The block vector b has wrong number of rows");
        if (Y->buf.n != X->buf.n || Y->buf.cols != X->buf.cols || Y->buf.p() == X->buf.p())
            fail(KR_ERR_ARG, "kr_spmm_dev: Y must be a distinct block of the same shape as X");
        KR_CUDA(cudaSetDevice(ctx->device));
        EpiPlain epi{Y->buf.p(), X->buf.p(), 1.0, 0.0};
        launch_spmm(ctx, A->dev, X->buf.p(), X->buf.panels, epi, nullptr, X->buf.cols);
    });
}

int kr_spmm(kr_ctx* ctx, const kr_matrix* A, int64_t k, const double* X, int64_t ldx, double* Y, int64_t ldy) {
    return guarded([&] {
        if (!ctx || !A || !X || !Y) fail(KR_ERR_ARG, "kr_spmm: null argument");
        KR_CUDA(cudaSetDevice(ctx->device));
        const int64_t n = A->dev.n;
        PanelBuf xb(ctx, n, (int)k), yb(ctx, n, (int)k);
        upload_cm(ctx, X, ldx, xb);
        EpiPlain epi{yb.p(), xb.p(), 1.0, 0.0};
        launch_spmm(ctx, A->dev, xb.p(), xb.panels, epi, nullptr, (int)k);
        download_cm(ctx, yb, Y, ldy);
    });
}

// ----------------------------------------------------------------------------- SLQ trace
static void slq_finish(const SlqResult& R, int64_t m, double* tr, double* vals, double* alpha, double* beta) {
    if (tr) *tr = R.tr;
    const size_t k = R.vals.size();
    if (vals) std::memcpy(vals, R.vals.data(), k * sizeof(double));
    if (alpha || beta)
        for (int64_t j = 0; j < m; ++j)
            for (size_t c = 0; c < k; ++c) {       // output is m x k column-major
                if (alpha) alpha[c * m + j] = R.alpha[(size_t)j * k + c];
                if (beta) beta[c * m + j] = R.beta[(size_t)j * k + c];
            }
}

int kr_slq_trace_dev(kr_ctx* ctx, const kr_matrix* A, const kr_dense* Z, int64_t m, int fun, double* tr,
                     double* vals, double* alpha, double* beta) {
    return guarded([&] {
        if (!ctx || !A || !Z) fail(KR_ERR_ARG, "kr_slq_trace_dev: null argument");
        if (fun < 0 || fun > 2) fail(KR_ERR_ARG, "unsupported function selector");
        KR_CUDA(cudaSetDevice(ctx->device));
        // work on a copy: the caller's probe block stays intact for the next step
        PanelBuf W(ctx, Z->buf.n, Z->buf.cols);
        KR_CUDA(cudaMemcpyAsync(W.p(), Z->buf.p(), (size_t)W.elems() * sizeof(double), cudaMemcpyDeviceToDevice,
                                ctx->stream));
        SlqResult R = slq_run(ctx, A, W, (int)m, fun, alpha || beta);
        slq_finish(R, m, tr, vals, alpha, beta);
    });
}

}  // extern "C"

// Host-buffer SLQ pipeline shared by kr_slq_trace (fp64 probes) and kr_slq_trace_sign (int8 sign probes).
template <class T>
static int slq_trace_host(kr_ctx* ctx, const kr_matrix* A, int64_t k, const T* Z, int64_t ldz, int64_t m, int fun,
                          double* tr, double* vals, double* alpha, double* beta) {
    return guarded([&] {
        if (!ctx || !A || !Z) fail(KR_ERR_ARG, "kr_slq_trace: null argument");
        if (fun < 0 || fun > 2) fail(KR_ERR_ARG, "unsupported function selector");
        KR_CUDA(cudaSetDevice(ctx->device));
        const int64_t n = A->dev.n;
        if (ldz < n) fail(KR_ERR_ARG, "The block vector b has wrong number of rows");
        if (k <= 0) fail(KR_ERR_ARG, "kr_slq_trace: no probe columns");
        // Probe columns are independent, so the block is processed in column chunks: chunk c+1 is copied
        // host -> device and re-laid out on a second stream while chunk c runs its m Lanczos steps, and
        // chunk c+1 is enqueued before the host waits for chunk c (the GPU never drains between chunks).
        // The first chunk is small so that compute starts after a few milliseconds of upload.
        std::vector<int64_t> cstart, cwidth;
        for (int64_t c0 = 0; c0 < k;) {
            const int64_t cw = std::min<int64_t>(k - c0, cstart.empty() ? 2 * PW : (cstart.size() == 1 ? 6 * PW : 8 * PW));
            cstart.push_back(c0);
            cwidth.push_back(cw);
            c0 += cw;
        }
        if (cstart.empty()) { cstart.push_back(0); cwidth.push_back(0); }
        const int64_t nch = (int64_t)cstart.size();
        if (!ctx->copy_stream) KR_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        std::vector<std::unique_ptr<PanelBuf>> W(nch);
        std::vector<std::unique_ptr<DevBuf<T>>> stage(nch);
        std::vector<cudaEvent_t> ready(nch, nullptr);
        for (int64_t c = 0; c < nch; ++c) {
            W[c].reset(new PanelBuf(ctx, n, (int)cwidth[c]));
            stage[c].reset(new DevBuf<T>(ctx, (size_t)std::max<int64_t>(n * cwidth[c], 1)));
        }
        KR_CUDA(cudaStreamSynchronize(ctx->stream));     // pool buffers may still be in use by earlier work
        auto issue_copy = [&](int64_t c) {
            const int64_t c0 = cstart[c], cw = cwidth[c];
            if (n > 0 && cw > 0) {
                KR_CUDA(cudaMemcpy2DAsync(stage[c]->p, n * sizeof(T), Z + c0 * ldz, ldz * sizeof(T),
                                          n * sizeof(T), cw, cudaMemcpyHostToDevice, ctx->copy_stream));
                ctx->counters[3] += n * cw * (int64_t)sizeof(T);
            }
            cm_to_panel(ctx, stage[c]->p, n, *W[c], ctx->copy_stream);
            KR_CUDA(cudaEventCreateWithFlags(&ready[c], cudaEventDisableTiming));
            KR_CUDA(cudaEventRecord(ready[c], ctx->copy_stream));
        };
        std::vector<double> all_vals((size_t)k), all_a, all_b;
        if (alpha || beta) { all_a.resize((size_t)m * k); all_b.resize((size_t)m * k); }
        auto harvest = [&](int64_t c, SlqJob& job) {
            const int64_t c0 = cstart[c], cw = cwidth[c];
            SlqResult R = job.collect();
            for (int64_t q = 0; q < cw; ++q) all_vals[(size_t)(c0 + q)] = R.vals[(size_t)q];
            if (alpha || beta)
                for (int64_t j = 0; j < m; ++j)
                    for (int64_t q = 0; q < cw; ++q) {
                        all_a[(size_t)(j * k + c0 + q)] = R.alpha[(size_t)(j * cw + q)];
                        all_b[(size_t)(j * k + c0 + q)] = R.beta[(size_t)(j * cw + q)];
                    }
        };
        try {
            issue_copy(0);
            std::unique_ptr<SlqJob> prev;
            for (int64_t c = 0; c < nch; ++c) {
                KR_CUDA(cudaStreamWaitEvent(ctx->stream, ready[c], 0));
                std::unique_ptr<SlqJob> job(new SlqJob(ctx, A, *W[c], (int)m, fun, alpha || beta));   // enqueue chunk c
                job->mark();
                if (c + 1 < nch) issue_copy(c + 1);      // overlaps with chunk c (also when the host buffer is
                                                         // pageable and the copy call blocks)
                if (prev) harvest(c - 1, *prev);
                prev = std::move(job);
            }
            if (prev) harvest(nch - 1, *prev);
        } catch (...) {
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamSynchronize(ctx->stream);
            for (auto e : ready) if (e) cudaEventDestroy(e);
            throw;
        }
        KR_CUDA(cudaStreamSynchronize(ctx->copy_stream));
        for (auto e : ready) if (e) cudaEventDestroy(e);
        SlqResult R;
        R.vals = all_vals;
        R.alpha = all_a;
        R.beta = all_b;
        double s = 0.0;
        for (int64_t q = 0; q < k; ++q) s += all_vals[(size_t)q];
        R.tr = k ? s / (double)k : 0.0;
        slq_finish(R, m, tr, vals, alpha, beta);
    });
}

// Probe columns split contiguously across the replicas of A (SURVEY.md 8e: A replicated, columns sharded), one host
// thread per GPU; the exchange step is the sum of the per-GPU partial traces, done on the host.
template <class T>
static int slq_trace_sharded(kr_ctx* ctx, const kr_matrix* A, int64_t k, const T* Z, int64_t ldz, int64_t m, int fun,
                             double* tr, double* vals, double* alpha, double* beta) {
    const int R = 1 + (int)A->peers.size();
    if (R == 1 || k < 2 * R || !Z) return slq_trace_host<T>(ctx, A, k, Z, ldz, m, fun, tr, vals, alpha, beta);
    std::vector<int> status(R, 0);
    std::vector<std::string> msg(R);
    std::vector<double> part(R, 0.0);
    std::vector<std::thread> th;
    for (int r = 0; r < R; ++r)
        th.emplace_back([&, r] {
            const int64_t lo = k * r / R, hi = k * (r + 1) / R;
            const kr_matrix* Ar = r == 0 ? A : A->peers[(size_t)r - 1];
            status[r] = slq_trace_host<T>(r == 0 ? ctx : Ar->ctx, Ar, hi - lo, Z + lo * ldz, ldz, m, fun, &part[r],
                                          vals ? vals + lo : nullptr, alpha ? alpha + lo * m : nullptr,
                                          beta ? beta + lo * m : nullptr);
            if (status[r]) msg[r] = kr_last_error();
        });
    for (auto& t : th) t.join();
    cudaSetDevice(ctx->device);
    for (int r = 0; r < R; ++r)
        if (status[r]) { tls_error() = msg[r]; return status[r]; }
    double s = 0.0;
    for (int r = 0; r < R; ++r) s += part[r] * (double)(k * (r + 1) / R - k * r / R);     // fixed order
    if (tr) *tr = s / (double)k;
    return KR_OK;
}

extern "C" {

int kr_slq_trace(kr_ctx* ctx, const kr_matrix* A, int64_t k, const double* Z, int64_t ldz, int64_t m, int fun,
                 double* tr, double* vals, double* alpha, double* beta) {
    if (!ctx || !A) { tls_error() = "kr_slq_trace: null argument"; return KR_ERR_ARG; }
    return slq_trace_sharded<double>(ctx, A, k, Z, ldz, m, fun, tr, vals, alpha, beta);
}

int kr_slq_trace_sign(kr_ctx* ctx, const kr_matrix* A, int64_t k, const signed char* Z, int64_t ldz, int64_t m, int fun,
                      double* tr, double* vals, double* alpha, double* beta) {
    if (!ctx || !A) { tls_error() = "kr_slq_trace: null argument"; return KR_ERR_ARG; }
    return slq_trace_sharded<signed char>(ctx, A, k, Z, ldz, m, fun, tr, vals, alpha, beta);
}

int kr_theta(double theta[100]) {
    return guarded([&] { std::memcpy(theta, KR_THETA, sizeof(KR_THETA)); });
}

}  // extern "C"

#include "api_l2.inc"

