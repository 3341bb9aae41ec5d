// csr.cuh - device-resident CSR adjacency + host-side preprocessing (row binning / tiling).
//
// Replaces MATLAB's sparse A on the path `w = A*w` (functions/lanczos_krylov.m:81,
// functions/arnoldi_krylov.m:86, functions/expmv.m:77, functions/normAm.m:20).
//
// Layout in HBM: the ROWS are stored sorted by decreasing length (`row_order[s]` = original index of
// stored row s): row_ptr int32[n+1] over the stored order, col_idx int32[nnz] (ORIGINAL column
// numbers - X and Y keep the caller's row numbering), val fp64[nnz] (omitted when every stored value
// is the same number -> 4 B per nonzero instead of 12).  `tiles` cuts the stored order into CTA work
// items: a tile is a run of rows of one lanes-per-row class whose nonzeros are CONTIGUOUS and fit the
// CTA's shared-memory staging buffer (SPMM_CAP), so the kernel streams a tile's indices with coalesced
// loads once and only the X gathers remain as dependent global loads.  Rows longer than
// SPMM_LONG_ROW get a tile (and a whole CTA) of their own.
#pragma once
#include <algorithm>
#include <map>
#include <numeric>

#include "common.cuh"

namespace kr {

struct RowTile {
    int start;      // offset into row_order
    int count;      // rows in this tile
    int lanes_log2; // log2 of the nonzero slots per row (0..3); 6 = one long row for the whole CTA
    int pad;
};

struct CsrHost {
    int64_t n = 0;
    std::vector<int64_t> row_ptr;
    std::vector<int32_t> col;
    std::vector<double> val;
};

struct CsrDevView {
    int n;
    int ntiles;
    const int* __restrict__ row_ptr;  // over the stored (sorted) row order
    const int* __restrict__ col;
    const double* __restrict__ val;   // nullptr => all values == uval
    double uval;
    const int* __restrict__ row_order;
    const int* __restrict__ row_pos;  // inverse of row_order: stored position of original row i
    const RowTile* __restrict__ tiles;
    // pending edge edits (kr_matrix_set_edges between two rounds of the greedy loop, functions/krylov_miobi.m:127-135):
    // A = stored CSR + sum of delta entries.  Sorted by stored row; dl_tile_begin[t] .. [t+1] are tile t's entries,
    // dl_row_begin-less lookups scan that (tiny) range.  All null when there is nothing pending.
    const int* __restrict__ dl_tile_begin;   // [ntiles + 1]
    const int* __restrict__ dl_rowlocal;     // row index inside its tile
    const int* __restrict__ dl_pos;          // stored row position
    const int* __restrict__ dl_col;          // column (original numbering)
    const double* __restrict__ dl_val;       // new value - stored value
    int dl_count;
};

#ifndef KR_SPMM_CAP
#define KR_SPMM_CAP 4096
#endif
#ifndef KR_SPMM_MAX_ROWS
#define KR_SPMM_MAX_ROWS 1024
#endif
constexpr int SPMM_CAP = KR_SPMM_CAP;             // nonzeros staged in shared memory per multi-row tile
constexpr int SPMM_MAX_ROWS = KR_SPMM_MAX_ROWS;   // rows per tile
constexpr int SPMM_LONG_ROW = 1024;   // rows at least this long are processed by a whole CTA
// Stored entries up to which a CSR (4-12 B per entry) and a few n-vectors stay L2-resident: there the one-CTA paths
// (pair_small_kernel, the single-CTA power iterations of leading_vector_dev and normest_dev) replace launch-bound loops.
constexpr int64_t CSR_L2_RESIDENT_NNZ = 400000;

struct CsrDev {
    int64_t n = 0, nnz = 0;
    DevBuf<int> row_ptr, col, row_order, row_pos;
    DevBuf<double> val;
    DevBuf<RowTile> tiles;
    DevBuf<int> dl_tile_begin, dl_rowlocal, dl_pos, dl_col;
    DevBuf<double> dl_val;
    int dl_count = 0;
    std::vector<RowTile> tiles_host;          // host copies for locating an edited row's tile
    std::vector<int> row_pos_host;
    int ntiles = 0;
    bool pattern_only = false;
    double uval = 1.0;
    CsrDevView view() const {
        CsrDevView v;
        v.n = (int)n;
        v.ntiles = ntiles;
        v.row_ptr = row_ptr.p;
        v.col = col.p;
        v.val = pattern_only ? nullptr : val.p;
        v.uval = uval;
        v.row_order = row_order.p;
        v.row_pos = row_pos.p;
        v.tiles = tiles.p;
        const bool dl = dl_count > 0;
        v.dl_tile_begin = dl ? dl_tile_begin.p : nullptr;
        v.dl_rowlocal = dl ? dl_rowlocal.p : nullptr;
        v.dl_pos = dl ? dl_pos.p : nullptr;
        v.dl_col = dl ? dl_col.p : nullptr;
        v.dl_val = dl ? dl_val.p : nullptr;
        v.dl_count = dl_count;
        return v;
    }
};

inline CsrHost transpose(const CsrHost& A) {
    CsrHost T;
    T.n = A.n;
    const int64_t nnz = A.row_ptr[A.n];
    T.row_ptr.assign(A.n + 1, 0);
    T.col.resize(nnz);
    T.val.resize(nnz);
    for (int64_t p = 0; p < nnz; ++p) T.row_ptr[A.col[p] + 1]++;
    for (int64_t i = 0; i < A.n; ++i) T.row_ptr[i + 1] += T.row_ptr[i];
    std::vector<int64_t> next(T.row_ptr.begin(), T.row_ptr.end() - 1);
    for (int64_t i = 0; i < A.n; ++i)
        for (int64_t p = A.row_ptr[i]; p < A.row_ptr[i + 1]; ++p) {
            int64_t q = next[A.col[p]]++;
            T.col[q] = (int32_t)i;
            T.val[q] = A.val[p];
        }
    return T;
}

// Rows must have sorted, duplicate-free columns for the symmetry comparison to be exact.
inline void canonicalize(CsrHost& A) {
    const int64_t n = A.n;
    int sorted = 1;
#pragma omp parallel for reduction(&& : sorted) schedule(static)
    for (int64_t i = 0; i < n; ++i)
        for (int64_t p = A.row_ptr[i] + 1; p < A.row_ptr[i + 1]; ++p)
            sorted = sorted && (A.col[p - 1] < A.col[p]);
    if (sorted) return;
    CsrHost T = transpose(A);      // two transposes = stable counting sort by column
    A = transpose(T);
    // merge duplicates (sum, as MATLAB's sparse() does)
    std::vector<int64_t> rp(n + 1, 0);
    int64_t w = 0;
    for (int64_t i = 0; i < n; ++i) {
        int64_t begin = w;
        for (int64_t p = A.row_ptr[i]; p < A.row_ptr[i + 1]; ++p) {
            if (w > begin && A.col[w - 1] == A.col[p]) A.val[w - 1] += A.val[p];
            else { A.col[w] = A.col[p]; A.val[w] = A.val[p]; ++w; }
        }
        rp[i + 1] = w;
    }
    A.row_ptr = rp;
    A.col.resize(w);
    A.val.resize(w);
}

// Host-side layout of the device CSR (everything upload_csr ships): rows in stored (length-sorted) order.
struct PreparedCsr {
    int64_t n = 0, nnz = 0;
    bool uniform = false;
    double uval = 1.0;
    std::vector<int> srp, order;
    std::vector<int32_t> scol;
    std::vector<double> sval;
    std::vector<RowTile> tiles;
};

inline int lane_class_of(int len) {
    return len >= SPMM_LONG_ROW ? 6 : len >= 256 ? 3 : len >= 64 ? 2 : len >= 16 ? 1 : 0;
}

// Pure host work (no CUDA calls): value uniformity, the stable decreasing-length row order (a counting sort,
// O(n + max length)), the re-packed index / value arrays (OpenMP over rows) and the tile list.
inline PreparedCsr prepare_csr(const CsrHost& H) {
    PreparedCsr P;
    const int64_t n = H.n, nnz = H.row_ptr[n];
    if (n >= (int64_t(1) << 31) - 64 || nnz >= (int64_t(1) << 31) - 64)
        fail(KR_ERR_UNSUPPORTED, "matrix too large for 32-bit device indices (n=%lld nnz=%lld)",
             (long long)n, (long long)nnz);
    P.n = n;
    P.nnz = nnz;
    int uniform = nnz > 0;
    const double v0 = nnz > 0 ? H.val[0] : 1.0;
#pragma omp parallel for reduction(&& : uniform) schedule(static)
    for (int64_t p = 0; p < nnz; ++p) uniform = uniform && (H.val[p] == v0);
    P.uniform = uniform != 0;
    P.uval = P.uniform ? v0 : 1.0;
    // ---- stored order: decreasing length, stable in the row index
    int maxlen = 0;
    for (int64_t i = 0; i < n; ++i) maxlen = std::max(maxlen, (int)(H.row_ptr[i + 1] - H.row_ptr[i]));
    std::vector<int64_t> start((size_t)maxlen + 2, 0);
    for (int64_t i = 0; i < n; ++i) start[(size_t)(maxlen - (int)(H.row_ptr[i + 1] - H.row_ptr[i])) + 1]++;
    for (size_t b = 1; b < start.size(); ++b) start[b] += start[b - 1];
    P.order.resize(n);
    for (int64_t i = 0; i < n; ++i) P.order[(size_t)start[(size_t)(maxlen - (int)(H.row_ptr[i + 1] - H.row_ptr[i]))]++] = (int)i;
    P.srp.assign(n + 1, 0);
    for (int64_t s = 0; s < n; ++s) {
        const int r = P.order[s];
        P.srp[s + 1] = P.srp[s] + (int)(H.row_ptr[r + 1] - H.row_ptr[r]);
    }
    P.scol.resize((size_t)std::max<int64_t>(nnz, 1));
    P.sval.resize(P.uniform ? 1 : (size_t)std::max<int64_t>(nnz, 1));
#pragma omp parallel for schedule(dynamic, 4096)
    for (int64_t s = 0; s < n; ++s) {
        const int r = P.order[s];
        std::copy(H.col.begin() + H.row_ptr[r], H.col.begin() + H.row_ptr[r + 1], P.scol.begin() + P.srp[s]);
        if (!P.uniform) std::copy(H.val.begin() + H.row_ptr[r], H.val.begin() + H.row_ptr[r + 1], P.sval.begin() + P.srp[s]);
    }
    // ---- tiles: runs of one lane class, nonzeros <= SPMM_CAP, rows <= SPMM_MAX_ROWS; long rows alone
    int64_t i = 0;
    while (i < n) {
        const int cls = lane_class_of(P.srp[i + 1] - P.srp[i]);
        int64_t j = i + 1;
        if (cls != 6) {
            int64_t acc = P.srp[i + 1] - P.srp[i];
            while (j < n && j - i < SPMM_MAX_ROWS) {
                const int len = P.srp[j + 1] - P.srp[j];
                if (lane_class_of(len) != cls || acc + len > SPMM_CAP) break;
                acc += len;
                ++j;
            }
        }
        P.tiles.push_back(RowTile{(int)i, (int)(j - i), cls, 0});
        i = j;
    }
    return P;
}

inline void upload_csr(kr_ctx* ctx, const CsrHost& H, CsrDev& D) {
    const PreparedCsr P = prepare_csr(H);
    const int64_t n = P.n, nnz = P.nnz;
    D.n = n;
    D.nnz = nnz;
    D.pattern_only = P.uniform;
    D.uval = P.uval;
    D.row_ptr.reset(ctx, n + 1);
    D.row_ptr.upload(P.srp.data(), n + 1);
    D.col.reset(ctx, std::max<int64_t>(nnz, 1));
    if (nnz) D.col.upload(P.scol.data(), nnz);
    if (!P.uniform) {
        D.val.reset(ctx, std::max<int64_t>(nnz, 1));
        if (nnz) D.val.upload(P.sval.data(), nnz);
    } else {
        D.val.free();
    }
    D.ntiles = (int)P.tiles.size();
    D.row_order.reset(ctx, std::max<int64_t>(n, 1));
    if (n) D.row_order.upload(P.order.data(), n);
    std::vector<int> pos((size_t)std::max<int64_t>(n, 1), 0);
    for (int64_t s = 0; s < n; ++s) pos[(size_t)P.order[(size_t)s]] = (int)s;
    D.row_pos.reset(ctx, std::max<int64_t>(n, 1));
    if (n) D.row_pos.upload(pos.data(), n);
    D.tiles_host = P.tiles;
    D.row_pos_host = pos;
    D.dl_count = 0;
    D.tiles.reset(ctx, std::max<size_t>(P.tiles.size(), 1));
    if (!P.tiles.empty()) D.tiles.upload(P.tiles.data(), P.tiles.size());
    KR_CUDA(cudaStreamSynchronize(ctx->stream));   // host staging vectors die here
}

}  // namespace kr

struct kr_matrix {
    kr_ctx* ctx = nullptr;
    kr::CsrHost host;          // kept for kr_matrix_set_edges and host-side glue (the STORED matrix: pending edits not applied)
    std::map<std::pair<int64_t, int64_t>, double> pending;    // (row, col) -> new value - stored value (both triangles)
    kr::CsrDev dev;            // A
    kr::CsrDev devT;           // A' (only when !symmetric)
    bool symmetric = true;
    bool nonnegative = true;
    double trace = 0.0;
    double norm1 = 0.0;        // max column abs sum
    // replicas of this matrix on other GPUs of the same process (kr_matrix_replicate): each owns its context
    std::vector<kr_matrix*> peers;
    bool is_peer = false;
    const kr::CsrDev& T() const { return symmetric ? dev : devT; }
};

namespace kr {

// keep_symmetric: the caller guarantees the edit preserved symmetry (kr_matrix_set_edges writes both
// triangles), so the O(nnz) transpose + comparison is skipped and ||A||_1 is the max row abs-sum.
// A == A' for a canonical (sorted, duplicate-free) CSR without building the transpose: walking the rows in
// ascending order, the entries (j, i) of row j are met in ascending i, so a per-row cursor finds the partner of
// every stored (i, j, v) in O(1) - the counting-sort transpose without its output arrays.
inline bool is_symmetric_csr(const CsrHost& H) {
    const int64_t n = H.n;
    std::vector<int64_t> cur(H.row_ptr.begin(), H.row_ptr.end() - 1);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t p = H.row_ptr[i]; p < H.row_ptr[i + 1]; ++p) {
            const int32_t j = H.col[p];
            const int64_t q = cur[j];
            if (q >= H.row_ptr[j + 1] || H.col[q] != (int32_t)i || H.val[q] != H.val[p]) return false;
            cur[j] = q + 1;
        }
    return true;    // every row's cursor consumed exactly its entries (counts match because all nnz partners were found)
}

inline void analyse_and_upload(kr_matrix* M, bool keep_symmetric = false) {
    CsrHost& H = M->host;
    canonicalize(H);
    const int64_t n = H.n;
    CsrHost T;
    if (!(keep_symmetric && M->symmetric)) {
        M->symmetric = is_symmetric_csr(H);
        if (!M->symmetric) T = transpose(H);
    }
    int nonneg = 1;
    double tr = 0.0, norm1 = 0.0;
    const CsrHost& C = M->symmetric ? H : T;       // column abs-sums of A = row abs-sums of A'
    // the trace feeds expmv's shift mu = trace / n: summed sequentially in row order (diagonal entry by binary
    // search) so that it does not depend on the thread count
    for (int64_t i = 0; i < n; ++i) {
        const int32_t* b = H.col.data() + H.row_ptr[i];
        const int32_t* e = H.col.data() + H.row_ptr[i + 1];
        const int32_t* q = std::lower_bound(b, e, (int32_t)i);
        if (q != e && *q == (int32_t)i) tr += H.val[(size_t)(q - H.col.data())];
    }
#pragma omp parallel for reduction(&& : nonneg) reduction(max : norm1) schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        for (int64_t p = H.row_ptr[i]; p < H.row_ptr[i + 1]; ++p)
            if (H.val[p] < 0) nonneg = 0;
        double sabs = 0;
        for (int64_t p = C.row_ptr[i]; p < C.row_ptr[i + 1]; ++p) sabs += std::abs(C.val[p]);
        norm1 = std::max(norm1, sabs);
    }
    M->nonnegative = nonneg != 0;
    M->trace = tr;
    M->norm1 = norm1;
    upload_csr(M->ctx, H, M->dev);
    if (!M->symmetric) upload_csr(M->ctx, T, M->devT);
    else { M->devT = CsrDev(); }
}

// stored value of A(i, j) in the host CSR (0 when absent)
inline double host_entry(const CsrHost& H, int64_t i, int64_t j) {
    const int32_t* b = H.col.data() + H.row_ptr[i];
    const int32_t* e = H.col.data() + H.row_ptr[i + 1];
    const int32_t* q = std::lower_bound(b, e, (int32_t)j);
    return (q != e && *q == (int32_t)j) ? H.val[(size_t)(q - H.col.data())] : 0.0;
}

constexpr size_t KR_MAX_PENDING = 8192;      // beyond this many delta entries the CSR is re-built

// ship the pending delta entries to the device (a few hundred bytes + one int per tile)
inline void upload_pending(kr_matrix* M) {
    kr_ctx* ctx = M->ctx;
    CsrDev& D = M->dev;
    struct Ent { int pos, col; double val; };
    std::vector<Ent> ents;
    ents.reserve(M->pending.size());
    for (auto& kv : M->pending)
        if (kv.second != 0.0) ents.push_back(Ent{D.row_pos_host[(size_t)kv.first.first], (int)kv.first.second, kv.second});
    std::sort(ents.begin(), ents.end(), [](const Ent& a, const Ent& b) { return a.pos != b.pos ? a.pos < b.pos : a.col < b.col; });
    D.dl_count = (int)ents.size();
    if (ents.empty()) return;
    const int nt = D.ntiles;
    std::vector<int> tb((size_t)nt + 1, 0), rl(ents.size()), ps(ents.size()), cl(ents.size());
    std::vector<double> vl(ents.size());
    size_t t = 0;
    for (size_t e = 0; e < ents.size(); ++e) {
        while (t + 1 < D.tiles_host.size() && D.tiles_host[t + 1].start <= ents[e].pos) ++t;
        tb[t + 1] += 1;
        rl[e] = ents[e].pos - D.tiles_host[t].start;
        ps[e] = ents[e].pos;
        cl[e] = ents[e].col;
        vl[e] = ents[e].val;
    }
    for (int q = 0; q < nt; ++q) tb[(size_t)q + 1] += tb[(size_t)q];
    if (D.dl_tile_begin.count < tb.size()) D.dl_tile_begin.reset(ctx, tb.size());
    if (D.dl_rowlocal.count < ents.size()) {
        const size_t cap = std::max<size_t>(256, 2 * ents.size());
        D.dl_rowlocal.reset(ctx, cap);
        D.dl_pos.reset(ctx, cap);
        D.dl_col.reset(ctx, cap);
        D.dl_val.reset(ctx, cap);
    }
    D.dl_tile_begin.upload(tb.data(), tb.size());
    D.dl_rowlocal.upload(rl.data(), rl.size());
    D.dl_pos.upload(ps.data(), ps.size());
    D.dl_col.upload(cl.data(), cl.size());
    D.dl_val.upload(vl.data(), vl.size());
    KR_CUDA(cudaStreamSynchronize(ctx->stream));      // host staging vectors die here (a few KB)
}

// fold the pending edits into the stored CSR (host rebuild + re-analysis + upload): every entry point that reads
// the CSR outside the SpMM / candidate-seed kernels calls this first; the greedy loop itself never does.
inline void flush_pending(kr_matrix* M) {
    if (M->pending.empty()) return;
    CsrHost& H = M->host;
    const int64_t n = H.n;
    std::map<int64_t, std::map<int32_t, double>> edits;
    for (auto& kv : M->pending) edits[kv.first.first][(int32_t)kv.first.second] = kv.second;
    std::map<int64_t, std::vector<std::pair<int32_t, double>>> rebuilt;
    for (auto& ed : edits) {
        const int64_t i = ed.first;
        std::map<int32_t, double> row;
        for (int64_t p = H.row_ptr[i]; p < H.row_ptr[i + 1]; ++p) row[H.col[p]] = H.val[p];
        for (auto& kv : ed.second) row[kv.first] += kv.second;               // stored + delta = new value
        auto& out = rebuilt[i];
        for (auto& kv : row)
            if (kv.second != 0.0) out.emplace_back(kv.first, kv.second);     // MATLAB sparse assignment of 0 removes the entry
    }
    CsrHost N;
    N.n = n;
    N.row_ptr.assign(n + 1, 0);
    {
        auto it = rebuilt.begin();
        for (int64_t i = 0; i < n; ++i) {
            int64_t len = H.row_ptr[i + 1] - H.row_ptr[i];
            if (it != rebuilt.end() && it->first == i) { len = (int64_t)it->second.size(); ++it; }
            N.row_ptr[i + 1] = N.row_ptr[i] + len;
        }
    }
    N.col.resize((size_t)N.row_ptr[n]);
    N.val.resize((size_t)N.row_ptr[n]);
#pragma omp parallel for schedule(dynamic, 4096)
    for (int64_t i = 0; i < n; ++i) {
        auto it = rebuilt.find(i);
        if (it == rebuilt.end()) {
            std::copy(H.col.begin() + H.row_ptr[i], H.col.begin() + H.row_ptr[i + 1], N.col.begin() + N.row_ptr[i]);
            std::copy(H.val.begin() + H.row_ptr[i], H.val.begin() + H.row_ptr[i + 1], N.val.begin() + N.row_ptr[i]);
        } else {
            int64_t w = N.row_ptr[i];
            for (auto& kv : it->second) { N.col[(size_t)w] = kv.first; N.val[(size_t)w] = kv.second; ++w; }
        }
    }
    H = std::move(N);
    M->pending.clear();
    analyse_and_upload(M, /*keep_symmetric=*/true);
}
inline void materialize(const kr_matrix* M) { flush_pending(const_cast<kr_matrix*>(M)); }

}  // namespace kr

