// spmm.cuh - CSR x dense-block product over k-wide fp64 blocks, with fused epilogues.
//
// Dense blocks on the device are PANEL-MAJOR: the k columns are cut into panels of PW columns
// (PW = 16 by default: 128 B = one cache line per row; PW = 8 also builds and passes the tests);
// panel p is a contiguous row-major n x PW array.  Element (i, c) lives at
// base[(c / PW) * n * PW + i * PW + (c % PW)].  A nonzero A(r, c) therefore gathers ONE row-tile of X
// per panel: LPT = PW/2 lanes x one 128-bit load, one L1 wavefront.  blockIdx.y (slow index) walks the
// panels so that one panel of X at a time competes for L2 with the streaming CSR arrays.
//
// Scheduling: one CTA (8 warps) per RowTile (csr.cuh).  The CTA first streams the tile's row
// pointers / row numbers / column indices (and values) into shared memory with coalesced loads, so
// the only dependent global loads left are the X gathers; inside a tile every row gets L = 4/8/16/32
// lanes and every lane issues U (4 or 8) independent 128-bit gathers before its first FMA.  Rows with
// >= 1024 nonzeros get a whole CTA.  Partial sums are folded with warp shuffles / shared memory in a fixed order, so results are
// bit-reproducible run to run (no float atomics).
//
// HBM roofline (DESIGN.md): algorithmic bytes per launch = 12*nnz + 4*(n+1) + 16*n*k.
#pragma once
#include "csr.cuh"

namespace kr {

#ifndef KR_PW
#define KR_PW 16
#endif
constexpr int PW = KR_PW;          // panel width (columns): 8 (64 B row-tiles) or 16 (128 B row-tiles)
constexpr int LPT = PW / 2;        // lanes per row-tile (one double2 per lane)
static_assert(PW == 8 || PW == 16, "panel width must be 8 or 16");
#ifndef KR_SPMM_THREADS
#define KR_SPMM_THREADS 256
#endif
constexpr int SPMM_THREADS = KR_SPMM_THREADS;  // warps per SpMM CTA = SPMM_THREADS / 32
constexpr int COL_WARPS = 8;                   // the streaming per-column kernels always use 256 threads
constexpr int SPMM_WARPS = SPMM_THREADS / 32;
#ifndef KR_SPMM_MIN_CTAS
#define KR_SPMM_MIN_CTAS 4
#endif
constexpr int SPMM_MIN_CTAS = KR_SPMM_MIN_CTAS;   // resident CTAs per SM the register allocation is bounded for

struct PanelBlock {                // non-owning view of a panel-major block
    double* p;
    int64_t n;
    int cols;                      // logical columns
    int panels;                    // ceil(cols / 8)
    __host__ __device__ double* panel(int q) const { return p + (int64_t)q * n * PW; }
};

// A lane of the SpMM handles CPL consecutive columns of a row-tile with ONE load:
//   CPL = 2: 128-bit gathers, 8 lanes per row-tile (the candidate-pair epilogue: one candidate per lane)
//   CPL = 4: 256-bit gathers (LDG.E.256), 4 lanes per row-tile (EpiPlain, EpiDot, EpiTaylor) - half the load /
//            address / index instructions per byte; the sustained SLQ pass is power-capped, so instructions per byte matter.
template <int CPL>
struct Vec {
    double v[CPL];
};
template <int CPL>
__device__ __forceinline__ Vec<CPL> vzero() {
    Vec<CPL> r;
#pragma unroll
    for (int i = 0; i < CPL; ++i) r.v[i] = 0.0;
    return r;
}
template <int CPL>
__device__ __forceinline__ Vec<CPL> ld_x(const double* p);          // gathered operand: keep in L1/L2
template <>
__device__ __forceinline__ Vec<2> ld_x<2>(const double* p) {
    const double2 t = __ldg(reinterpret_cast<const double2*>(p));
    Vec<2> r;
    r.v[0] = t.x; r.v[1] = t.y;
    return r;
}
template <>
__device__ __forceinline__ Vec<4> ld_x<4>(const double* p) {
    Vec<4> r;
    asm("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];"
        : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
    return r;
}
// int8 sign panels (dense.cuh): the 4 signs of a lane's columns are one 32-bit word
__device__ __forceinline__ Vec<4> signs_to_vec(unsigned w) {
    Vec<4> r;
#pragma unroll
    for (int i = 0; i < 4; ++i) r.v[i] = (double)(signed char)(w >> (8 * i));
    return r;
}
template <int CPL>
__device__ __forceinline__ Vec<CPL> ld_xv(const double* p) { return ld_x<CPL>(p); }
template <int CPL>
__device__ __forceinline__ Vec<CPL> ld_xv(const signed char* p) {
    static_assert(CPL == 4, "sign gathers use 4 columns per lane");
    return signs_to_vec(__ldg(reinterpret_cast<const unsigned*>(p)));
}
__device__ __forceinline__ Vec<4> ld_row(const double* p) {           // row-local operand (plain cached load)           // row-local operand (plain cached load)
    Vec<4> r;
    asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];"
                 : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
    return r;
}
__device__ __forceinline__ Vec<4> ld_row(const signed char* p) {
    return signs_to_vec(*reinterpret_cast<const unsigned*>(p));
}
__device__ __forceinline__ void st_row(double* p, const Vec<4>& a) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a.v[0]), "d"(a.v[1]), "d"(a.v[2]), "d"(a.v[3]) : "memory");
}
__device__ __forceinline__ void st_stream(double* p, const Vec<4>& a) {
    asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a.v[0]), "d"(a.v[1]), "d"(a.v[2]), "d"(a.v[3]) : "memory");
}
// L2 prefetch of a row-tile of X that a later round will gather: the demand gathers are latency-bound
// (every lane already holds U row-tiles in flight in registers) and 39 % of them miss L2 because one
// panel of X is as large as L2; a prefetch holds no register, so the DRAM part of the latency is paid
// KR_SPMM_PF rounds ahead of the demand load (measured: 7.6 -> 6.6 ms per k=512 SpMM, DESIGN.md section 5).
// Only the 128-bit lanes prefetch: with 256-bit lanes the kernel runs into the L2 slice throughput cap and the
// extra requests cost more than they hide (6.79 ms with, 6.48 ms without; profiles/r02b_spmm_variants.jsonl).
#ifndef KR_SPMM_PF
#define KR_SPMM_PF 1
#endif
__device__ __forceinline__ void prefetch_x(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
__device__ __forceinline__ void prefetch_l1(const void* p) {
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ int ld_stream(const int* p) { return __ldcs(p); }
__device__ __forceinline__ double ld_stream(const double* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(double* p, double2 v) {
    __stcs(reinterpret_cast<double2*>(p), v);
}

// Sum NV per-thread values over all threads of the CTA that share (lane % LP), deterministically,
// and hand the totals to lanes 0..LP-1 of warp 0.  smem: WARPS * LP * NV doubles.
template <int NV, int WARPS = COL_WARPS, int LP = LPT>
__device__ __forceinline__ void cta_reduce_by_sub(double (&v)[NV], double* smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = v[i];
#pragma unroll
        for (int off = LP; off < 32; off <<= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
        v[i] = x;
    }
    if (lane < LP) {
#pragma unroll
        for (int i = 0; i < NV; ++i) smem[(warp * LP + lane) * NV + i] = v[i];
    }
    __syncthreads();
    if (warp == 0 && lane < LP) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            double s = 0.0;
            for (int w = 0; w < WARPS; ++w) s += smem[(w * LP + lane) * NV + i];
            v[i] = s;
        }
    }
}

// ------------------------------------------------------------------------------- epilogues
// An epilogue sees, for one (row, CPL columns) slice, the finished dot products y and may read other
// row-local operands.  finish() runs once per CTA.  `sub` = the lane's slice index inside the row-tile
// (columns sub*CPL .. sub*CPL + CPL - 1 of the panel).

// Y = alpha * (A*X - mu*X)
struct EpiPlain {
    static constexpr int CPL = 4;
    double* __restrict__ Y;        // panel base
    const double* __restrict__ X;  // panel base (for the shift term)
    double alpha, mu;
    __device__ __forceinline__ void init(int q, int64_t stride) {
        Y += q * stride;
        X += q * stride;
    }
    // Row-local operands: the 4 x 32-byte gathers in flight need the registers, so pre() only pulls the line
    // towards the SM and row() loads it afterwards.
    Vec<CPL> xr;
    __device__ __forceinline__ void pre(int r, int sub) {
        if (mu != 0.0 && sub == 0) prefetch_l1(X + (int64_t)r * PW);
    }
    __device__ __forceinline__ void row(int r, int sub, Vec<CPL> y, unsigned) {
        if (mu != 0.0) xr = ld_row(X + (int64_t)r * PW + sub * CPL);
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
            if (mu != 0.0) y.v[i] -= mu * xr.v[i];
            y.v[i] *= alpha;
        }
        st_stream(Y + (int64_t)r * PW + sub * CPL, y);
    }
    __device__ __forceinline__ void finish(int, int, double*) {}
};

// Y = A*X and partial[tile][col] = sum_rows X(r,col) * Y(r,col)      (Lanczos alpha, SLQ path)
// XT: element type of X (double, or signed char for an int8 sign panel of +-1 probes);
// STORE = false: the last Lanczos step, whose Y no update reads (only the dot is kept).
template <class XT, bool STORE>
struct EpiDotT {
    static constexpr int CPL = 4;
    double* __restrict__ Y;
    const XT* __restrict__ X;
    double* __restrict__ partial;  // [ntiles][panels*PW]
    int total_cols;                // panels * PW
    double acc[CPL];
    __device__ __forceinline__ void init(int q, int64_t stride) {
        Y += q * stride;
        X += q * stride;
#pragma unroll
        for (int i = 0; i < CPL; ++i) acc[i] = 0.0;
    }
    Vec<CPL> xr;
    __device__ __forceinline__ void pre(int r, int sub) {
        if (sub == 0) prefetch_l1(X + (int64_t)r * PW);
    }
    __device__ __forceinline__ void row(int r, int sub, Vec<CPL> y, unsigned) {
        xr = ld_row(X + (int64_t)r * PW + sub * CPL);      // (a non-volatile load here: no gain, profiles/r02aj_*)
#pragma unroll
        for (int i = 0; i < CPL; ++i) acc[i] += xr.v[i] * y.v[i];
        if (STORE) st_stream(Y + (int64_t)r * PW + sub * CPL, y);
    }
    __device__ __forceinline__ void finish(int tile, int panel, double* smem) {
        cta_reduce_by_sub<CPL, SPMM_WARPS, PW / CPL>(acc, smem);
        if (threadIdx.x < PW / CPL) {
            double* o = partial + (int64_t)tile * total_cols + panel * PW + threadIdx.x * CPL;
#pragma unroll
            for (int i = 0; i < CPL; ++i) o[i] = acc[i];
        }
    }
};

using EpiDot = EpiDotT<double, true>;

// Candidate pairs (columns 2c, 2c+1): Y = A*C and raw Gram blocks P'Y, C'Y (2x2 each)
// partial[tile][cand][8] = {P'Y (row-major 2x2), C'Y (row-major 2x2)}
struct EpiGram2 {
    static constexpr int CPL = 2;
    double* __restrict__ Y;
    const double* __restrict__ P;  // previous block panel base (may be nullptr at step 1)
    const double* __restrict__ C;  // current block panel base (== X)
    double* __restrict__ partial;  // [ntiles][ncand_padded][8]
    int ncand;                     // panels * LPT
    double acc[8];
    __device__ __forceinline__ void init(int q, int64_t stride) {
        Y += q * stride;
        C += q * stride;
        if (P) P += q * stride;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.0;
    }
    // the row operands are pulled towards the SM before the gathers and loaded after them: holding them in
    // registers across the gather rounds (8 accumulators + 8 row-tiles in flight) spills at the 64-register cap
    __device__ __forceinline__ void pre(int r, int sub) {
        if (sub == 0) {
            prefetch_l1(C + (int64_t)r * PW);
            if (P) prefetch_l1(P + (int64_t)r * PW);
        }
    }
    __device__ __forceinline__ void row(int r, int sub, Vec<2> yv, unsigned) {
        const int64_t o = (int64_t)r * PW + sub * 2;
        const double2 y = make_double2(yv.v[0], yv.v[1]);
        const double2 c = *reinterpret_cast<const double2*>(C + o);
        if (P) {
            const double2 p = *reinterpret_cast<const double2*>(P + o);
            acc[0] += p.x * y.x; acc[1] += p.x * y.y;
            acc[2] += p.y * y.x; acc[3] += p.y * y.y;
        }
        acc[4] += c.x * y.x; acc[5] += c.x * y.y;
        acc[6] += c.y * y.x; acc[7] += c.y * y.y;
        st_stream(Y + o, y);
    }
    __device__ __forceinline__ void finish(int tile, int panel, double* smem) {
        cta_reduce_by_sub<8, SPMM_WARPS>(acc, smem);
        if (threadIdx.x < LPT) {
            double* o = partial + ((int64_t)tile * ncand + panel * LPT + threadIdx.x) * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = acc[i];
        }
    }
};

// Device-side control block of one expmv call (expmv.cuh): the early-termination test of
// functions/expmv.m:83 is evaluated on the device so that a whole call is enqueued without host syncs.
struct TaylorCtl {
    double c1;                         // ||b||_inf of the previous term
    double c2, nf;                     // last ||b'||_inf, ||f||_inf (diagnostics)
    int done;                          // early-termination flag of the current stage
    int mv;                            // products actually computed
    unsigned long long mb_bits, mf_bits;   // running maxima (bit patterns of non-negative doubles)
    unsigned int ticket;               // CTAs that have finished the current term
};

__device__ __forceinline__ void taylor_decide(TaylorCtl* ctl, double c2, double nf, int full_term, double tol) {
    ctl->mv += 1;
    ctl->c2 = c2;
    ctl->nf = nf;
    if (!full_term) {
        if (ctl->c1 + c2 <= tol * nf) ctl->done = 1;
        else ctl->c1 = c2;
    }
}

// expmv Taylor term (functions/expmv.m:77-80): b' = coef*(A*b - mu*b); f += b'.  The matrix inf-norms
// (max over rows of the abs-sum over ALL columns) are needed for the termination test:
//  * one panel (q <= PW, the mc_trace case): row sums are complete inside the CTA; maxima go through
//    atomicMax on the bit patterns (max of non-negative doubles is order independent, hence still
//    deterministic) and the LAST CTA to finish evaluates the test - one launch per Taylor term;
//  * several panels: rowabs_b[panel][r] / rowabs_f[panel][r] are written and reduced by
//    taylor_norms_ctl_kernel (expmv.cuh) - two launches per term.
// Every launch returns immediately once *done != 0.
struct EpiTaylor {
    static constexpr int CPL = 4;
    double* __restrict__ Bn;       // output b' panel
    const double* __restrict__ Bo; // input b panel (== X)
    double* __restrict__ F;        // f panel (read-modify-write)
    double* __restrict__ rab;      // rowabs of b' for this panel [n]   (multi-panel mode)
    double* __restrict__ raf;      // rowabs of f  for this panel [n]
    double coef, mu;
    TaylorCtl* ctl;                // non-null: single-panel fused control
    int total_ctas, full_term;
    double tol;
    double mb, mf;
    __device__ __forceinline__ void init(int q, int64_t stride) {
        Bn += q * stride;
        Bo += q * stride;
        F += q * stride;
        if (!ctl) {
            rab += q * (stride / PW);
            raf += q * (stride / PW);
        }
        mb = mf = 0.0;
    }
    Vec<CPL> xr, fr;
    __device__ __forceinline__ void pre(int r, int sub) {
        if (sub == 0) {
            if (mu != 0.0) prefetch_l1(Bo + (int64_t)r * PW);
            prefetch_l1(F + (int64_t)r * PW);
        }
    }
    __device__ __forceinline__ void row(int r, int sub, Vec<CPL> y, unsigned m) {
        const int64_t o = (int64_t)r * PW + sub * CPL;
        if (mu != 0.0) xr = ld_row(Bo + o);
        fr = ld_row(F + o);
        Vec<CPL> f = fr;
        double ab = 0.0, af = 0.0;
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
            if (mu != 0.0) y.v[i] -= mu * xr.v[i];
            y.v[i] *= coef;
            f.v[i] += y.v[i];
            ab += fabs(y.v[i]);
            af += fabs(f.v[i]);
        }
        st_row(F + o, f);
        st_stream(Bn + o, y);
        // the slot-0 lanes of a row hold its PW columns: fold over sub.  m = ballot of the lanes that
        // entered the epilogue (the subs of a row always enter together).
#pragma unroll
        for (int off = 1; off < PW / CPL; off <<= 1) {
            ab += __shfl_xor_sync(m, ab, off);
            af += __shfl_xor_sync(m, af, off);
        }
        if (ctl) {
            mb = fmax(mb, ab);
            mf = fmax(mf, af);
        } else if (sub == 0) {
            rab[r] = ab;
            raf[r] = af;
        }
    }
    __device__ __forceinline__ void finish(int, int, double* smem) {
        if (!ctl) return;
        // CTA maxima -> global maxima -> last CTA decides
        double a = mb, b = mf;
        for (int off = 16; off; off >>= 1) {
            a = fmax(a, __shfl_xor_sync(0xffffffffu, a, off));
            b = fmax(b, __shfl_xor_sync(0xffffffffu, b, off));
        }
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) { smem[2 * warp] = a; smem[2 * warp + 1] = b; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < SPMM_WARPS; ++w) { a = fmax(a, smem[2 * w]); b = fmax(b, smem[2 * w + 1]); }
            atomicMax(&ctl->mb_bits, (unsigned long long)__double_as_longlong(a));
            atomicMax(&ctl->mf_bits, (unsigned long long)__double_as_longlong(b));
            __threadfence();
            const unsigned t = atomicAdd(&ctl->ticket, 1u);
            if (t == (unsigned)total_ctas - 1u) {
                __threadfence();
                const double c2 = __longlong_as_double((long long)atomicAdd(&ctl->mb_bits, 0ull));
                const double nf = __longlong_as_double((long long)atomicAdd(&ctl->mf_bits, 0ull));
                taylor_decide(ctl, c2, nf, full_term, tol);
                ctl->mb_bits = 0ull;
                ctl->mf_bits = 0ull;
                ctl->ticket = 0u;
                __threadfence();
            }
        }
    }
};

// ------------------------------------------------------------------------------- kernel
// dynamic shared memory carve-up (bytes): col | rp | rid | [val]
constexpr size_t SPMM_SMEM_PATTERN = SPMM_CAP * sizeof(int) + (SPMM_MAX_ROWS + 1 + SPMM_MAX_ROWS + 3) * sizeof(int);
constexpr size_t SPMM_SMEM_VALUED = SPMM_SMEM_PATTERN + SPMM_CAP * sizeof(double);

// U independent gathers of one lane, issued back to back before the first FMA.  PRED = false: the caller
// guarantees that all U nonzeros exist (no per-gather predicate, no zero-fill); PRED = true: the row's last,
// partial round (no index / X traffic past the row end).
template <bool HAS_VAL, int U, int CPL, bool PRED>
__device__ __forceinline__ void gather_block(int p, int p_end, int stride, const int* __restrict__ scol,
                                             const double* __restrict__ sval, const double* __restrict__ xs,
                                             Vec<CPL>& acc0, Vec<CPL>& acc1) {
    Vec<CPL> x[U];
    double v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int q = p + u * stride;
        if (PRED) {
            x[u] = vzero<CPL>();
            v[u] = 1.0;
        }
        if (!PRED || q < p_end) {
            x[u] = ld_x<CPL>(xs + (int64_t)scol[q] * PW);
            if (HAS_VAL) v[u] = sval[q];
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
            const bool second = (u & 1) && CPL == 2;      // two accumulator sets only where registers allow
            if (HAS_VAL) {
                if (second) acc1.v[i] = fma(v[u], x[u].v[i], acc1.v[i]);
                else acc0.v[i] = fma(v[u], x[u].v[i], acc0.v[i]);
            } else {
                if (second) acc1.v[i] += x[u].v[i];
                else acc0.v[i] += x[u].v[i];
            }
        }
    }
}

// One lane's share of a row: nonzeros p_first, p_first+stride, ... < p_end (tile-relative, indices in
// shared memory).  Full rounds of U independent gathers run without any per-gather predicate; the row's
// last partial round is ONE predicated round (splitting it into 4 + 2 + 1 unpredicated gathers costs a full
// L2 latency per piece - measured 7.1 vs 6.6 ms per k = 512 SpMM, profiles/r02a_spmm_variants.jsonl).  A
// cp.async ring that parks the in-flight data in shared memory instead of registers is SLOWER here
// (profiles/r01_d_*).
template <bool HAS_VAL, int U, int CPL>
__device__ __forceinline__ Vec<CPL> gather_accumulate(int p_first, int p_end, int stride, const int* __restrict__ scol,
                                                      const double* __restrict__ sval, const double* __restrict__ xs,
                                                      const double* __restrict__ xpanel, int pf_sub) {
    Vec<CPL> acc0 = vzero<CPL>(), acc1 = vzero<CPL>();
    int p = p_first;
    for (; p + (U - 1) * stride < p_end; p += U * stride) {
#if KR_SPMM_PF > 0
        if (CPL == 2) {   // lane `pf_sub` of the group prefetches slot u = pf_sub of the round KR_SPMM_PF ahead
            const int qpf = p + (KR_SPMM_PF * U + pf_sub) * stride;
            if (pf_sub < U && qpf < p_end) prefetch_x(xpanel + (int64_t)scol[qpf] * PW);
        }
#endif
        gather_block<HAS_VAL, U, CPL, false>(p, p_end, stride, scol, sval, xs, acc0, acc1);
    }
    if (p < p_end) gather_block<HAS_VAL, U, CPL, true>(p, p_end, stride, scol, sval, xs, acc0, acc1);
    if (CPL == 2) {
#pragma unroll
        for (int i = 0; i < CPL; ++i) acc0.v[i] += acc1.v[i];
    }
    return acc0;
}

// Sign flavour of the gathers (XT = signed char: an int8 panel of +-1 probes, step 0 of the SLQ pass): one 32-bit
// load of 4 signs per lane and nonzero, a 16 B row-tile instead of 128 B.  Pattern-only A sums the signs in integers
// (IDP4A), which is exact, so the result equals the fp64 path's sum of +-1.0 in any order.  Valued A turns the signs
// into +-1.0 and runs the fp64 path's fma chain in its order, zero-filled partial round included: bit-identical.
template <bool HAS_VAL, int U, bool PRED>
__device__ __forceinline__ void sign_gather_block(int p, int p_end, int stride, const int* __restrict__ scol,
                                                  const double* __restrict__ sval, const signed char* __restrict__ xs,
                                                  Vec<4>& accd, int (&acci)[4]) {
    unsigned w[U];
    double v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int q = p + u * stride;
        if (PRED) {
            w[u] = 0u;
            v[u] = 1.0;
        }
        if (!PRED || q < p_end) {
            w[u] = __ldg(reinterpret_cast<const unsigned*>(xs + (int64_t)scol[q] * PW));
            if (HAS_VAL) v[u] = sval[q];
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (HAS_VAL) {
            const Vec<4> x = signs_to_vec(w[u]);
#pragma unroll
            for (int i = 0; i < 4; ++i) accd.v[i] = fma(v[u], x.v[i], accd.v[i]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) acci[i] = __dp4a((int)w[u], 1 << (8 * i), acci[i]);
        }
    }
}
template <bool HAS_VAL, int U, int CPL>
__device__ __forceinline__ Vec<CPL> gather_accumulate(int p_first, int p_end, int stride, const int* __restrict__ scol,
                                                      const double* __restrict__ sval, const signed char* __restrict__ xs,
                                                      const signed char*, int) {
    static_assert(CPL == 4, "sign gathers use 4 columns per lane");
    Vec<4> accd = vzero<4>();
    int acci[4] = {0, 0, 0, 0};
    int p = p_first;
    for (; p + (U - 1) * stride < p_end; p += U * stride)
        sign_gather_block<HAS_VAL, U, false>(p, p_end, stride, scol, sval, xs, accd, acci);
    if (p < p_end) sign_gather_block<HAS_VAL, U, true>(p, p_end, stride, scol, sval, xs, accd, acci);
    if (!HAS_VAL) {
#pragma unroll
        for (int i = 0; i < 4; ++i) accd.v[i] = (double)acci[i];
    }
    return accd;
}

// Multi-row tile: indices are already staged in shared memory; every row gets L lanes.
template <int L, bool HAS_VAL, int U, bool DELTA, class Epi, class XT>
__device__ __forceinline__ void spmm_tile(const RowTile t, const int* __restrict__ srp, const int* __restrict__ srid,
                                          const int* __restrict__ scol, const double* __restrict__ sval,
                                          const XT* __restrict__ Xp, double uval, Epi& epi, const CsrDevView& A,
                                          int e0, int e1) {
    constexpr int CPL = Epi::CPL;
    constexpr int LP = PW / CPL;        // lanes per row-tile
    constexpr int S = L / LP;           // nonzero slots per row
    constexpr int RPW = 32 / L;         // rows per warp per pass
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LP;
    const int slot = (lane % L) / LP;
    const int rlocal = lane / L;
    const XT* xs = Xp + sub * CPL;
    for (int base = warp * RPW; base < t.count; base += SPMM_WARPS * RPW) {
        const int rr = base + rlocal;
        const bool valid = rr < t.count;
        int row = 0, p0 = 0, p1 = 0;
        if (valid) {
            row = srid[rr];
            p0 = srp[rr];
            p1 = srp[rr + 1];
        }
        const bool emit = valid && slot == 0;
        if (emit) epi.pre(row, sub);    // row-local operands: issue their loads before the gathers
#if KR_SPMM_PF > 0
        if (CPL == 2) {   // the row this lane group serves KR_SPMM_PF passes from now: prefetch its first KR_SPMM_PF rounds
            const int rn = rr + KR_SPMM_PF * SPMM_WARPS * RPW;
            if (rn < t.count) {
                const int q0 = srp[rn], q1 = srp[rn + 1];
#pragma unroll
                for (int k = 0; k < KR_SPMM_PF; ++k) {
                    const int q = q0 + slot + (k * U + sub) * S;
                    if (sub < U && q < q1) prefetch_x(Xp + (int64_t)scol[q] * PW);
                }
            }
        }
#endif
        Vec<CPL> acc = gather_accumulate<HAS_VAL, U, CPL>(p0 + slot, p1, S, scol, sval, xs, Xp, sub);
#pragma unroll
        for (int off = LP; off < L; off <<= 1) {
#pragma unroll
            for (int i = 0; i < CPL; ++i) acc.v[i] += __shfl_xor_sync(0xffffffffu, acc.v[i], off);
        }
        if (!HAS_VAL) {
#pragma unroll
            for (int i = 0; i < CPL; ++i) acc.v[i] *= uval;
        }
        if (DELTA && e1 > e0 && emit) {   // pending edge edits of this tile (kr_matrix_set_edges): y_row += delta * x_col
            for (int e = e0; e < e1; ++e)
                if (A.dl_rowlocal[e] == rr) {
                    const Vec<CPL> x = ld_xv<CPL>(xs + (int64_t)A.dl_col[e] * PW);
                    const double d = A.dl_val[e];
#pragma unroll
                    for (int i = 0; i < CPL; ++i) acc.v[i] = fma(d, x.v[i], acc.v[i]);
                }
        }
        const unsigned m = __ballot_sync(0xffffffffu, emit);
        if (emit) epi.row(row, sub, acc, m);
    }
}

// One work item = (tile, panel): the CTA stages the tile's indices, serves its rows for this panel and writes the
// epilogue's per-CTA partials.
template <class Epi, bool HAS_VAL, int U, bool DELTA, class XT>
__device__ __forceinline__ void spmm_item(const CsrDevView& A, const XT* __restrict__ X, const Epi& epi_proto,
                                          int64_t panel_stride, int tile, int panel, double* red, unsigned char* dyn_smem) {
    constexpr int CPL = Epi::CPL;
    constexpr int LP = PW / CPL;
    int* scol = reinterpret_cast<int*>(dyn_smem);
    int* srp = scol + SPMM_CAP;
    int* srid = srp + SPMM_MAX_ROWS + 1;
    double* sval = reinterpret_cast<double*>(dyn_smem + SPMM_SMEM_PATTERN);
    const RowTile t = A.tiles[tile];
    const int pb = __ldg(A.row_ptr + t.start);
    const int nz = __ldg(A.row_ptr + t.start + t.count) - pb;
    const bool long_row = t.lanes_log2 == 6;   // class 6: one row, whole CTA
    // pending edge edits (kr_matrix_set_edges) are a template flavour of their own: carrying the (empty) range through
    // the row loop costs the Lanczos flavour 0.7 ms per k = 512 launch (7.86 -> 7.17 ms, profiles/r02ah_*) - the
    // kernel sits at the 64-register cap and the two live values displace gathers in flight
    const int e0 = DELTA && A.dl_tile_begin ? A.dl_tile_begin[tile] : 0;
    const int e1 = DELTA && A.dl_tile_begin ? A.dl_tile_begin[tile + 1] : 0;
    Epi epi = epi_proto;
    epi.init(panel, panel_stride);
    const XT* Xp = X + (int64_t)panel * panel_stride;
    if (!long_row) {
        // stage the tile's row pointers, row numbers and column indices (coalesced streams)
        for (int i = threadIdx.x; i <= t.count; i += SPMM_THREADS) srp[i] = __ldg(A.row_ptr + t.start + i) - pb;
        for (int i = threadIdx.x; i < t.count; i += SPMM_THREADS) srid[i] = __ldg(A.row_order + t.start + i);
        for (int p = threadIdx.x; p < nz; p += SPMM_THREADS) scol[p] = ld_stream(A.col + pb + p);
        if (HAS_VAL)
            for (int p = threadIdx.x; p < nz; p += SPMM_THREADS) sval[p] = ld_stream(A.val + pb + p);
        __syncthreads();
        switch (t.lanes_log2) {          // slots per row = 1 << lanes_log2, lanes per row = LP << lanes_log2 (<= 32)
            case 0: spmm_tile<LP, HAS_VAL, U, DELTA>(t, srp, srid, scol, sval, Xp, A.uval, epi, A, e0, e1); break;
            case 1: spmm_tile<2 * LP, HAS_VAL, U, DELTA>(t, srp, srid, scol, sval, Xp, A.uval, epi, A, e0, e1); break;
            case 2: spmm_tile<(4 * LP > 32 ? 32 : 4 * LP), HAS_VAL, U, DELTA>(t, srp, srid, scol, sval, Xp, A.uval, epi, A, e0, e1); break;
            default: spmm_tile<(8 * LP > 32 ? 32 : 8 * LP), HAS_VAL, U, DELTA>(t, srp, srid, scol, sval, Xp, A.uval, epi, A, e0, e1); break;
        }
    } else {
        // one long row, whole CTA: stage the indices chunk by chunk, SPMM_THREADS / LP nonzero slots
        const int sub = threadIdx.x % LP, slot = threadIdx.x / LP;
        const int row = __ldg(A.row_order + t.start);
        const bool emit = threadIdx.x < LP;
        if (emit) epi.pre(row, sub);
        double v[CPL];
#pragma unroll
        for (int i = 0; i < CPL; ++i) v[i] = 0.0;
        for (int c0 = 0; c0 < nz; c0 += SPMM_CAP) {
            const int cn = min(SPMM_CAP, nz - c0);
            __syncthreads();
            for (int p = threadIdx.x; p < cn; p += SPMM_THREADS) scol[p] = ld_stream(A.col + pb + c0 + p);
            if (HAS_VAL)
                for (int p = threadIdx.x; p < cn; p += SPMM_THREADS) sval[p] = ld_stream(A.val + pb + c0 + p);
            __syncthreads();
            Vec<CPL> a = gather_accumulate<HAS_VAL, U, CPL>(slot, cn, SPMM_THREADS / LP, scol, sval, Xp + sub * CPL, Xp, sub);
#pragma unroll
            for (int i = 0; i < CPL; ++i) v[i] += a.v[i];
        }
        cta_reduce_by_sub<CPL, SPMM_WARPS, LP>(v, red);      // totals in threads 0..LP-1
        Vec<CPL> acc;
#pragma unroll
        for (int i = 0; i < CPL; ++i) acc.v[i] = HAS_VAL ? v[i] : v[i] * A.uval;
        if (DELTA && e1 > e0 && emit) {
            for (int e = e0; e < e1; ++e) {      // a long-row tile holds one row: every entry is its
                const Vec<CPL> x = ld_xv<CPL>(Xp + sub * CPL + (int64_t)A.dl_col[e] * PW);
                const double d = A.dl_val[e];
#pragma unroll
                for (int i = 0; i < CPL; ++i) acc.v[i] = fma(d, x.v[i], acc.v[i]);
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, emit);
        if (emit) epi.row(row, sub, acc, m);
        __syncthreads();                               // red[] is reused by epi.finish
    }
    epi.finish(tile, panel, red);
}

// grid = (ntiles, panels); X panel q at X + q*n*PW.  `done` (may be null): skip everything if set.
template <class Epi, bool HAS_VAL, int U, bool DELTA, class XT>
__global__ void __launch_bounds__(SPMM_THREADS, SPMM_MIN_CTAS)
spmm_kernel(CsrDevView A, const XT* __restrict__ X, Epi epi_proto, int64_t panel_stride,
            const int* __restrict__ done, const int* __restrict__ panel_active) {
    if (done && *done) return;
    const int panel = blockIdx.y;
    if (panel_active && !panel_active[panel]) return;   // every column of this panel has converged
    __shared__ double red[SPMM_WARPS * LPT * 8];
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    spmm_item<Epi, HAS_VAL, U, DELTA, XT>(A, X, epi_proto, panel_stride, (int)blockIdx.x, panel, red, dyn_smem);
}

// A persistent flavour (SMs x 4 CTAs walking the (panel, tile) items in order, no CTA launch / drain per item) was
// measured and removed: 9.35 ms against 6.40 ms per k = 512 launch (profiles/r02ag_spmm_variants.jsonl) - the
// hardware's dynamic CTA scheduler balances the very unequal tiles (a hub row against 1 024 short rows), a static
// round-robin does not, and the per-item CTA barrier stalls the warps that finish early.

// per-device one-time setup flag (cudaFuncSetAttribute applies to the current device's context)
inline bool first_use_on_device(bool (&flags)[64], int device) {
    if (device < 0 || device >= 64 || flags[device]) return false;
    flags[device] = true;
    return true;
}

template <class Epi, int U, class XT>
inline void launch_spmm_impl(kr_ctx* ctx, const CsrDev& A, const XT* X, int panels, const Epi& epi,
                             const int* done, const int* panel_active) {
    static bool attr_set[64] = {};              // one table per Epi instantiation
    if (first_use_on_device(attr_set, ctx->device)) {
        KR_CUDA(cudaFuncSetAttribute(spmm_kernel<Epi, false, U, false, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPMM_SMEM_PATTERN));
        KR_CUDA(cudaFuncSetAttribute(spmm_kernel<Epi, true, U, false, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPMM_SMEM_VALUED));
        KR_CUDA(cudaFuncSetAttribute(spmm_kernel<Epi, false, U, true, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPMM_SMEM_PATTERN));
        KR_CUDA(cudaFuncSetAttribute(spmm_kernel<Epi, true, U, true, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPMM_SMEM_VALUED));
    }
    const int64_t ps = (int64_t)A.n * PW;
    const dim3 grid((unsigned)A.ntiles, (unsigned)panels);
    if (A.dl_count > 0) {
        if (A.pattern_only) spmm_kernel<Epi, false, U, true, XT><<<grid, SPMM_THREADS, SPMM_SMEM_PATTERN, ctx->stream>>>(A.view(), X, epi, ps, done, panel_active);
        else spmm_kernel<Epi, true, U, true, XT><<<grid, SPMM_THREADS, SPMM_SMEM_VALUED, ctx->stream>>>(A.view(), X, epi, ps, done, panel_active);
    } else {
        if (A.pattern_only) spmm_kernel<Epi, false, U, false, XT><<<grid, SPMM_THREADS, SPMM_SMEM_PATTERN, ctx->stream>>>(A.view(), X, epi, ps, done, panel_active);
        else spmm_kernel<Epi, true, U, false, XT><<<grid, SPMM_THREADS, SPMM_SMEM_VALUED, ctx->stream>>>(A.view(), X, epi, ps, done, panel_active);
    }
}

// independent gathers per lane and round: U2 for the 128-bit lanes (CPL = 2), U4 for the 256-bit lanes (CPL = 4)
#ifndef KR_SPMM_U2
#define KR_SPMM_U2 8
#endif
#ifndef KR_SPMM_U4
#define KR_SPMM_U4 4
#endif

// Host-side launcher.  Epilogues carry panel-0 pointers; init() advances them to the CTA's panel.
template <class Epi, class XT>
inline void launch_spmm(kr_ctx* ctx, const CsrDev& A, const XT* X, int panels, const Epi& epi,
                        const int* done = nullptr, int logical_cols = -1, const int* panel_active = nullptr) {
    if (A.ntiles == 0 || panels == 0) return;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (ctx->timing) {
        ctx->timing_events(&e0, &e1);
        KR_CUDA(cudaEventRecord(e0, ctx->stream));
    }
    launch_spmm_impl<Epi, Epi::CPL == 4 ? KR_SPMM_U4 : KR_SPMM_U2, XT>(ctx, A, X, panels, epi, done, panel_active);
    check_launch(ctx, "spmm_kernel");
    if (ctx->timing) {
        KR_CUDA(cudaEventRecord(e1, ctx->stream));
        ctx->spmm_events.emplace_back(e0, e1);
    }
    ctx->counters[1] += 1;
    ctx->counters[2] += logical_cols >= 0 ? logical_cols : (int64_t)panels * PW;
}

}  // namespace kr
