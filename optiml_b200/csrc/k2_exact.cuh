// K2e: K2's product w = Q u, BIT FOR BIT, from the upper triangle of an exactly symmetric matrix -- device code (included
// by pg.cu only).  The default pass of one rank over a self-Gram K1 built (gram.cu puts the norm of the smaller index inside
// the Gaussian fma, so Q[s][t] == Q[t][s] exactly for every kernel).
//
// K2's tree for row j (matvec_seg_kernel): inside a column segment of MV_SEG columns, thread t of MV_NT runs ONE fma chain
// over the column pairs (2t + 2 MV_NT k, +1), k ascending, x before y; lane 0's xor butterfly joins the chains of a warp;
// the warp sums are added in warp order from 0.0; the segment partials are added in segment order.  By symmetry, chain t
// of row j over segment A holds the elements Q[a][j] for the 2 EX_KS rows a = c0(A) + 2t + 2 MV_NT k (+1) of A.  So:
//
//   work item (A, t, B >= A): the EX_ROWS rows of chain t in A, all columns of B, rows in ascending order
//     row side     every row gets K2's own chain over B (thread tid owns the columns K2's thread tid owns), the lane
//                  butterfly and the ordered warp sum: wpart[B][row], K2's bits
//     column side  (B > A) thread tid carries, for each of its 2 EX_KS columns j, the fma chain over the item's rows in
//                  order -- K2's chain t of row j over A -- and stores it to colchain[A][t][j]
//   diagonal blocks (B == A) are read in full, row side only: the chains of their rows cross the diagonal.  Blocks strictly
//   below the diagonal blocks are never read.
//   combine       per column j and segment A < seg(j): K2's lane butterfly and warp sum over colchain[A][.][j], then
//                  K2's group combine (segment order, w, the shares of u'w), so the vector kernels cannot tell the passes
//                  apart.
//
// The matrix streams through K2s's machinery (k2_symv.cuh): a thread-private cp.async ring and u at the thread's columns
// fetched once per item; the row sums of TR rows are reduced by symv_warp_rows, whose tree for every row is the plain
// xor butterfly's (each step adds the partial of lane l ^ o to the partial of lane l, the same pairs in the same order).
#pragma once
#include "k2_symv.cuh"

constexpr int EX_KS = MV_SEG / (2 * MV_NT);  // column pairs K2's thread visits in a full segment (16)
constexpr int EX_ROWS = 2 * EX_KS;           // rows of one chain (32)
static_assert(MV_SEG % (2 * MV_NT) == 0 && MV_SEG % MV_GROUP == 0, "segments must hold whole chains and 64-row groups");

#ifndef SVMB200_EXACT_TR
#define SVMB200_EXACT_TR 8       // rows whose sums a thread holds at a time
#endif
#ifndef SVMB200_EXACT_LB
#define SVMB200_EXACT_LB 8       // 128-bit copies per batch
#endif
#ifndef SVMB200_EXACT_STAGES
#define SVMB200_EXACT_STAGES 6   // batches in flight per thread (ring depth)
#endif
#ifndef SVMB200_EXACT_MINB
#define SVMB200_EXACT_MINB 1     // CTAs per SM the register budget is cut for
#endif

template <int TR_, int LB_, int STAGES_, int MINB_>
struct ExactShape {
    static constexpr int TR = TR_, LB = LB_, STAGES = STAGES_, MINB = MINB_;
    static constexpr int RING_BYTES = STAGES_ * LB_ * MV_NT * 16;
    static constexpr int NBATCH = EX_KS * TR_ / LB_;   // load batches per sub-block of TR rows
    static_assert((TR_ & (TR_ - 1)) == 0 && TR_ >= 2 && TR_ <= EX_ROWS, "TR: a power of two up to a chain's rows");
    static_assert(TR_ % LB_ == 0 && STAGES_ >= 2 && STAGES_ <= NBATCH, "batches must tile a sub-block");
};
using ExactDefault = ExactShape<SVMB200_EXACT_TR, SVMB200_EXACT_LB, SVMB200_EXACT_STAGES, SVMB200_EXACT_MINB>;

// offset of colchain[A] (MV_NT rows of ld - c1(A) columns each) in the scratch
__host__ __device__ __forceinline__ long long exact_colchain_off(int A, long long ld) {
    return (long long)MV_NT * ((long long)A * ld - (long long)MV_SEG * A * (A + 1) / 2);
}

struct ExactArgs {
    const double* Q;      // n x ld, exactly symmetric
    long long ld, n, nrows_pad;
    const double* u;      // ld entries, zero beyond n
    double* wpart;        // K2's segment partials [nseg][nrows_pad]
    double* colchain;     // column chains, exact_colchain_off
    const int2* pairs;    // (A, B) of every MV_NT consecutive items
    const int* done;
};

template <class S, bool COLS>
__device__ __forceinline__ void exact_item(const ExactArgs& a, const int A, const int B, const int t, const int rows,
                                           const double* ush, double (*wsum)[EX_ROWS], double2* ring) {
    constexpr int TR = S::TR, KS = EX_KS, LB = S::LB, BPC = TR / LB, NBATCH = S::NBATCH, ST = S::STAGES;
    const int tid = (int)threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long c0B = (long long)B * MV_SEG;
    const int widthB = (int)((c0B + MV_SEG < a.ld ? c0B + MV_SEG : a.ld) - c0B);
    const int nch = (widthB + 2 * MV_NT - 1) / (2 * MV_NT);   // chunks of the segment (a ragged last one: fewer)
    // the thread's columns in B, K2's: 2 tid + 2 MV_NT k; one beyond the segment reads the segment's first column against
    // u = 0 (an exact no-op: a chain that starts at +0.0 never holds -0.0)
    bool cok[KS];
    double2 ucs[KS], colacc[KS];
#pragma unroll
    for (int k = 0; k < KS; ++k) {
        cok[k] = k * 2 * MV_NT + 2 * tid < widthB;
        ucs[k] = cok[k] ? __ldg(reinterpret_cast<const double2*>(a.u + c0B + k * 2 * MV_NT + 2 * tid)) : make_double2(0.0, 0.0);
        colacc[k] = make_double2(0.0, 0.0);
    }
    // row i of the item is row c0(A) + 2t + 2 MV_NT (i / 2) + i % 2 of the matrix
    const double* __restrict__ qitem = a.Q + ((long long)A * MV_SEG + 2 * t) * a.ld + c0B + 2 * tid;
    const int nrb = (rows + TR - 1) / TR;
    double2* const myring = ring + tid;   // ring[slot][j][thread]

    auto issue = [&](const int rb, const int b, const int slot) {
        const int k = b / BPC, rbase = (b % BPC) * LB;
        if (rb < nrb && k < nch) {
            const int last = (rows - rb * TR < TR ? rows - rb * TR : TR) - 1;
            const int koff = cok[k] ? k * 2 * MV_NT : -2 * tid;   // column c0(B) of the row
#pragma unroll
            for (int j = 0; j < LB; ++j) {
                const int i = rb * TR + (rbase + j < last ? rbase + j : last);
                sy_cp_async16(myring + (slot * LB + j) * MV_NT, qitem + (long long)((i >> 1) * 2 * MV_NT + (i & 1)) * a.ld + koff);
            }
        }
        sy_cp_async_commit();
    };

#pragma unroll
    for (int b = 0; b < ST; ++b) issue(0, b, b);
    int slot = 0;
#pragma unroll 1
    for (int rb = 0; rb < nrb; ++rb) {
        double rowacc[TR];
#pragma unroll
        for (int r = 0; r < TR; ++r) rowacc[r] = 0.0;
#pragma unroll
        for (int b = 0; b < NBATCH; ++b) {
            sy_cp_async_wait<ST - 1>();
            const int k = b / BPC, rb0 = (b % BPC) * LB;
            if (k < nch) {  // uniform over the CTA
                const double2 uc = ucs[k];
#pragma unroll
                for (int j = 0; j < LB; ++j) {
                    const double2 v = myring[(slot * LB + j) * MV_NT];
                    rowacc[rb0 + j] = fma(v.x, uc.x, rowacc[rb0 + j]);
                    rowacc[rb0 + j] = fma(v.y, uc.y, rowacc[rb0 + j]);
                    if (COLS && rb * TR + rb0 + j < rows) {   // a re-read row past the item's last one adds nothing
                        const double ur = ush[rb * TR + rb0 + j];
                        colacc[k].x = fma(v.x, ur, colacc[k].x);
                        colacc[k].y = fma(v.y, ur, colacc[k].y);
                    }
                }
            }
            if (b + ST < NBATCH) issue(rb, b + ST, slot);
            else issue(rb + 1, b + ST - NBATCH, slot);
            slot = slot + 1 == ST ? 0 : slot + 1;
        }
        const double tot = symv_warp_rows<TR>(rowacc, lane);
        if (lane < TR) wsum[wid][rb * TR + lane] = tot;
    }
    sy_cp_async_wait<0>();
    __syncthreads();
    for (int i = tid; i < rows; i += MV_NT) {   // K2's warp sum: warps in order, from 0.0
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < MV_NT / 32; ++w) v += wsum[w][i];
        a.wpart[(size_t)B * a.nrows_pad + (long long)A * MV_SEG + 2 * t + (i >> 1) * 2 * MV_NT + (i & 1)] = v;
    }
    if (COLS) {
        const long long c1A = (long long)(A + 1) * MV_SEG;
        double* cc = a.colchain + exact_colchain_off(A, a.ld) + (long long)t * (a.ld - c1A) + (c0B - c1A) + 2 * tid;
#pragma unroll
        for (int k = 0; k < KS; ++k)
            if (cok[k]) *reinterpret_cast<double2*>(cc + k * 2 * MV_NT) = colacc[k];
    }
}

template <class S>
__global__ void __launch_bounds__(MV_NT, S::MINB) matvec_exact_tile_kernel(const ExactArgs a) {
    pdl_wait();               // u (and the done flag) come from the vector launch before this one
    pdl_launch_dependents();
    if (a.done != nullptr && *a.done) return;
#ifndef SVMB200_HOST_EMULATION
    extern __shared__ __align__(16) unsigned char ex_smem_raw[];
    double2* ring = reinterpret_cast<double2*>(ex_smem_raw);
#else
    double2* ring = reinterpret_cast<double2*>(emu::dynamic_smem());
#endif
    __shared__ double ush[EX_ROWS];
    __shared__ double wsum[MV_NT / 32][EX_ROWS];
    const int2 pr = a.pairs[blockIdx.x / MV_NT];
    const int t = (int)(blockIdx.x % MV_NT);
    const long long c0A = (long long)pr.x * MV_SEG;
    const long long widthA = (c0A + MV_SEG < a.ld ? c0A + MV_SEG : a.ld) - c0A;
    // rows of chain t that exist: inside A and below n (a prefix of the EX_ROWS)
    int rows = 0;
    for (int i = 0; i < EX_ROWS; ++i) {
        const long long off = 2 * t + (long long)(i >> 1) * 2 * MV_NT + (i & 1);
        if (off < widthA && c0A + off < a.n) rows = i + 1;
    }
    if (rows == 0) return;
    for (int i = (int)threadIdx.x; i < EX_ROWS; i += MV_NT)
        ush[i] = i < rows ? a.u[c0A + 2 * t + (i >> 1) * 2 * MV_NT + (i & 1)] : 0.0;
    __syncthreads();
    if (pr.y > pr.x) exact_item<S, true>(a, pr.x, pr.y, t, rows, ush, wsum, ring);
    else exact_item<S, false>(a, pr.x, pr.y, t, rows, ush, wsum, ring);
}

struct ExactCombineArgs {
    const double* wpart;
    const double* colchain;
    long long ld, nrows, nrows_pad;
    int nseg;
    const double* u_rows;   // u at the rows, or null
    double* w;
    double* denpart;        // one per 64-row group, or null
    const int* done;
};

// one CTA of MV_NT threads per 64-row group; thread (p, jj): chains of warps 2p, 2p + 1 for row jj of the group
__global__ void __launch_bounds__(MV_NT) matvec_exact_combine_kernel(const ExactCombineArgs a) {
    pdl_wait();
    pdl_launch_dependents();
    if (a.done != nullptr && *a.done) return;
    constexpr int NW = MV_NT / 32;
    static_assert(NW == 2 * (MV_NT / MV_GROUP), "each thread joins the chains of two warps");
    __shared__ double ws[NW][MV_GROUP];
    __shared__ double red[2];
    // the groups of the last segments have the most column chains to join: they go first
    const unsigned group = gridDim.x - 1u - blockIdx.x;
    const int jj = (int)threadIdx.x % MV_GROUP, p = (int)threadIdx.x / MV_GROUP;
    const long long j = (long long)group * MV_GROUP + jj;
    const int segj = (int)(((long long)group * MV_GROUP) / MV_SEG);   // uniform: a group lies inside one segment
    double v = 0.0;
    for (int A = 0; A < segj; ++A) {
        const long long c1A = (long long)(A + 1) * MV_SEG, L = a.ld - c1A;
        if (j < a.nrows) {
            const double* cc = a.colchain + exact_colchain_off(A, a.ld) + (j - c1A);
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                const int wsel = 2 * p + h;
                double c[32];
#pragma unroll
                for (int l = 0; l < 32; ++l) c[l] = __ldcg(cc + (size_t)(wsel * 32 + l) * L);
                // K2's xor butterfly as seen by lane 0: lane l adds lane l + o's partial to its own
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int l = 0; l < o; ++l) c[l] = c[l] + c[l + o];
                }
                ws[wsel][jj] = c[0];
            }
        }
        __syncthreads();
        if (p == 0 && j < a.nrows) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < NW; ++k) s += ws[k][jj];
            v += s;
        }
        __syncthreads();
    }
    // K2's group combine, from segment seg(j) on the partials the tile pass stored
    if (threadIdx.x < MV_GROUP) {
        double dv = 0.0;
        if (j < a.nrows) {
            for (int s = segj; s < a.nseg; ++s) v += __ldcg(&a.wpart[(size_t)s * a.nrows_pad + j]);
            a.w[j] = v;
            if (a.u_rows != nullptr) dv = __dmul_rn(a.u_rows[j], v);
        }
        if (a.denpart != nullptr) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) dv = __dadd_rn(dv, __shfl_xor_sync(0xffffffffu, dv, o));
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dv;
        }
    }
    if (a.denpart != nullptr) {
        __syncthreads();
        if (threadIdx.x == 0) a.denpart[group] = __dadd_rn(red[0], red[1]);
    }
}
