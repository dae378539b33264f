// K2: streaming FP64 matrix-vector product(s) over the resident matrix -- device code (included by pg.cu only).
//   matvec_seg_kernel            one vector operand per pass (the roofline kernel of a fit)
//   matvec_seg_multi_kernel<NB>  NB <= 4 operands per pass (problems that share the matrix: one-vs-rest, multi-target)
// Both can deliver their results straight into every rank's exchange arena (tagged 16-byte entries, ll_store/ll_load).
#pragma once
#include "common.cuh"
#include <math.h>

// ------------------------------------------------------------------------------------------ K2
// Work item = MV_R consecutive rows x one column segment of MV_SEG doubles.  Every thread keeps
// MV_R*MV_U independent 128-bit streaming loads in flight (L1 no-allocate: Q is touched once per
// pass); the vector operand comes through L1/L2.  Rows are grouped by MV_GROUP (64): the CTA that
// finishes a group last (one atomic ticket per group) adds the segment partials of its 64 rows in
// segment order, stores w and the group's share of u'w.  Segmenting keeps the grid at >= 20 waves
// even for a 1/8 row shard (tail effect) and every work item at 256 KB.
constexpr int MV_R = 4;
constexpr int MV_NT = 256;
constexpr int MV_U = 4;
// the segment width is a build-time knob for the host emulation only (small problems with several segments); the sm_100a
// build uses 8192
#ifndef SVMB200_MV_SEG
#define SVMB200_MV_SEG 8192
#endif
constexpr int MV_SEG = SVMB200_MV_SEG;
constexpr int MV_MINB = 3;
constexpr int MV_GROUP = 64;            // rows per group (one u'w share per group)
constexpr int ROW_ALIGN = MV_GROUP;     // row shards start on multiples of this, see svmb200_shard_rows
constexpr int MV_BPG = MV_GROUP / MV_R;  // row blocks per group

struct MatvecArgs {
    const double* Q;        // nrows x ld shard
    long long ld, nrows;
    const double* u;        // ld entries, zero beyond n
    double* w;              // nrows results
    double* wpart;          // nseg x nrows_pad segment partials
    long long nrows_pad;
    unsigned* tickets;      // one per group, zero on entry, zero again on exit
    const double* u_rows;   // u at this shard's rows (u + row0), or null
    double* denpart;        // one per group: sum over the group's rows of u_rows[r] * w[r], or null
    int nseg;
    const int* done;
    // fused exchange (nranks_x > 0): the group combiner stores w / u'w shares straight into every rank's
    // gathered buffer as self-validating 16-byte entries {lo32 | tag, hi32 | tag} (two single-copy-atomic
    // 8-byte words, tag = sequence number of the product): no fence, no flag, no counter -- the reader
    // spins on the entry it needs until both tags match (the "LL" idea of NCCL, widened to FP64)
    int nranks_x;
    unsigned tag;
    ulonglong2* peer_w[SVM_MAX_RANKS];           // this rank's slot in rank r's gathered buffer
    const int* fault;       // the context's sticky exchange-fault flag (see ll_load), or null
};

#ifndef SVMB200_HOST_EMULATION
__device__ __forceinline__ void ll_store(ulonglong2* p, double v, unsigned tag) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v), t = (unsigned long long)tag << 32;
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"((b & 0xffffffffull) | t), "l"((b >> 32) | t)
                 : "memory");
}
// Bounded spin: after 20 s without the entry (a peer died or fell out of step) the reader raises the context's fault
// flag and gives up.  The flag is sticky and context-fatal: every later wait -- of this thread, of the other threads, of
// the launches already enqueued behind this one -- sees it (first miss and every 1024 spins) and returns at once, K2 / K3
// return at entry, and the host turns it into SVMB200_ERR_STATE at its next poll: one 20 s time-out per failure, not one
// per missing entry.  The values computed after a fault are garbage and are never handed out.
__device__ __forceinline__ double ll_load(const ulonglong2* p, unsigned tag, int* fault) {
    unsigned long long w0, w1, t0 = 0, now = 0;
    for (unsigned spins = 0;; ++spins) {
        asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(p) : "memory");
        if ((unsigned)(w0 >> 32) == tag && (unsigned)(w1 >> 32) == tag) break;
        if ((spins & 1023u) == 0u) {
            if (*reinterpret_cast<volatile int*>(fault)) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 20000000000ull) {
                *reinterpret_cast<volatile int*>(fault) = 1;
                break;
            }
        }
    }
    return __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
}

__device__ __forceinline__ double2 ld_stream_f64x2(const double2* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
#else
// tests/cuda_emu compiles this file for the host (the kernels run thread by thread on fibers, ranks are host threads):
// same entry format, same wait-until-both-tags-match protocol, without the PTX
__device__ __forceinline__ void ll_store(ulonglong2* p, double v, unsigned tag) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v), t = (unsigned long long)tag << 32;
    __atomic_store_n(&p->x, (b & 0xffffffffull) | t, __ATOMIC_RELEASE);
    __atomic_store_n(&p->y, (b >> 32) | t, __ATOMIC_RELEASE);
}
__device__ __forceinline__ double ll_load(const ulonglong2* p, unsigned tag, int* fault) {
    unsigned long long w0, w1;
    for (unsigned long long spins = 0;; ++spins) {
        w0 = __atomic_load_n(&p->x, __ATOMIC_ACQUIRE);
        w1 = __atomic_load_n(&p->y, __ATOMIC_ACQUIRE);
        if ((unsigned)(w0 >> 32) == tag && (unsigned)(w1 >> 32) == tag) break;
        if ((spins & 1023u) == 0u && __atomic_load_n(fault, __ATOMIC_ACQUIRE)) break;  // sticky: somebody already timed out
        if (emu::spin_wait(spins)) {  // yields the host thread; true after 20 s
            __atomic_store_n(fault, 1, __ATOMIC_RELEASE);
            break;
        }
    }
    return __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
}
__device__ __forceinline__ double2 ld_stream_f64x2(const double2* p) { return *p; }
#endif

__global__ void __launch_bounds__(MV_NT, MV_MINB) matvec_seg_kernel(const MatvecArgs a) {
    pdl_wait();               // u (and the done flag) come from the vector launch before this one
    pdl_launch_dependents();  // once every CTA of this grid has started, the vector launch may be scheduled behind it
    if (a.done != nullptr && *a.done) return;
    if (a.fault != nullptr && *a.fault) return;  // the exchange is broken: nothing downstream will be used
    constexpr int R = MV_R, NT = MV_NT, U = MV_U;
    const unsigned items_per_group = (unsigned)(MV_BPG * a.nseg);
    // Work items in launch order: all FULL column segments first, the short last segment (ld mod 8192 columns: 848 of
    // them at n = 50 000, a tenth of an item) at the end of the grid.  The grid's tail -- SMs that run out of work while
    // the last 256 KB items finish, ~half an item time, 2 % of a pass over a 1/8 shard -- is then filled with small
    // items.  Which CTA computes an item never changes a bit: partials are combined per group in segment order.
    const unsigned nbig = (a.ld % MV_SEG == 0 || a.nseg == 1) ? (unsigned)a.nseg : (unsigned)a.nseg - 1u;
    const unsigned ngroups = gridDim.x / items_per_group;
    const unsigned items_big = ngroups * (unsigned)MV_BPG * nbig;
    unsigned group, rb_in_group;
    int seg;
    if (blockIdx.x < items_big) {
        group = blockIdx.x / ((unsigned)MV_BPG * nbig);
        const unsigned within = blockIdx.x - group * ((unsigned)MV_BPG * nbig);
        rb_in_group = within / nbig;
        seg = (int)(within - rb_in_group * nbig);
    } else {
        const unsigned idx = blockIdx.x - items_big;
        group = idx / (unsigned)MV_BPG;
        rb_in_group = idx - group * (unsigned)MV_BPG;
        seg = a.nseg - 1;
    }
    const long long row_base = (long long)group * MV_GROUP + (long long)rb_in_group * R;
    __shared__ double red[NT / 32][R];
    __shared__ unsigned is_last;

    if (row_base < a.nrows) {
        const long long c0 = (long long)seg * MV_SEG;
        long long c1 = c0 + MV_SEG;
        if (c1 > a.ld) c1 = a.ld;
        const int nvec = (int)((c1 - c0) >> 1);
        const double2* __restrict__ u2 = reinterpret_cast<const double2*>(a.u + c0);
        const double2* rows[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            long long rr = row_base + r;
            if (rr >= a.nrows) rr = a.nrows - 1;  // clamp: read a valid row, result discarded below
            rows[r] = reinterpret_cast<const double2*>(a.Q + rr * a.ld + c0);
        }
        double acc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = 0.0;

        int c = threadIdx.x;
        for (; c + (U - 1) * NT < nvec; c += U * NT) {
            double2 qv[U][R];
            double2 uv[U];
#pragma unroll
            for (int j = 0; j < U; ++j) {
#pragma unroll
                for (int r = 0; r < R; ++r) qv[j][r] = ld_stream_f64x2(rows[r] + c + j * NT);
            }
#pragma unroll
            for (int j = 0; j < U; ++j) uv[j] = __ldg(u2 + c + j * NT);
#pragma unroll
            for (int j = 0; j < U; ++j) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    acc[r] = fma(qv[j][r].x, uv[j].x, acc[r]);
                    acc[r] = fma(qv[j][r].y, uv[j].y, acc[r]);
                }
            }
        }
        for (; c < nvec; c += NT) {
            double2 qv[R];
#pragma unroll
            for (int r = 0; r < R; ++r) qv[r] = ld_stream_f64x2(rows[r] + c);
            const double2 uv = __ldg(u2 + c);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                acc[r] = fma(qv[r].x, uv.x, acc[r]);
                acc[r] = fma(qv[r].y, uv.y, acc[r]);
            }
        }
        // warp butterfly, then fixed-order sum over warps
#pragma unroll
        for (int r = 0; r < R; ++r) {
            double v = acc[r];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            acc[r] = v;
        }
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        if (lane == 0) {
#pragma unroll
            for (int r = 0; r < R; ++r) red[wid][r] = acc[r];
        }
        __syncthreads();
        if (threadIdx.x < R && row_base + threadIdx.x < a.nrows) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < NT / 32; ++k) v += red[k][threadIdx.x];
            a.wpart[(size_t)seg * a.nrows_pad + row_base + threadIdx.x] = v;
        }
    }
    // ---- one ticket per group; the last arriver combines the group
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicInc(&a.tickets[group], items_per_group - 1) == items_per_group - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x < MV_GROUP) {
        const long long rr = (long long)group * MV_GROUP + threadIdx.x;
        double dv = 0.0;
        if (rr < a.nrows) {
            double v = 0.0;
            for (int s = 0; s < a.nseg; ++s) v += __ldcg(&a.wpart[(size_t)s * a.nrows_pad + rr]);
            if (a.nranks_x > 0) {
                for (int p = 0; p < a.nranks_x; ++p) ll_store(a.peer_w[p] + rr, v, a.tag);  // NVLink stores (one is local)
            } else {
                a.w[rr] = v;
            }
            if (a.u_rows != nullptr) dv = __dmul_rn(a.u_rows[rr], v);
        }
        if (a.denpart != nullptr) {
            // fixed tree over the 64 rows: butterfly inside each warp, then warp 0 + warp 1
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) dv = __dadd_rn(dv, __shfl_xor_sync(0xffffffffu, dv, o));
            if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = dv;
        }
    }
    if (a.denpart != nullptr) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const double tot = __dadd_rn(red[0][0], red[0][1]);
            if (a.nranks_x > 0) {
                const size_t off = (size_t)(a.denpart - a.w) + group;  // share slot relative to the w slot
                for (int p = 0; p < a.nranks_x; ++p) ll_store(a.peer_w[p] + off, tot, a.tag);
            } else {
                a.denpart[group] = tot;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ K2 x NB
// Several products against ONE pass over the matrix (SURVEY.md 8f-4: the binary problems of a one-vs-rest fit, or the
// targets of a multi-output regression, share the resident M): a work item streams its R x MV_SEG tile once and feeds
// NB accumulator sets.  Per row and per thread the columns are visited in the order of matvec_seg_kernel (c, c + NT,
// ... ; x then y), the warp / CTA / segment reductions are the same trees, so every w_b is BIT-IDENTICAL to the
// single-vector kernel's -- a batched fit reproduces the sequential fits exactly.  The vector operands (NB x 64 KB per
// item) come through L2: R rows amortise them, the ratio of L2 to HBM bytes is NB / R.
constexpr int MV_MULTI_MAX = 4;  // vectors per launch; larger batches are split into balanced launches

// shape knobs, overridable at build time (scripts/sweep_multi.py): any R that divides 64 and any U keep the results
// bit-identical, they only move the register budget and the L2 : HBM traffic ratio (NB / R)
#ifndef SVMB200_MULTI_R
#define SVMB200_MULTI_R 4
#endif
#ifndef SVMB200_MULTI_U
#define SVMB200_MULTI_U 2
#endif
#ifndef SVMB200_MULTI_MINB
#define SVMB200_MULTI_MINB 0
#endif
#ifndef SVMB200_MULTI_H
#define SVMB200_MULTI_H 1
#endif
template <int NB>
struct MultiCfg {
    static constexpr int R = SVMB200_MULTI_R;  // rows per work item
    static constexpr int U = SVMB200_MULTI_U;  // 128-bit loads in flight per row and thread
    // CTAs per SM the register budget is cut for
    static constexpr int MINB = SVMB200_MULTI_MINB > 0 ? SVMB200_MULTI_MINB : (NB <= 2 ? 3 : 2);
    // H groups of 256 threads per CTA, each with its own R rows of the same column segment: the vector operands the
    // groups read at about the same time are served once from L2 and H - 1 times from L1 (same results bit for bit)
    static constexpr int H = SVMB200_MULTI_H;
};

struct MatvecMultiArgs {
    const double* Q;
    long long ld, nrows, nrows_pad;
    double* wpart;      // [NB][nseg][nrows_pad]
    unsigned* tickets;
    int nseg;
    const double* u[MV_MULTI_MAX];       // ld entries each, zero beyond n
    double* w[MV_MULTI_MAX];             // nrows results each
    const double* u_rows[MV_MULTI_MAX];  // u at this shard's rows, or null
    double* denpart[MV_MULTI_MAX];       // one share of u'w per 64-row group, or null
    const int* done[MV_MULTI_MAX];       // problem b finished: its results are not stored (may be null)
    // fused exchange (nranks_x > 0), as in MatvecArgs: results of problem b go to peer_w[p] + b * xstride (+ row for
    // w, + share_off + group for the u'w share) in every rank's arena as tagged entries
    int nranks_x;
    unsigned tag;
    long long xstride, share_off;
    ulonglong2* peer_w[SVM_MAX_RANKS];
    const int* fault;   // the context's sticky exchange-fault flag, or null
};

template <int NB>
__global__ void __launch_bounds__(MV_NT * MultiCfg<NB>::H, MultiCfg<NB>::MINB) matvec_seg_multi_kernel(const MatvecMultiArgs a) {
    constexpr int R = MultiCfg<NB>::R, NT = MV_NT, U = MultiCfg<NB>::U, H = MultiCfg<NB>::H, BPG = MV_GROUP / (R * H);
    static_assert(NB >= 1 && NB <= MV_MULTI_MAX && NB * MV_GROUP <= NT * H && MV_GROUP % (R * H) == 0 && NT * H <= 1024,
                  "bad multi-vector shape");
    pdl_wait();
    pdl_launch_dependents();
    bool live[NB];
    bool any = false;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        live[b] = !(a.done[b] != nullptr && *a.done[b]);
        any = any || live[b];
    }
    if (!any) return;
    if (a.fault != nullptr && *a.fault) return;
    const int half = (int)threadIdx.x / NT;         // which group of 256 threads (whole warps)
    const int tid = (int)threadIdx.x - half * NT;   // the thread's index inside its group: the column it starts at
    const unsigned items_per_group = (unsigned)(BPG * a.nseg);
    const unsigned group = blockIdx.x / items_per_group;
    const unsigned within = blockIdx.x - group * items_per_group;
    const unsigned rb_in_group = within / (unsigned)a.nseg;
    const int seg = (int)(within - rb_in_group * (unsigned)a.nseg);
    const long long row_base = (long long)group * MV_GROUP + (long long)rb_in_group * (R * H) + (long long)half * R;
    const size_t pstride = (size_t)a.nseg * a.nrows_pad;  // wpart elements per problem
    __shared__ double red[H][NT / 32][NB][R];
    __shared__ double red2[NB][2];
    __shared__ unsigned is_last;
    const bool active = row_base < a.nrows;  // uniform inside a group of 256 threads

    if (active) {
        const long long c0 = (long long)seg * MV_SEG;
        long long c1 = c0 + MV_SEG;
        if (c1 > a.ld) c1 = a.ld;
        const int nvec = (int)((c1 - c0) >> 1);
        const double2* rows[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            long long rr = row_base + r;
            if (rr >= a.nrows) rr = a.nrows - 1;  // clamp: read a valid row, result discarded below
            rows[r] = reinterpret_cast<const double2*>(a.Q + rr * a.ld + c0);
        }
        double acc[NB][R];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
#pragma unroll
            for (int r = 0; r < R; ++r) acc[b][r] = 0.0;
        }
        int c = tid;
        for (; c + (U - 1) * NT < nvec; c += U * NT) {
            double2 qv[U][R];
#pragma unroll
            for (int j = 0; j < U; ++j) {
#pragma unroll
                for (int r = 0; r < R; ++r) qv[j][r] = ld_stream_f64x2(rows[r] + c + j * NT);
            }
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const double2* __restrict__ u2 = reinterpret_cast<const double2*>(a.u[b] + c0);
                double2 uv[U];
#pragma unroll
                for (int j = 0; j < U; ++j) uv[j] = __ldg(u2 + c + j * NT);
#pragma unroll
                for (int j = 0; j < U; ++j) {
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        acc[b][r] = fma(qv[j][r].x, uv[j].x, acc[b][r]);
                        acc[b][r] = fma(qv[j][r].y, uv[j].y, acc[b][r]);
                    }
                }
            }
        }
        for (; c < nvec; c += NT) {
            double2 qv[R];
#pragma unroll
            for (int r = 0; r < R; ++r) qv[r] = ld_stream_f64x2(rows[r] + c);
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const double2 uv = __ldg(reinterpret_cast<const double2*>(a.u[b] + c0) + c);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    acc[b][r] = fma(qv[r].x, uv.x, acc[b][r]);
                    acc[b][r] = fma(qv[r].y, uv.y, acc[b][r]);
                }
            }
        }
        // warp butterfly, then fixed-order sum over the group's warps (the trees of matvec_seg_kernel)
        const int lane = tid & 31, wid = tid >> 5;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                double v = acc[b][r];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) red[half][wid][b][r] = v;
            }
        }
    }
    __syncthreads();
    if (active && tid < NB * R) {
        const int b = tid / R, r = tid - b * R;
        if (row_base + r < a.nrows) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < NT / 32; ++k) v += red[half][k][b][r];
            a.wpart[(size_t)b * pstride + (size_t)seg * a.nrows_pad + row_base + r] = v;
        }
    }
    // ---- one ticket per group; the last arriver combines the group for every problem
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicInc(&a.tickets[group], items_per_group - 1) == items_per_group - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // thread t handles row (t % 64) of problem (t / 64): whole warps share a problem
    {
        const int b = (int)(threadIdx.x / MV_GROUP);
        const int t = (int)(threadIdx.x % MV_GROUP);
        double dv = 0.0;
        bool has_den = false;
#pragma unroll
        for (int bb = 0; bb < NB; ++bb) {  // static indexing of the per-problem pointer arrays
            if (bb != b) continue;
            has_den = a.denpart[bb] != nullptr;
            const long long rr = (long long)group * MV_GROUP + t;
            if (rr < a.nrows) {
                double v = 0.0;
                const double* wp = a.wpart + (size_t)bb * pstride + rr;
                for (int s = 0; s < a.nseg; ++s) v += __ldcg(wp + (size_t)s * a.nrows_pad);
                if (live[bb]) {
                    if (a.nranks_x > 0) {
                        for (int p = 0; p < a.nranks_x; ++p) ll_store(a.peer_w[p] + bb * a.xstride + rr, v, a.tag);
                    } else {
                        a.w[bb][rr] = v;
                    }
                }
                if (a.u_rows[bb] != nullptr) dv = __dmul_rn(a.u_rows[bb][rr], v);
            }
        }
        if (b < NB && has_den) {
            // fixed tree over the 64 rows: butterfly inside each warp, then the problem's two warps in order
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) dv = __dadd_rn(dv, __shfl_xor_sync(0xffffffffu, dv, o));
            if ((threadIdx.x & 31) == 0) red2[b][t >> 5] = dv;
        }
    }
    __syncthreads();
    if (threadIdx.x < NB) {
#pragma unroll
        for (int bb = 0; bb < NB; ++bb) {
            if (bb == (int)threadIdx.x && a.denpart[bb] != nullptr && live[bb]) {
                const double tot = __dadd_rn(red2[bb][0], red2[bb][1]);
                if (a.nranks_x > 0) {
                    for (int p = 0; p < a.nranks_x; ++p)
                        ll_store(a.peer_w[p] + bb * a.xstride + a.share_off + group, tot, a.tag);
                } else {
                    a.denpart[bb][group] = tot;
                }
            }
        }
    }
}
