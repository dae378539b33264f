// K11: SMO for the SVM dual with an unregularised intercept -- device code (included by pg.cu only).
//
//     min  a'Qa/2 + q'a   s.t.  y'a = 0,  0 <= a <= C          (libsvm's problem; y = label signs, or e = [1, -1] for SVR)
//
// libsvm's solver without shrinking (Fan, Chen & Lin 2005, working-set selection WSS2), one pair of variables per
// iteration:
//   i = argmax_{t in I_up} -y_t G_t  (= m),   j = argmin_{t in I_low, b_t > 0} -b_t^2 / a_t,   M = min_{t in I_low} -y_t G_t
//   b_t = m + y_t G_t,  a_t = Q_ii + Q_tt - 2 y_i y_t Q_it (TAU if <= 0);  ties go to the larger index (libsvm's >= / <=)
//   stop (optimal) when m - M < tol or no j exists; (stopped) at iter == max_iter
//   two-variable step with clipping, then  G_t += Q_it da_i + Q_jt da_j  for every t.
// An iteration needs two rows of Q (16 n bytes) and two arg-reductions over all variables: it is bound by latency, not by
// bandwidth -- the regime of the persistent PG loop (k_persistent.cuh).  So ONE cooperative launch runs many iterations:
//   CTA b owns the contiguous slice [b S, (b+1) S) of the variables; its alpha, G, sign, Q_tt, C and its part of row i
//   live in shared memory for the whole launch (Q_tt read once per launch from the diagonal).
//   phase 1  apply the previous step to the own G (Q_it from the cached row i, Q_jt streamed from row j); local
//            candidate for i -> partial slot
//   grid barrier
//   phase 2  (every CTA) reduce the partials to i and m; stream the own part of row i (cached for the next phase 1);
//            local candidate for j and local M -> partial slot
//   grid barrier
//   phase 3  (every CTA) reduce to j and M, stopping test (identical everywhere: all CTAs leave together), the step from
//            the published scalars and Q_ij; the owners of i and j write their alpha; CTA 0 records history and state.
// A published candidate carries every scalar another CTA needs (alpha, G, sign, Q_tt, C of the winner), so no CTA reads
// another's live alpha or G; the slots are double-buffered by iteration parity (as K8's partials).  The reductions are
// max / min under a total order (value, then index), so the result does not depend on arrival order: the solve is
// reproducible run to run.
// Q_st is always the element read from ROW s (Q[s][t]); the Gram matrix is not assumed to be bitwise symmetric.  Every
// operation of the step, of G's update and of the objective is an explicit _rn intrinsic (the library is built with
// --fmad=true): no contraction, so a NumPy restatement of the algorithm replays the whole trajectory bit for bit.
// Layouts: PLAIN, Q itself resident (SVC: y_s y_t K_st);  SVR, M = K resident (n x n) and Q_st = e_s e_t M[s mod n][t mod n].
//
// K12, the row source (template parameter ROWS).  SMO_ROWS_RESIDENT reads Q from HBM as above.  SMO_ROWS_COMPUTED reads
// no matrix: Q_st = sign_s sign_t k(x_{s mod n}, x_{t mod n}) (both layouts), the kernel value from X by kfn_value
// (kernel_fn.cuh), so a problem far larger than HBM runs.  A CTA only ever needs its own slice of row j (phase 1) and of
// row i (phase 2): it computes that slice, or reads it from a row cache in HBM --
//   `slots` rows of nvars doubles, keyed by the sample index (SVR rows s and s + n share a slot), unsigned values;
//   set-associative (sets x ways; every sample has its own slot when the cache holds all n rows), LRU within a set by
//   the stamp of the last use (2k for row j in phase 1 of iteration k, 2k + 1 for row i in phase 2);
//   every CTA keeps a private copy of the tags and stamps and updates it identically from the (i, j) sequence, and
//   reads and writes only its own slice of a slot: no inter-CTA traffic, no race.
// A value is the same whether it was cached or computed, so hits and misses never change a bit of the trajectory.
// Q_ij (phase 3) travels from j's owner, which holds Q_it for t = j in its part of row i, through a per-CTA slot
// published beside the j candidate.
//
// SMO_ROWS_SIGNED reads a shared, unsigned resident M (bias 0) and applies the sign row on read, as K12 does:
// Q_st = (sign_s == sign_t ? v : -v), v = M[s mod n][t mod n] (SVC: sign = the labels; SVR: sign = e, the SVR read above);
// the diagonal is read unsigned.  K1 signs a matrix by flipping the sign bit of fl(K + bias), the same operation, so a
// solve on the view is bit-identical to one on K1's signed Q, zeros included.  It is how the problems of one-vs-rest and
// multi-target fits share one M in HBM.
//
// K14, smo_batch_kernel: several problems on one shared M in ONE cooperative launch.  Problem b runs on its own contiguous
// range of CTAs with its own SmoArgs (state, candidate slots, histories) and its own grid barrier; the body below takes the
// CTA's index and grid size inside its problem instead of blockIdx.x / gridDim.x.  A solve does not depend on its grid
// (total-order reductions), so every problem follows the same bits whatever grid it is given, launch after launch.  The
// computed form stays single-problem: its per-CTA cache tags assume one problem owns the CTA's slice.
//
// Shrinking (libsvm's do_shrinking / be_shrunk / reconstruct_gradient; the SHRINK instantiations smo_shrink_kernel and
// smo_batch_shrink_kernel, the plain kernels are the SHRINK = false ones).  One active flag per variable (a bit per owned
// variable in shared memory, a byte per variable in HBM between launches: K14 changes slices between launches); held
// variables (ub = 0) are never active.  Selection, step and G update run over the active variables only: an inactive
// variable's G is not updated and its row entries are neither read nor computed.  l = the non-held variables, P = min(l,
// 1000); a counter that starts at P + 1 is decremented before the selection of every state, and at 0 (set back to P) the
// state is a shrink check:
//   phase 1 also carries the slice's min over the active I_low in `mlow`; after the barrier every CTA knows m and M;
//   the first time m - M <= 10 tol the solver reconstructs and reactivates everything (`unshrunk`);
//   every CTA deactivates its own variables at a bound that are only in I_low with -y_t G_t > m, or only in I_up with
//   -y_t G_t < M (free variables never), publishes a fresh i candidate (in the i slots of the other parity, free until
//   phase 1 of state k + 1) and its active count, and one more grid barrier follows.
// When the stopping test fires with inactive variables the solver reconstructs, reactivates everything, sets the counter
// to 1 and selects again at the same state (the history of state k is the evaluation that decided it); a max_iter stop
// reconstructs before G is written back.  Reconstruct: every CTA writes its alpha to HBM, grid barrier, then
// G_t = q_t + sum_{j ascending, alpha_j > 0} Q_jt alpha_j (one rounding per product and per sum) for its inactive, non-held
// t, with Q_jt read from row j (resident, signed) or computed by kfn_value; a computed-row CTA then clears its copy of the
// cache tags, so no cached row holds an entry skipped while its variable was inactive.  Every decision that adds a barrier
// (counter, m, M, gap, status, the grid's active count) is grid-uniform.  SmoShrink::on = 0 follows the plain bits.
#pragma once
#include "k_persistent.cuh"   // pk_grid_barrier
#include "kernel_fn.cuh"      // kfn_value

constexpr int SMO_NT = 256;
constexpr int SMO_ARRAYS = 6;        // doubles of shared memory per owned variable: alpha, G, sign, Q_tt, C, Q_it
constexpr double SMO_TAU = 1e-12;
constexpr int SMO_ROWS_RESIDENT = 0, SMO_ROWS_COMPUTED = 1, SMO_ROWS_SIGNED = 2;
constexpr int SMO_CACHE_WAYS = 8;
constexpr int SMO_ACT_WORDS = 148;   // shrinking: one bit per owned variable (pg.cu asserts the largest slice fits)
constexpr long long SMO_SHRINK_EVERY = 1000;

struct SmoCand {      // the winner of one CTA's slice (64 bytes)
    double key;       // i pass: -y_t G_t;  j pass: b_t^2 / a_t  (the larger wins, ties to the larger index)
    double idx;       // variable index (exact in a double), -1: no candidate
    double alpha, g, y, qd, c;
    double mlow;      // j pass: min of -y_t G_t over the slice's part of I_low (+inf if empty)
};

struct SmoArgs {
    const double* Q;        // resident matrix, n x ld
    long long ld, n, nvars;
    int svr;
    int slice;              // variables per CTA
    double *x, *g;          // alpha and G (nvars): read at the start of a launch, written back at its end
    const double *sgn, *ub; // sign vector and upper bounds (nvars)
    SmoCand* cand;          // [2 parities][2 passes][grid]
    unsigned* gbar;         // grid barrier (k_persistent.cuh)
    PGDeviceState* st;      // f, ng = gap, iter, done, status of the last evaluated state
    double *hist_f, *hist_gap;
    long long hist_cap;
    double tol;
    long long max_iter;
    long long k0;           // first state this launch evaluates
    long long niter;        // steps to take unless the stopping test fires first (states k0 .. k0 + niter are evaluated)
    // computed rows only
    KernelFn kf;
    double* qij;            // [2 parities][grid]: Q_it at t = the CTA's j candidate
    double* cache;          // slots x nvars, or null (no cache)
    int* tags;              // [grid][slots] sample index per slot (-1: empty)
    long long* stamps;      // [grid][slots] stamp of the last use
    long long sets, ways;
    unsigned long long* stats;  // hits, misses (CTA 0)
};

// shrinking: the grid-uniform state carried across launches (every CTA reads it at the start, CTA 0 writes it at the end)
struct SmoShrinkState {
    long long counter;          // decremented before the selection of every state: a check at 0
    long long unshrunk;         // the gap came within 10 tol once and everything was reactivated
    long long shrunk;           // some non-held variable is inactive
    long long prepared;         // the last state whose counter step ran: a launch that ends on its budget evaluates
                                // its last state, and the next launch evaluates it again without a second step
    long long checks, reconstructions;
    long long active;           // active variables after the last check
};

struct SmoShrink {
    const double* q;            // linear term (nvars): G of an inactive variable is rebuilt from it
    unsigned char* act;         // active flags (nvars): read at the start of a launch, written back at its end
    SmoShrinkState* st;
    long long l;                // variables that are not held (ub > 0)
    int on;                     // 0: no shrinking, the plain kernel's trajectory
};

// Q[s][t] as read from row s
__device__ __forceinline__ double smo_q(const SmoArgs& a, long long s, long long t) {
    if (!a.svr) return __ldg(a.Q + s * a.ld + t);
    const bool s_lo = s < a.n, t_lo = t < a.n;
    const double v = __ldg(a.Q + (s_lo ? s : s - a.n) * a.ld + (t_lo ? t : t - a.n));
    return s_lo == t_lo ? v : -v;
}

// SMO_ROWS_SIGNED: the unsigned M[s mod n][t mod n]
__device__ __forceinline__ double smo_m(const SmoArgs& a, long long s, long long t) {
    return __ldg(a.Q + (s < a.n ? s : s - a.n) * a.ld + (t < a.n ? t : t - a.n));
}

// SMO_ROWS_SIGNED: Q[s][t] from M and the signs of s and t
__device__ __forceinline__ double smo_q_signed(const SmoArgs& a, long long s, long long t, double ys, double yt) {
    const double v = smo_m(a, s, t);
    return ys == yt ? v : -v;
}

// thread 0 of a CTA: the slot of sample r in this CTA's copy of the cache tags (LRU victim on a miss), -1 without cache
__device__ __forceinline__ long long smo_cache_lookup(const SmoArgs& a, unsigned cta, long long r, long long stamp, int& hit) {
    hit = 0;
    long long slot = -1;
    if (a.sets > 0) {
        const long long slots = a.sets * a.ways, base = (r % a.sets) * a.ways;
        int* tags = a.tags + (size_t)cta * slots;
        long long* st = a.stamps + (size_t)cta * slots;
        // all ways are loaded before any is compared: independent loads, one round trip to L2 instead of `ways`
        int tg[SMO_CACHE_WAYS];
        long long sp[SMO_CACHE_WAYS];
#pragma unroll
        for (int w = 0; w < SMO_CACHE_WAYS; ++w) {
            tg[w] = w < a.ways ? tags[base + w] : -1;
            sp[w] = w < a.ways ? st[base + w] : 0;
        }
        long long oldest = 0;
#pragma unroll
        for (int w = 0; w < SMO_CACHE_WAYS; ++w) {
            if (w >= a.ways || hit) continue;
            if (tg[w] == (int)r) {
                slot = base + w;
                hit = 1;
            } else if (slot < 0 || sp[w] < oldest) {
                slot = base + w;
                oldest = sp[w];
            }
        }
        tags[slot] = (int)r;
        st[slot] = stamp;
    }
    if (cta == 0) a.stats[hit ? 0 : 1] += 1;
    return slot;
}

// unsigned K[r][t mod n] for the own variable t: from the cache slot on a hit, else from X (and into the slot)
__device__ __forceinline__ double smo_row_value(const SmoArgs& a, long long r, long long t, long long slot, int hit) {
    double* c = slot >= 0 ? a.cache + slot * a.nvars + t : nullptr;
    if (hit) return *c;
    const double v = kfn_value(a.kf, r, t < a.n ? t : t - a.n);
    if (c) *c = v;
    return v;
}

__device__ __forceinline__ bool smo_wins(double k, double i, double bk, double bi) { return k > bk || (k == bk && i > bi); }

// block-wide arg-max of (key, idx) and min of `low`; the result lands in thread 0
__device__ __forceinline__ void smo_block_reduce(double& key, double& idx, double& low, double (*red)[SMO_NT / 32]) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ok = __shfl_xor_sync(0xffffffffu, key, o), oi = __shfl_xor_sync(0xffffffffu, idx, o);
        const double ol = __shfl_xor_sync(0xffffffffu, low, o);
        if (smo_wins(ok, oi, key, idx)) {
            key = ok;
            idx = oi;
        }
        low = fmin(low, ol);
    }
    if (lane == 0) {
        red[0][wid] = key;
        red[1][wid] = idx;
        red[2][wid] = low;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < SMO_NT / 32; ++w) {
            if (smo_wins(red[0][w], red[1][w], key, idx)) {
                key = red[0][w];
                idx = red[1][w];
            }
            low = fmin(low, red[2][w]);
        }
    }
}

// reduce the grid's partial slots of one pass; thread 0 copies the winner's slot (the owner of the winning index: slices
// are contiguous, S variables each) to *out with mlow = the grid's minimum
__device__ __forceinline__ void smo_grid_reduce(const SmoCand* slots, unsigned grid, int S, double (*red)[SMO_NT / 32],
                                                SmoCand* out) {
    double key = -INFINITY, idx = -1.0, low = INFINITY;
    for (unsigned s = threadIdx.x; s < grid; s += SMO_NT) {
        const double k = __ldcg(&slots[s].key), i = __ldcg(&slots[s].idx), l = __ldcg(&slots[s].mlow);
        if (smo_wins(k, i, key, idx)) {
            key = k;
            idx = i;
        }
        low = fmin(low, l);
    }
    smo_block_reduce(key, idx, low, red);
    if (threadIdx.x == 0) {
        SmoCand w = {-INFINITY, -1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (idx >= 0.0) {
            const SmoCand* s = slots + (long long)idx / S;
            w.key = key;
            w.idx = idx;
            w.alpha = __ldcg(&s->alpha);
            w.g = __ldcg(&s->g);
            w.y = __ldcg(&s->y);
            w.qd = __ldcg(&s->qd);
            w.c = __ldcg(&s->c);
        }
        w.mlow = __dadd_rn(low, 0.0);   // -0 -> +0: fmin may return either zero
        *out = w;
    }
    __syncthreads();
}

__device__ __forceinline__ bool smo_is_active(const unsigned* act, int l) { return (act[l >> 5] >> (l & 31)) & 1u; }

// block-wide sum of v (exact for counts); the result is returned to every thread
__device__ __forceinline__ double smo_block_sum(double v, double (*red)[SMO_NT / 32]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();   // red may still be read by the previous reduction
    if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = v;
    __syncthreads();
    double sum = 0.0;
    for (int w = 0; w < SMO_NT / 32; ++w) sum += red[0][w];
    __syncthreads();
    return sum;
}

// shrinking: G_t = q_t + sum_{j ascending, alpha_j > 0} Q_jt alpha_j for the slice's inactive, non-held variables, which
// then become active (with every other non-held one).  Every CTA calls it (it holds a grid barrier).
template <int ROWS>
__device__ __forceinline__ void smo_reconstruct(const SmoArgs& a, const SmoShrink& s, const unsigned cta, const unsigned grid,
                                                const long long t0, const int len, unsigned* act, const double* s_alpha,
                                                double* s_g, const double* s_y, const double* s_c) {
    __shared__ double s_ya[SMO_NT];   // y_j alpha_j of one chunk of j (alpha_j >= 0: the sign is y_j where alpha_j > 0)
    const int tid = threadIdx.x, nwords = (len + 31) >> 5;
    for (int l = tid; l < len; l += SMO_NT) a.x[t0 + l] = s_alpha[l];
    pk_grid_barrier(a.gbar, grid);
    bool mine = false;   // this thread owns a variable to rebuild
    for (int l = tid; l < len; l += SMO_NT) {
        if (!smo_is_active(act, l) && s_c[l] > 0.0) {
            s_g[l] = __ldg(s.q + t0 + l);
            mine = true;
        }
    }
    for (long long j0 = 0; j0 < a.nvars; j0 += SMO_NT) {
        __syncthreads();
        const long long jt = j0 + tid;
        s_ya[tid] = jt < a.nvars ? __dmul_rn(__ldg(a.sgn + jt), __ldcg(a.x + jt)) : 0.0;
        __syncthreads();
        if (!mine) continue;
        const int cnt = a.nvars - j0 < SMO_NT ? (int)(a.nvars - j0) : SMO_NT;
        for (int b = 0; b < cnt; ++b) {
            const double v = s_ya[b];
            if (v == 0.0) continue;
            const long long j = j0 + b;
            const double aj = fabs(v), yj = v > 0.0 ? 1.0 : -1.0;
            for (int l = tid; l < len; l += SMO_NT) {
                if (smo_is_active(act, l) || !(s_c[l] > 0.0)) continue;
                const long long t = t0 + l;
                double qjt;
                if constexpr (ROWS == SMO_ROWS_COMPUTED) {
                    const double w = kfn_value(a.kf, j < a.n ? j : j - a.n, t < a.n ? t : t - a.n);
                    qjt = yj == s_y[l] ? w : -w;
                } else if constexpr (ROWS == SMO_ROWS_SIGNED) {
                    qjt = smo_q_signed(a, j, t, yj, s_y[l]);
                } else {
                    qjt = smo_q(a, j, t);
                }
                s_g[l] = __dadd_rn(s_g[l], __dmul_rn(qjt, aj));
            }
        }
    }
    __syncthreads();
    for (int w = tid; w < nwords; w += SMO_NT) {
        unsigned bits = 0u;
        for (int b = 0; b < 32 && 32 * w + b < len; ++b)
            if (s_c[32 * w + b] > 0.0) bits |= 1u << b;
        act[w] = bits;
    }
    if constexpr (ROWS == SMO_ROWS_COMPUTED) {
        // the CTA's copy of the tags, cleared identically everywhere: a cached row may lack the entries of variables
        // that were inactive when it was computed
        const long long slots = a.sets * a.ways;
        for (long long r = tid; r < slots; r += SMO_NT) {
            a.tags[(size_t)cta * slots + r] = -1;
            a.stamps[(size_t)cta * slots + r] = -1;
        }
    }
    __syncthreads();
}

// the solve of one problem by CTA `cta` of the `grid` CTAs that run it; SHRINK: with shrinking when s.on
template <int ROWS, bool SHRINK>
__device__ __forceinline__ void smo_solve(const SmoArgs& a, const SmoShrink& s, const unsigned cta, const unsigned grid) {
#ifndef SVMB200_HOST_EMULATION
    extern __shared__ __align__(16) unsigned char smo_smem_raw[];
    double* sm = reinterpret_cast<double*>(smo_smem_raw);
#else
    double* sm = reinterpret_cast<double*>(emu::dynamic_smem());
#endif
    __shared__ double red[3][SMO_NT / 32];
    __shared__ SmoCand win_i, win_j;
    __shared__ long long s_slot[2];   // computed rows: cache slot of row j (phase 1) and of row i (phase 2)
    __shared__ int s_hit[2];
    const int tid = threadIdx.x;
    const int S = a.slice;
    double *s_alpha = sm, *s_g = sm + S, *s_y = sm + 2 * S, *s_qd = sm + 3 * S, *s_c = sm + 4 * S, *s_qi = sm + 5 * S;
    const long long t0 = (long long)cta * S;
    const int len = t0 >= a.nvars ? 0 : (int)(a.nvars - t0 < S ? a.nvars - t0 : S);

    for (int l = tid; l < len; l += SMO_NT) {
        const long long t = t0 + l;
        s_alpha[l] = a.x[t];
        s_g[l] = a.g[t];
        s_y[l] = a.sgn[t];
        s_c[l] = a.ub[t];
        if constexpr (ROWS == SMO_ROWS_COMPUTED) {
            const long long tm = t < a.n ? t : t - a.n;
            s_qd[l] = kfn_value(a.kf, tm, tm);
        } else if constexpr (ROWS == SMO_ROWS_SIGNED) {
            s_qd[l] = smo_m(a, t, t);
        } else {
            s_qd[l] = smo_q(a, t, t);
        }
        s_qi[l] = 0.0;
    }
    double f = a.st->f;   // objective at state k0 (CTA 0 rewrites it only after the first grid barrier)
    // shrinking: the slice's active flags and the grid-uniform state (identical in every CTA)
    __shared__ unsigned s_act[SHRINK ? SMO_ACT_WORDS : 1];
    long long counter = 0, checks = 0, recons = 0, nact = 0, prepared = -1;
    bool unshrunk = false, shrunk = false, reselect = false;
    if constexpr (SHRINK) {
        for (int w = tid; w < (len + 31) >> 5; w += SMO_NT) {
            unsigned bits = 0u;
            for (int b = 0; b < 32 && 32 * w + b < len; ++b)
                if (!s.on || s.act[t0 + 32 * w + b]) bits |= 1u << b;
            s_act[w] = bits;
        }
        if (s.on) {
            counter = s.st->counter;
            unshrunk = s.st->unshrunk != 0;
            shrunk = s.st->shrunk != 0;
            prepared = s.st->prepared;
            checks = s.st->checks;
            recons = s.st->reconstructions;
            nact = s.st->active;
        }
    }
    __syncthreads();

    bool pending = false;          // a step whose G update phase 1 still has to apply
    long long pj = 0;
    double dai = 0.0, daj = 0.0;
    for (long long e = 0;; ++e) {
        const long long k = a.k0 + e;
        SmoCand* slots_i = a.cand + (size_t)((k & 1) * 2) * grid;
        SmoCand* slots_j = slots_i + grid;
        bool check = false;   // shrinking: this state is a shrink check
        if constexpr (SHRINK) {
            if (s.on && !reselect && k != prepared && --counter == 0) {
                counter = s.l < SMO_SHRINK_EVERY ? s.l : SMO_SHRINK_EVERY;
                check = true;
            }
            prepared = k;
            reselect = false;
        }
        // ================= phase 1: previous step on the own G, local candidate for i
        double key = -INFINITY, idx = -1.0, low = INFINITY;
        for (int l = tid; l < len; l += SMO_NT) {
            if constexpr (SHRINK) {
                if (!smo_is_active(s_act, l)) continue;
            }
            const long long t = t0 + l;
            double gt = s_g[l];
            if (pending) {
                double qjt;
                if constexpr (ROWS == SMO_ROWS_COMPUTED) {
                    const double v = smo_row_value(a, pj < a.n ? pj : pj - a.n, t, s_slot[0], s_hit[0]);
                    qjt = win_j.y == s_y[l] ? v : -v;
                } else if constexpr (ROWS == SMO_ROWS_SIGNED) {
                    qjt = smo_q_signed(a, pj, t, win_j.y, s_y[l]);
                } else {
                    qjt = smo_q(a, pj, t);
                }
                gt = __dadd_rn(gt, __dadd_rn(__dmul_rn(s_qi[l], dai), __dmul_rn(qjt, daj)));
                s_g[l] = gt;
            }
            const double y = s_y[l], al = s_alpha[l];
            const bool up = y > 0.0 ? al < s_c[l] : al > 0.0;
            const double v = -__dmul_rn(y, gt);
            if (up && v >= key) {   // own indices ascend: >= keeps the larger one on ties
                key = v;
                idx = (double)t;
            }
            if constexpr (SHRINK) {
                if (check && (y > 0.0 ? al > 0.0 : al < s_c[l])) low = fmin(low, v);
            }
        }
        smo_block_reduce(key, idx, low, red);
        if (tid == 0) {
            SmoCand c = {key, idx, 0.0, 0.0, 0.0, 0.0, 0.0, SHRINK ? low : INFINITY};
            if (idx >= 0.0) {
                const int l = (int)((long long)idx - t0);
                c.alpha = s_alpha[l];
                c.g = s_g[l];
                c.y = s_y[l];
                c.qd = s_qd[l];
                c.c = s_c[l];
            }
            slots_i[cta] = c;
        }
        pk_grid_barrier(a.gbar, grid);

        const SmoCand* src_i = slots_i;
        if constexpr (SHRINK) {
            if (check) {   // ================= shrink check
                smo_grid_reduce(slots_i, grid, S, red, &win_i);
                const double cm = win_i.key, cM = win_i.mlow;
                ++checks;
                if (!unshrunk && __dsub_rn(cm, cM) <= __dmul_rn(10.0, a.tol)) {
                    unshrunk = true;
                    smo_reconstruct<ROWS>(a, s, cta, grid, t0, len, s_act, s_alpha, s_g, s_y, s_c);
                    ++recons;
                }
                double cnt = 0.0;
                for (int w = tid; w < (len + 31) >> 5; w += SMO_NT) {
                    unsigned bits = s_act[w];
                    for (int b = 0; b < 32 && 32 * w + b < len; ++b) {
                        if (!((bits >> b) & 1u)) continue;
                        const int l = 32 * w + b;
                        const double y = s_y[l], al = s_alpha[l], c = s_c[l];
                        const bool up = y > 0.0 ? al < c : al > 0.0, lo = y > 0.0 ? al > 0.0 : al < c;
                        const double v = -__dmul_rn(y, s_g[l]);
                        if ((lo && !up && v > cm) || (up && !lo && v < cM)) bits &= ~(1u << b);
                        else cnt += 1.0;
                    }
                    s_act[w] = bits;
                }
                cnt = smo_block_sum(cnt, red);   // (its barriers also publish s_act)
                key = -INFINITY;
                idx = -1.0;
                low = INFINITY;
                for (int l = tid; l < len; l += SMO_NT) {
                    if (!smo_is_active(s_act, l)) continue;
                    const double y = s_y[l], al = s_alpha[l];
                    const bool up = y > 0.0 ? al < s_c[l] : al > 0.0;
                    const double v = -__dmul_rn(y, s_g[l]);
                    if (up && v >= key) {
                        key = v;
                        idx = (double)(t0 + l);
                    }
                }
                smo_block_reduce(key, idx, low, red);
                SmoCand* fresh = a.cand + (size_t)(((k + 1) & 1) * 2) * grid;
                if (tid == 0) {
                    SmoCand c = {key, idx, 0.0, 0.0, 0.0, 0.0, 0.0, cnt};   // mlow carries the slice's active count
                    if (idx >= 0.0) {
                        const int l = (int)((long long)idx - t0);
                        c.alpha = s_alpha[l];
                        c.g = s_g[l];
                        c.y = s_y[l];
                        c.qd = s_qd[l];
                        c.c = s_c[l];
                    }
                    fresh[cta] = c;
                }
                pk_grid_barrier(a.gbar, grid);
                double total = 0.0;
                for (unsigned b = 0; b < grid; ++b) total += __ldcg(&fresh[b].mlow);
                nact = (long long)total;
                shrunk = nact < s.l;
                src_i = fresh;
            }
        }

        // ================= phase 2: i and m; own part of row i; local candidate for j, local M
        smo_grid_reduce(src_i, grid, S, red, &win_i);
        const double m = win_i.key, yi = win_i.y, qii = win_i.qd;
        const long long i = (long long)win_i.idx;
        if constexpr (ROWS == SMO_ROWS_COMPUTED) {
            if (tid == 0 && i >= 0) s_slot[1] = smo_cache_lookup(a, cta, i < a.n ? i : i - a.n, 2 * k + 1, s_hit[1]);
            __syncthreads();
        }
        key = -INFINITY;
        idx = -1.0;
        low = INFINITY;
        for (int l = tid; l < len; l += SMO_NT) {
            if constexpr (SHRINK) {
                if (!smo_is_active(s_act, l)) continue;
            }
            const long long t = t0 + l;
            double qit = 0.0;
            if constexpr (ROWS == SMO_ROWS_COMPUTED) {
                if (i >= 0) {
                    const double v = smo_row_value(a, i < a.n ? i : i - a.n, t, s_slot[1], s_hit[1]);
                    qit = yi == s_y[l] ? v : -v;
                }
            } else if constexpr (ROWS == SMO_ROWS_SIGNED) {
                qit = i >= 0 ? smo_q_signed(a, i, t, yi, s_y[l]) : 0.0;
            } else {
                qit = i >= 0 ? smo_q(a, i, t) : 0.0;
            }
            s_qi[l] = qit;
            const double y = s_y[l], al = s_alpha[l];
            const bool lowset = y > 0.0 ? al > 0.0 : al < s_c[l];
            if (lowset) {
                const double ygt = __dmul_rn(y, s_g[l]);
                low = fmin(low, -ygt);
                const double b = __dadd_rn(m, ygt);
                if (b > 0.0) {
                    double at = __dsub_rn(__dadd_rn(qii, s_qd[l]), __dmul_rn(2.0 * yi * y, qit));
                    if (at <= 0.0) at = SMO_TAU;
                    const double v = __ddiv_rn(__dmul_rn(b, b), at);   // -(objective): -b^2/a is exact negation
                    if (v >= key) {
                        key = v;
                        idx = (double)t;
                    }
                }
            }
        }
        smo_block_reduce(key, idx, low, red);
        if (tid == 0) {
            SmoCand c = {key, idx, 0.0, 0.0, 0.0, 0.0, 0.0, low};
            if (idx >= 0.0) {
                const int l = (int)((long long)idx - t0);
                c.alpha = s_alpha[l];
                c.g = s_g[l];
                c.y = s_y[l];
                c.qd = s_qd[l];
                c.c = s_c[l];
                if constexpr (ROWS == SMO_ROWS_COMPUTED) a.qij[(size_t)(k & 1) * grid + cta] = s_qi[l];
            }
            slots_j[cta] = c;
        }
        pk_grid_barrier(a.gbar, grid);

        // ================= phase 3: j and M, stopping test, the step
        smo_grid_reduce(slots_j, grid, S, red, &win_j);
        const long long j = (long long)win_j.idx;
        const double gap = __dsub_rn(m, win_j.mlow);
        if (cta == 0 && tid == 0) {
            if (k < a.hist_cap) {
                a.hist_f[k] = f;
                a.hist_gap[k] = gap;
            }
            a.st->f = f;
            a.st->ng = gap;
            a.st->iter = k;
        }
        int stop = 0;
        if (j < 0 || gap < a.tol) stop = SVMB200_STATUS_OPTIMAL;
        else if (k >= a.max_iter) stop = SVMB200_STATUS_STOPPED;
        if (stop) {
            if constexpr (SHRINK) {
                if (shrunk) {   // the full problem decides: rebuild G, reactivate everything
                    smo_reconstruct<ROWS>(a, s, cta, grid, t0, len, s_act, s_alpha, s_g, s_y, s_c);
                    ++recons;
                    shrunk = false;
                    if (stop == SVMB200_STATUS_OPTIMAL) {   // select again at the same state, check at the next
                        counter = 1;
                        reselect = true;
                        pending = false;
                        --e;
                        continue;
                    }
                }
            }
            if (cta == 0 && tid == 0) {
                a.st->status = stop;
                __threadfence();
                a.st->done = 1;
            }
            break;
        }
        if (e == a.niter) break;   // the budget ends at an evaluated state
        // libsvm's two-variable step on the signed Q (Q_ij = y_i y_j K_ij for SVC).  y_i != y_j: the step keeps
        // a_i - a_j, quad = Q_ii + Q_jj + 2 Q_ij;  y_i == y_j: it keeps a_i + a_j, quad = Q_ii + Q_jj - 2 Q_ij.  With
        // Q_ij = y_i y_j K_ij both are K_ii + K_jj - 2 K_ij, the curvature along the feasible direction.
        const double qjj = win_j.qd, gi = win_i.g, gj = win_j.g, ci = win_i.c, cj = win_j.c;
        double qij;
        if constexpr (ROWS == SMO_ROWS_COMPUTED) qij = __ldcg(a.qij + (size_t)(k & 1) * grid + j / S);
        else if constexpr (ROWS == SMO_ROWS_SIGNED) qij = smo_q_signed(a, i, j, yi, win_j.y);
        else qij = smo_q(a, i, j);
        const double ai0 = win_i.alpha, aj0 = win_j.alpha;
        double ai = ai0, aj = aj0;
        if (yi != win_j.y) {
            double quad = __dadd_rn(__dadd_rn(qii, qjj), __dmul_rn(2.0, qij));
            if (quad <= 0.0) quad = SMO_TAU;
            const double delta = __ddiv_rn(__dsub_rn(-gi, gj), quad);
            const double diff = __dsub_rn(ai, aj);
            ai = __dadd_rn(ai, delta);
            aj = __dadd_rn(aj, delta);
            if (diff > 0.0) {
                if (aj < 0.0) { aj = 0.0; ai = diff; }
            } else {
                if (ai < 0.0) { ai = 0.0; aj = -diff; }
            }
            if (diff > __dsub_rn(ci, cj)) {
                if (ai > ci) { ai = ci; aj = __dsub_rn(ci, diff); }
            } else {
                if (aj > cj) { aj = cj; ai = __dadd_rn(cj, diff); }
            }
        } else {
            double quad = __dsub_rn(__dadd_rn(qii, qjj), __dmul_rn(2.0, qij));
            if (quad <= 0.0) quad = SMO_TAU;
            const double delta = __ddiv_rn(__dsub_rn(gi, gj), quad);
            const double sum = __dadd_rn(ai, aj);
            ai = __dsub_rn(ai, delta);
            aj = __dadd_rn(aj, delta);
            if (sum > ci) {
                if (ai > ci) { ai = ci; aj = __dsub_rn(sum, ci); }
            } else {
                if (aj < 0.0) { aj = 0.0; ai = sum; }
            }
            if (sum > cj) {
                if (aj > cj) { aj = cj; ai = __dsub_rn(sum, cj); }
            } else {
                if (ai < 0.0) { ai = 0.0; aj = sum; }
            }
        }
        dai = __dsub_rn(ai, ai0);
        daj = __dsub_rn(aj, aj0);
        // f += da_i G_i + da_j G_j + (da_i^2 Q_ii + da_j^2 Q_jj) / 2 + da_i da_j Q_ij   (old G)
        const double lin = __dadd_rn(__dmul_rn(dai, gi), __dmul_rn(daj, gj));
        const double sq = __dadd_rn(__dmul_rn(__dmul_rn(dai, dai), qii), __dmul_rn(__dmul_rn(daj, daj), qjj));
        f = __dadd_rn(f, __dadd_rn(__dadd_rn(lin, __dmul_rn(0.5, sq)), __dmul_rn(__dmul_rn(dai, daj), qij)));
        if (tid == 0) {
            if (i >= t0 && i < t0 + len) s_alpha[i - t0] = ai;
            if (j >= t0 && j < t0 + len) s_alpha[j - t0] = aj;
        }
        pending = true;
        pj = j;
        if constexpr (ROWS == SMO_ROWS_COMPUTED) {
            if (tid == 0) s_slot[0] = smo_cache_lookup(a, cta, j < a.n ? j : j - a.n, 2 * (k + 1), s_hit[0]);
        }
        __syncthreads();   // alpha of i / j in place for the next phase 1
    }
    for (int l = tid; l < len; l += SMO_NT) {
        a.x[t0 + l] = s_alpha[l];
        a.g[t0 + l] = s_g[l];
    }
    if constexpr (SHRINK) {
        if (s.on) {
            for (int l = tid; l < len; l += SMO_NT) s.act[t0 + l] = smo_is_active(s_act, l) ? 1 : 0;
            if (cta == 0 && tid == 0) {
                s.st->counter = counter;
                s.st->unshrunk = unshrunk;
                s.st->shrunk = shrunk;
                s.st->prepared = prepared;
                s.st->checks = checks;
                s.st->reconstructions = recons;
                s.st->active = nact;
            }
        }
    }
}

template <int ROWS>
__global__ void __launch_bounds__(SMO_NT, 1) smo_persistent_kernel(const SmoArgs a) {
    smo_solve<ROWS, false>(a, SmoShrink{}, blockIdx.x, gridDim.x);
}

// the solver's arguments and its shrinking state (one launch argument)
struct SmoShrinkArgs {
    SmoArgs a;
    SmoShrink s;
};

template <int ROWS>
__global__ void __launch_bounds__(SMO_NT, 1) smo_shrink_kernel(const SmoShrinkArgs p) {
    smo_solve<ROWS, true>(p.a, p.s, blockIdx.x, gridDim.x);
}

// K14: one problem of a batch -- its arguments and its CTAs [cta0, cta0 + grid) of the launch
struct SmoBatchProblem {
    SmoArgs a;
    int cta0, grid;
    SmoShrink s;      // smo_batch_shrink_kernel only (s.on = 0: the problem does not shrink)
};

struct SmoBatchArgs {
    const SmoBatchProblem* probs;   // in ascending cta0, the CTA ranges back to back from 0
    int count;
};

template <int ROWS, bool SHRINK>
__device__ __forceinline__ void smo_batch(const SmoBatchArgs& b) {
    __shared__ SmoArgs pa;   // the problem's arguments, read once per launch
    __shared__ SmoShrink ps;
    __shared__ unsigned p_cta, p_grid;
    if (threadIdx.x == 0) {
        int p = 0;
        while (p + 1 < b.count && (int)blockIdx.x >= b.probs[p + 1].cta0) ++p;
        pa = b.probs[p].a;
        if constexpr (SHRINK) ps = b.probs[p].s;
        p_cta = blockIdx.x - (unsigned)b.probs[p].cta0;
        p_grid = (unsigned)b.probs[p].grid;
    }
    __syncthreads();
    smo_solve<ROWS, SHRINK>(pa, ps, p_cta, p_grid);
}

template <int ROWS>
__global__ void __launch_bounds__(SMO_NT, 1) smo_batch_kernel(const SmoBatchArgs b) {
    smo_batch<ROWS, false>(b);
}

// K14 with shrinking: each problem's SmoShrink::on says whether it shrinks
template <int ROWS>
__global__ void __launch_bounds__(SMO_NT, 1) smo_batch_shrink_kernel(const SmoBatchArgs b) {
    smo_batch<ROWS, true>(b);
}
