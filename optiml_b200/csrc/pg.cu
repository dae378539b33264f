// K2 (streaming FP64 matvec), K3 (vector phase) and the projected-gradient driver.
//
// Algorithm restated from optiml/opti/constrained/projected_gradient.py:76-143 (reference, NumPy):
//   loop:  f = x'Qx/2 + q'x ; g = Qx + q ; d = -g projected on the active box faces ; ng = |d|
//          callback ; ng <= eps -> optimal ; iter >= max_iter -> stopped
//          max_t = largest feasible step ; den = d'Qd ; t = den<=1e-16 ? max_t : min(-g'd/den, max_t)
//          x += t d ; iter += 1
// The reference streams Q three times per iteration.  Here Q is streamed ONCE per iteration:
//   w = Q u  (K2; u = d, or d+ - d- for the SVR block Hessian),  den = u'w,  g <- g + t w,
//   f = x'(g+q)/2,  -g'd == d'd  (K3).
//
// Every reduction has a fixed shape that depends on the problem size only -- never on the number of
// GPUs, the grid or the arrival order -- so the iterate is bit-identical for 1, 2, 4 and 8 GPUs.
#include "common.cuh"
#include "al_math.cuh"
#include "k2_matvec.cuh"   // K2, K2 x NB (device code)
#include "k2_symv.cuh"     // K2s: one pass over the upper triangle of a symmetric matrix (opt-in)
#include "k2_exact.cuh"    // K2e: K2's bits from the upper triangle of an exactly symmetric matrix
#include "k3_vector.cuh"   // K3 vector phases and kernel entry points (device code)
#include "k_persistent.cuh"  // the whole loop in one cooperative kernel, matrix in shared memory (small problems)
#include "k_smo.cuh"         // K11: SMO with the equality constraint, one cooperative kernel for many iterations
#include <algorithm>
#include <math.h>
#include <stdlib.h>
#include <memory>

// ------------------------------------------------------------------------------------------ product launchers
// Every product w = Q u of a solver runs one of three passes over the matrix: K2 (the full pass), K2s (the upper triangle,
// opt-in) or K2e (the upper triangle with K2's bits, for exactly symmetric self-Grams).  launch_product checks the
// operands and runs the pass a solver chose at creation (product_pass).
enum ProductPass : int { PASS_FULL, PASS_SYMMETRIC, PASS_EXACT };

// a grow-only device buffer of the context's product scratch
struct ScratchBuf {
    void* p = nullptr;
    size_t bytes = 0;
    template <typename T>
    T* as() const { return static_cast<T*>(p); }
};

struct MatvecScratch {
    ScratchBuf wpart, tickets;   // segment partials (K2, K2 x NB, K2e); one ticket per row group (K2), zero between passes
    // K2s: row / column partials, work items, row-sum slots + band of every `unit` rows, and the plan of the
    // (n, ld, rank, ranks) they were last built for
    ScratchBuf sy_rowpart, sy_colpart, sy_items, sy_tables;
    int64_t sy_n = -1, sy_ld = -1;
    int sy_rank = -1, sy_P = -1;
    SymvPlan sy_plan;
    // K2e: column chains and the (A, B) segment pairs of the grid, for ex_nseg segments
    ScratchBuf ex_colchain, ex_pairs;
    int ex_nseg = -1;
};

static MatvecScratch& matvec_scratch(svmb200_ctx* ctx) {
    if (!ctx->matvec_scratch) ctx->matvec_scratch = new MatvecScratch();
    return *static_cast<MatvecScratch*>(ctx->matvec_scratch);
}

void svm_release_matvec_scratch(svmb200_ctx* ctx) {
    MatvecScratch* s = static_cast<MatvecScratch*>(ctx->matvec_scratch);
    if (!s) return;
    for (ScratchBuf* b : {&s->wpart, &s->tickets, &s->sy_rowpart, &s->sy_colpart, &s->sy_items, &s->sy_tables,
                          &s->ex_colchain, &s->ex_pairs})
        if (b->p) cudaFree(b->p);
    delete s;
    ctx->matvec_scratch = nullptr;
}

// `count` elements of T at least, and never an empty buffer (the kernels take its address either way)
template <typename T>
static int reserve(svmb200_ctx* ctx, ScratchBuf& b, size_t count) {
    return svm_scratch_reserve(ctx, &b.p, &b.bytes, (count ? count : 1) * sizeof(T));
}

static int mv_nseg(int64_t ld) { return (int)((ld + MV_SEG - 1) / MV_SEG); }

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// the context's sticky exchange-fault flag (see ll_load)
static int* exchange_fault(svmb200_ctx* ctx) { return reinterpret_cast<int*>(ctx->arena + ARENA_LOCAL_OFF + 8); }

// the checks of every product: the leading dimension against the rule of its pass, 16-byte matrix and vectors
static int check_operands(bool ld_ok, const char* ld_rule, bool aligned) {
    if (!ld_ok) {
        svmb200_set_error("product: ld must be %s", ld_rule);
        return SVMB200_ERR_ARG;
    }
    if (!aligned) {
        svmb200_set_error("product: operands must be 16-byte aligned");
        return SVMB200_ERR_ARG;
    }
    return SVMB200_OK;
}

static int matvec_scratch_reserve(svmb200_ctx* ctx, MatvecScratch& s, int64_t nrows, int64_t ld, int nvec = 1) {
    SVM_TRY(reserve<double>(ctx, s.wpart, (size_t)nvec * mv_nseg(ld) * (size_t)round_up64(nrows, 16)));
    const size_t had = s.tickets.bytes;
    SVM_TRY(reserve<unsigned>(ctx, s.tickets, (size_t)((nrows + MV_GROUP - 1) / MV_GROUP)));
    if (s.tickets.bytes != had) SVM_CUDA(cudaMemsetAsync(s.tickets.p, 0, s.tickets.bytes, ctx->stream));
    return SVMB200_OK;
}

struct ExchangeTargets {
    int nranks = 0;
    unsigned tag = 0;
    ulonglong2* peer_w[SVM_MAX_RANKS] = {};
};

// One product: w = Q u over the n x ld matrix, or over this rank's shard of nrows rows (K2).  With u_rows / denpart, also
// the shares of u'w per 64-row group; with `done`, nothing runs once the solver's device state says so.  With xt, the
// results go straight into every rank's gathered buffer (fused exchange; w and denpart then only carry the slot
// geometry), under sequence number seq; rpr is the rows per rank of that exchange.  phase: see launch_symv.
struct ProductOperands {
    const double* Q = nullptr;
    int64_t n = 0, nrows = 0, ld = 0, rpr = 0;
    const double* u = nullptr;
    double* w = nullptr;
    const double* u_rows = nullptr;
    double* denpart = nullptr;
    const int* done = nullptr;
    const ExchangeTargets* xt = nullptr;
    unsigned long long seq = 0;
    int phase = 0;
};

static int launch_matvec(svmb200_ctx* ctx, const ProductOperands& op) {
    MatvecScratch& s = matvec_scratch(ctx);
    SVM_TRY(matvec_scratch_reserve(ctx, s, op.nrows, op.ld));
    MatvecArgs a;
    a.Q = op.Q;
    a.ld = op.ld;
    a.nrows = op.nrows;
    a.u = op.u;
    a.w = op.w;
    a.wpart = s.wpart.as<double>();
    a.nrows_pad = round_up64(op.nrows, 16);
    a.tickets = s.tickets.as<unsigned>();
    a.u_rows = op.u_rows;
    a.denpart = op.denpart;
    a.nseg = mv_nseg(op.ld);
    a.done = op.done;
    const int64_t ngroups = (op.nrows + MV_GROUP - 1) / MV_GROUP;
    a.nranks_x = 0;
    a.tag = 0;
    a.fault = nullptr;
    if (op.xt != nullptr) {
        a.nranks_x = op.xt->nranks;
        a.tag = op.xt->tag;
        a.fault = exchange_fault(ctx);
        for (int r = 0; r < op.xt->nranks; ++r) a.peer_w[r] = op.xt->peer_w[r];
    }
    const int64_t nitems = ngroups * MV_BPG * a.nseg;
    if (nitems >= (1ll << 31)) {
        svmb200_set_error("matvec: grid too large");
        return SVMB200_ERR_ARG;
    }
    SVM_CUDA(svm_launch_chained(matvec_seg_kernel, dim3((unsigned)nitems), dim3(MV_NT), ctx->stream, a));
    ctx->launches++;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ K2s launcher
// w = Q u from the upper triangle of the symmetric matrix (see k2_symv.cuh); same outputs as launch_matvec.  One rank
// holding the whole matrix, or the ranks of a fused peer exchange (op.xt != null): `phase` 1 = tile pass + the column sums
// for the other ranks, 2 = combine (waits for the column sums of the others), 0 = both.  A single host thread that drives
// several ranks issues phase 1 for all of them before phase 2 (the host emulation runs launches synchronously; on hardware
// the order is immaterial).
constexpr size_t symv_inbox_bytes(int64_t rpr, int P) { return (size_t)P * (size_t)rpr * sizeof(ulonglong2); }
static size_t symv_inbox_off(const svmb200_ctx* ctx) { return ctx->arena_bytes / 2; }

// resident CTAs of the tile kernel the planner balances the grid for (a build-time override exists for the tests on the host
// emulation, whose problems are far too small to fill 296 slots)
static int symv_plan_slots(int sm_count) {
#ifdef SVMB200_SYMV_PLAN_SLOTS
    (void)sm_count;
    return SVMB200_SYMV_PLAN_SLOTS;
#else
    return SymvDefault::MINB * (sm_count > 0 ? sm_count : 148);
#endif
}

static int launch_symv(svmb200_ctx* ctx, const ProductOperands& op) {
    using S = SymvDefault;
    const ExchangeTargets* xt = op.xt;
    const int64_t n = op.n, ld = op.ld, rpr = op.rpr;
    const int P = xt ? xt->nranks : 1, rank = xt ? ctx->rank : 0;
    MatvecScratch& s = matvec_scratch(ctx);
    if (s.sy_n != n || s.sy_ld != ld || s.sy_rank != rank || s.sy_P != P) {
        s.sy_n = -1;   // until the tables of the new plan are on the device
        SymvPlan& plan = s.sy_plan;
        symv_build_plan<S>(n, ld, rank, P, P == 1 ? n : rpr, plan, symv_plan_slots(ctx->sm_count));
        SVM_TRY(reserve<double>(ctx, s.sy_rowpart, (size_t)plan.nseg_max * (size_t)round_up64(plan.nrows, 16)));
        SVM_TRY(reserve<double>(ctx, s.sy_colpart, (size_t)plan.nbands * ld));
        SVM_TRY(reserve<SymvItem>(ctx, s.sy_items, plan.items.size()));
        SVM_TRY(reserve<int>(ctx, s.sy_tables, plan.nseg.size() + plan.band_of_unit.size()));
        if (!plan.items.empty())
            SVM_CUDA(cudaMemcpyAsync(s.sy_items.p, plan.items.data(), plan.items.size() * sizeof(SymvItem), cudaMemcpyHostToDevice,
                                     ctx->stream));
        if (!plan.nseg.empty())
            SVM_CUDA(cudaMemcpyAsync(s.sy_tables.p, plan.nseg.data(), plan.nseg.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        if (!plan.band_of_unit.empty())
            SVM_CUDA(cudaMemcpyAsync(s.sy_tables.as<int>() + plan.nseg.size(), plan.band_of_unit.data(),
                                     plan.band_of_unit.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        SVM_CUDA(cudaStreamSynchronize(ctx->stream));  // once per problem size; the tables stay valid for every later pass
        s.sy_n = n;
        s.sy_ld = ld;
        s.sy_rank = rank;
        s.sy_P = P;
    }
    const SymvPlan& plan = s.sy_plan;
    if (plan.nrows <= 0) return SVMB200_OK;
    const long long n_pad = round_up64(plan.nrows, 16);
    int* fault = xt ? exchange_fault(ctx) : nullptr;
    const unsigned tag = xt ? xt->tag : 0u;
    const size_t inbox_par = xt ? symv_inbox_off(ctx) + (size_t)(op.seq & 1) * symv_inbox_bytes(rpr, P) : 0;
    if (op.phase == 0 || op.phase == 1) {
        SymvArgs a;
        a.Q = op.Q;
        a.ld = ld;
        a.nrows = plan.nrows;
        a.row0 = plan.row0;
        a.n_pad = n_pad;
        a.u = op.u;
        a.rowpart = s.sy_rowpart.as<double>();
        a.colpart = s.sy_colpart.as<double>();
        a.items = s.sy_items.as<SymvItem>();
        a.done = op.done;
        a.fault = fault;
        SVM_TRY(svm_opt_in_smem<symv_tile_kernel<S>>(ctx, S::RING_BYTES));
        SVM_CUDA(svm_launch_chained_smem(symv_tile_kernel<S>, dim3((unsigned)plan.items.size()), dim3(SY_NT),
                                         (size_t)S::RING_BYTES, ctx->stream, a));
        ctx->launches++;
        if (!plan.sends.empty()) {
            SymvSendArgs sa = {};
            sa.colpart = s.sy_colpart.as<double>();
            sa.ld = ld;
            sa.nsend = (int)plan.sends.size();
            long long total = 0;
            for (int i = 0; i < sa.nsend; ++i) {
                sa.sends[i] = plan.sends[(size_t)i];
                sa.inbox[i] = reinterpret_cast<ulonglong2*>(ctx->peer_arena[plan.sends[(size_t)i].dest] + inbox_par) + (size_t)rank * rpr;
                total += plan.sends[(size_t)i].ncols;
            }
            sa.tag = tag;
            sa.done = op.done;
            sa.fault = fault;
            SVM_CUDA(svm_launch_chained(symv_send_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), ctx->stream, sa));
            ctx->launches++;
        }
    }
    if (op.phase == 0 || op.phase == 2) {
        SymvCombineArgs c = {};
        c.rowpart = s.sy_rowpart.as<double>();
        c.colpart = s.sy_colpart.as<double>();
        c.ld = ld;
        c.nrows = plan.nrows;
        c.row0 = plan.row0;
        c.n_pad = n_pad;
        c.unit = plan.unit;
        c.band_of_unit = s.sy_tables.as<int>() + plan.nseg.size();
        c.nseg = s.sy_tables.as<int>();
        c.u_rows = op.u_rows;
        c.w = op.w;
        c.denpart = op.denpart;
        c.done = op.done;
        c.nrecv = (int)plan.recvs.size();
        for (int i = 0; i < c.nrecv; ++i) c.recvs[i] = plan.recvs[(size_t)i];
        c.inbox = xt ? reinterpret_cast<const ulonglong2*>(ctx->arena + inbox_par) : nullptr;
        c.rpr = rpr;
        c.tag = tag;
        c.fault = fault;
        if (xt != nullptr) {
            c.nranks_x = xt->nranks;
            c.share_off = (long long)(op.denpart - op.w);
            for (int r = 0; r < xt->nranks; ++r) c.peer_w[r] = xt->peer_w[r];
        }
        const int64_t ngroups = (plan.nrows + MV_GROUP - 1) / MV_GROUP;
        SVM_CUDA(svm_launch_chained(symv_combine_kernel, dim3((unsigned)ngroups), dim3(MV_GROUP * SY_CPARTS), ctx->stream, c));
        ctx->launches++;
    }
    return SVMB200_OK;
}

// bytes of the matrix one symmetric pass streams (diagonal blocks in full + everything to their right) and the shape of
// its tiles -- what a roofline of K2s is computed from
extern "C" int svmb200_symv_geometry(int64_t n, int64_t ld, int64_t* streamed_bytes, int64_t* band_rows, int64_t* panel_cols,
                                     int64_t* items) {
    using S = SymvDefault;
    SVM_CHECK_ARG(n >= 0 && ld >= n, "bad argument");
    SymvPlan plan;
    symv_build_plan<S>(n, ld, 0, 1, n, plan);
    if (streamed_bytes) *streamed_bytes = 8 * plan.streamed_elems;
    if (items) *items = (int64_t)plan.items.size();
    if (band_rows) *band_rows = S::BH;
    if (panel_cols) *panel_cols = S::BW;
    return SVMB200_OK;
}

static int64_t rows_per_rank(int64_t n, int nranks);

// the plan of rank `rank` of `nranks` (svmb200_shard_rows blocks) for the shipped tile shape: bands (tall + short), work items,
// ratio of the simulated finish time to a perfectly balanced one -- for tests and tuning; any output pointer may be NULL
extern "C" int svmb200_symv_plan_info(int64_t n, int64_t ld, int rank, int nranks, int sm_count, int64_t* bands,
                                      int64_t* short_bands, int64_t* items, double* finish_over_ideal) {
    using S = SymvDefault;
    SVM_CHECK_ARG(n >= 0 && ld >= n && nranks >= 1 && rank >= 0 && rank < nranks, "bad argument");
    SymvPlan plan;
    const int slots = symv_plan_slots(sm_count);
    symv_build_plan<S>(n, ld, rank, nranks, nranks == 1 ? n : rows_per_rank(n, nranks), plan, slots);
    int64_t nshort = 0;
    for (int64_t I = 0; I + 1 < plan.nbands; ++I) nshort += plan.band_lr0[(size_t)I + 1] - plan.band_lr0[(size_t)I] < S::BH;
    std::vector<double> cost;
    double total = 0.0;
    for (const SymvItem& it : plan.items) {
        cost.push_back((double)it.rows * it.width + SVMB200_SYMV_PLAN_OVERHEAD);
        total += cost.back();
    }
    if (bands) *bands = plan.nbands;
    if (short_bands) *short_bands = nshort;
    if (items) *items = (int64_t)plan.items.size();
    if (finish_over_ideal) *finish_over_ideal = total > 0.0 ? symv_makespan(cost, slots) / (total / slots) : 1.0;
    return SVMB200_OK;
}

// the work items of that plan, seven ints each {first local row, rows, band, first column, columns, row-sum slot, 1 if the
// item also feeds column sums}, and the first global row of the rank's block -- so that a test can check, on the host, that
// the plans of all ranks cover every pair of rows exactly once
extern "C" int svmb200_symv_plan_items(int64_t n, int64_t ld, int rank, int nranks, int sm_count, int32_t* items7, int64_t capacity,
                                       int64_t* count, int64_t* row0) {
    using S = SymvDefault;
    SVM_CHECK_ARG(n >= 0 && ld >= n && nranks >= 1 && rank >= 0 && rank < nranks && count != nullptr, "bad argument");
    SymvPlan plan;
    symv_build_plan<S>(n, ld, rank, nranks, nranks == 1 ? n : rows_per_rank(n, nranks), plan, symv_plan_slots(sm_count));
    *count = (int64_t)plan.items.size();
    if (row0) *row0 = plan.row0;
    if (items7 != nullptr) {
        SVM_CHECK_ARG(capacity >= *count, "items7 is too small");
        for (size_t i = 0; i < plan.items.size(); ++i) {
            const SymvItem& it = plan.items[i];
            const int32_t v[7] = {it.lr0, it.rows, it.band, it.c0, it.width, it.seg, it.cols};
            memcpy(items7 + 7 * i, v, sizeof(v));
        }
    }
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ K2e launcher
// w = Q u with K2's bits from the upper triangle of an exactly symmetric n x n matrix (see k2_exact.cuh); same outputs as
// launch_matvec on one rank.

// at least two segments, and every segment but the last one made of real rows (the column chains of a segment cover all
// of its rows)
static bool exact_shape_ok(int64_t n, int64_t ld) {
    const int nseg = mv_nseg(ld);
    return n > 0 && ld >= n && ld % 2 == 0 && nseg >= 2 && n > (int64_t)(nseg - 1) * MV_SEG;
}

// (A, B) segment pairs, B >= A, in launch order: the full off-diagonal blocks first, the diagonal blocks last
static std::vector<int2> exact_pairs(int nseg) {
    std::vector<int2> v;
    for (int A = 0; A < nseg; ++A)
        for (int B = A + 1; B < nseg - 1; ++B) v.push_back(make_int2(A, B));
    for (int A = 0; A < nseg - 1; ++A) v.push_back(make_int2(A, nseg - 1));
    for (int A = 0; A < nseg; ++A) v.push_back(make_int2(A, A));
    return v;
}

static int exact_scratch_reserve(svmb200_ctx* ctx, MatvecScratch& s, int64_t n, int64_t ld) {
    SVM_TRY(matvec_scratch_reserve(ctx, s, n, ld));
    const int nseg = mv_nseg(ld);
    SVM_TRY(reserve<double>(ctx, s.ex_colchain, (size_t)exact_colchain_off(nseg - 1, ld)));
    if (s.ex_nseg != nseg) {
        s.ex_nseg = -1;   // until the new table is on the device
        const std::vector<int2> pairs = exact_pairs(nseg);
        SVM_TRY(reserve<int2>(ctx, s.ex_pairs, pairs.size()));
        SVM_CUDA(cudaMemcpyAsync(s.ex_pairs.p, pairs.data(), pairs.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream));
        SVM_CUDA(cudaStreamSynchronize(ctx->stream));  // once per segment count; the table stays valid for every later pass
        s.ex_nseg = nseg;
    }
    return SVMB200_OK;
}

static int launch_matvec_exact(svmb200_ctx* ctx, const ProductOperands& op) {
    using S = ExactDefault;
    MatvecScratch& s = matvec_scratch(ctx);
    SVM_TRY(exact_scratch_reserve(ctx, s, op.n, op.ld));
    const int nseg = mv_nseg(op.ld);
    const long long nrows_pad = round_up64(op.n, 16);
    ExactArgs a;
    a.Q = op.Q;
    a.ld = op.ld;
    a.n = op.n;
    a.nrows_pad = nrows_pad;
    a.u = op.u;
    a.wpart = s.wpart.as<double>();
    a.colchain = s.ex_colchain.as<double>();
    a.pairs = s.ex_pairs.as<int2>();
    a.done = op.done;
    SVM_TRY(svm_opt_in_smem<matvec_exact_tile_kernel<S>>(ctx, S::RING_BYTES));
    const unsigned nitems = (unsigned)((size_t)nseg * (nseg + 1) / 2 * MV_NT);
    SVM_CUDA(svm_launch_chained_smem(matvec_exact_tile_kernel<S>, dim3(nitems), dim3(MV_NT), (size_t)S::RING_BYTES, ctx->stream, a));
    ctx->launches++;
    ExactCombineArgs c;
    c.wpart = s.wpart.as<double>();
    c.colchain = s.ex_colchain.as<double>();
    c.ld = op.ld;
    c.nrows = op.n;
    c.nrows_pad = nrows_pad;
    c.nseg = nseg;
    c.u_rows = op.u_rows;
    c.w = op.w;
    c.denpart = op.denpart;
    c.done = op.done;
    SVM_CUDA(svm_launch_chained(matvec_exact_combine_kernel, dim3((unsigned)((op.n + MV_GROUP - 1) / MV_GROUP)), dim3(MV_NT),
                                ctx->stream, c));
    ctx->launches++;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ one launch path
static int launch_product(svmb200_ctx* ctx, ProductPass pass, const ProductOperands& op) {
    static const char* const ld_rule[] = {"a positive multiple of 2", "even and at least n",
                                          "even and at least n, with n reaching into the last of two or more column segments"};
    if (pass == PASS_FULL ? op.nrows <= 0 : pass == PASS_SYMMETRIC && op.n <= 0)
        return SVMB200_OK;   // an empty shard has nothing to compute or to send
    const bool ld_ok = pass == PASS_FULL      ? op.ld > 0 && op.ld % 2 == 0
                     : pass == PASS_SYMMETRIC ? op.ld % 2 == 0 && op.ld >= op.n
                                              : exact_shape_ok(op.n, op.ld);
    SVM_TRY(check_operands(ld_ok, ld_rule[pass], aligned16(op.Q) && aligned16(op.u)));
    return pass == PASS_FULL ? launch_matvec(ctx, op) : pass == PASS_SYMMETRIC ? launch_symv(ctx, op) : launch_matvec_exact(ctx, op);
}

// w = Q u over an n x ld matrix (K2: over nrows = n rows of it) with no exchange, no shares of u'w
static int launch_plain(svmb200_ctx* ctx, ProductPass pass, const double* dQ, int64_t n, int64_t ld, const double* du,
                        double* dw, const int* d_done = nullptr) {
    ProductOperands op;
    op.Q = dQ;
    op.n = op.nrows = op.rpr = n;
    op.ld = ld;
    op.u = du;
    op.w = dw;
    op.done = d_done;
    return launch_product(ctx, pass, op);
}

int svm_launch_matvec(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, const double* du, double* dw,
                      const int* d_done) {
    return launch_plain(ctx, PASS_FULL, dQ, nrows, ld, du, dw, d_done);
}

extern "C" int svmb200_matvec(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, const double* du,
                              double* dw) {
    SVM_TRY(svm_use(ctx));
    return launch_plain(ctx, PASS_FULL, dQ, nrows, ld, du, dw);
}

// w = Q u for a symmetric n x n matrix from its upper triangle (the lower one is never read)
extern "C" int svmb200_symv(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, const double* du, double* dw) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dQ != nullptr && du != nullptr && dw != nullptr && n >= 0, "bad argument");
    return launch_plain(ctx, PASS_SYMMETRIC, dQ, n, ld, du, dw);
}

extern "C" int svmb200_matvec_exact(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, const double* du, double* dw) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dQ != nullptr && du != nullptr && dw != nullptr, "null operand");
    return launch_plain(ctx, PASS_EXACT, dQ, n, ld, du, dw);
}

extern "C" int svmb200_exact_symv_geometry(int64_t n, int64_t ld, int64_t* matrix_bytes, int64_t* scratch_bytes,
                                           int64_t* items) {
    SVM_CHECK_ARG(exact_shape_ok(n, ld), "the exact symmetric pass does not apply to this shape");
    const int nseg = mv_nseg(ld);
    int64_t elems = 0;
    for (const int2 pr : exact_pairs(nseg)) {
        const int64_t rowsA = std::min<int64_t>((int64_t)(pr.x + 1) * MV_SEG, n) - (int64_t)pr.x * MV_SEG;
        const int64_t colsB = std::min<int64_t>((int64_t)(pr.y + 1) * MV_SEG, ld) - (int64_t)pr.y * MV_SEG;
        elems += rowsA * colsB;
    }
    if (matrix_bytes) *matrix_bytes = 8 * elems;
    if (scratch_bytes) *scratch_bytes = 2 * 8 * exact_colchain_off(nseg - 1, ld);   // written by the tile pass, read by the combine
    if (items) *items = (int64_t)exact_pairs(nseg).size() * MV_NT;
    return SVMB200_OK;
}

static int launch_matvec_multi(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, int nb,
                               const double* const* du, double* const* dw, const double* const* du_rows,
                               double* const* ddenpart, const int* const* d_done, const ExchangeTargets* xt = nullptr,
                               long long xstride = 0, long long share_off = 0) {
    if (nrows <= 0) return SVMB200_OK;
    if (nb < 1 || nb > MV_MULTI_MAX) {
        svmb200_set_error("matvec_multi: between 1 and %d vectors per launch", MV_MULTI_MAX);
        return SVMB200_ERR_ARG;
    }
    bool aligned = aligned16(dQ);
    for (int b = 0; b < nb; ++b) aligned = aligned && aligned16(du[b]);
    SVM_TRY(check_operands(ld > 0 && ld % 2 == 0, "a positive multiple of 2", aligned));
    MatvecScratch& s = matvec_scratch(ctx);
    SVM_TRY(matvec_scratch_reserve(ctx, s, nrows, ld, nb));
    MatvecMultiArgs a = {};
    a.Q = dQ;
    a.ld = ld;
    a.nrows = nrows;
    a.nrows_pad = round_up64(nrows, 16);
    a.wpart = s.wpart.as<double>();
    a.tickets = s.tickets.as<unsigned>();
    a.nseg = mv_nseg(ld);
    for (int b = 0; b < nb; ++b) {
        a.u[b] = du[b];
        a.w[b] = dw[b];
        a.u_rows[b] = du_rows ? du_rows[b] : nullptr;
        a.denpart[b] = ddenpart ? ddenpart[b] : nullptr;
        a.done[b] = d_done ? d_done[b] : nullptr;
    }
    if (xt != nullptr) {
        a.nranks_x = xt->nranks;
        a.tag = xt->tag;
        a.xstride = xstride;
        a.share_off = share_off;
        a.fault = exchange_fault(ctx);
        for (int r = 0; r < xt->nranks; ++r) a.peer_w[r] = xt->peer_w[r];
    }
    const int64_t ngroups = (nrows + MV_GROUP - 1) / MV_GROUP;
    int64_t nitems = 0;
    cudaError_t launch_err = cudaSuccess;
    switch (nb) {
#define LAUNCH_MULTI(NB)                                                                                \
    case NB:                                                                                            \
        nitems = ngroups * (MV_GROUP / (MultiCfg<NB>::R * MultiCfg<NB>::H)) * a.nseg;                   \
        if (nitems >= (1ll << 31)) break;                                                               \
        launch_err = svm_launch_chained(matvec_seg_multi_kernel<NB>, dim3((unsigned)nitems),            \
                                        dim3(MV_NT * MultiCfg<NB>::H), ctx->stream, a);                 \
        break;
        LAUNCH_MULTI(1)
        LAUNCH_MULTI(2)
        LAUNCH_MULTI(3)
        LAUNCH_MULTI(4)
#undef LAUNCH_MULTI
    }
    if (nitems >= (1ll << 31)) {
        svmb200_set_error("matvec: grid too large");
        return SVMB200_ERR_ARG;
    }
    ctx->launches++;
    SVM_CUDA(launch_err);
    return SVMB200_OK;
}

// dw[b][i] = sum_j dQ[i][j] du[b][j] for `count` vectors, ceil(count / 4) passes over the matrix
extern "C" int svmb200_matvec_multi(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld,
                                    const double* const* du, double* const* dw, int count) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dQ != nullptr && du != nullptr && dw != nullptr && count >= 1, "bad argument");
    for (int b = 0; b < count; ++b) SVM_CHECK_ARG(du[b] != nullptr && dw[b] != nullptr, "null vector");
    const int nlaunch = (count + MV_MULTI_MAX - 1) / MV_MULTI_MAX;
    for (int l = 0, b0 = 0; l < nlaunch; ++l) {
        const int nb = (count - b0 + (nlaunch - l) - 1) / (nlaunch - l);  // balanced split
        SVM_TRY(launch_matvec_multi(ctx, dQ, nrows, ld, nb, du + b0, dw + b0, nullptr, nullptr, nullptr));
        b0 += nb;
    }
    return SVMB200_OK;
}

static int64_t rows_per_rank(int64_t n, int nranks) { return round_up64((n + nranks - 1) / nranks, ROW_ALIGN); }

extern "C" int svmb200_shard_rows(int64_t n, int rank, int nranks, int64_t* row0, int64_t* nrows) {
    SVM_CHECK_ARG(n >= 0 && nranks >= 1 && rank >= 0 && rank < nranks && row0 && nrows, "bad argument");
    const int64_t rpr = rows_per_rank(n, nranks);
    int64_t r0 = (int64_t)rank * rpr;
    if (r0 > n) r0 = n;
    int64_t nr = n - r0;
    if (nr > rpr) nr = rpr;
    *row0 = r0;
    *nrows = nr;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ driver
enum SolverKind : int {
    SOLVER_PG = 0,   // projected gradient
    SOLVER_FW = 1,   // Frank-Wolfe
    SOLVER_AL = 2,   // augmented Lagrangian + stochastic rule
    SOLVER_SMO = 3,  // SMO (K11 / K12)
};

// SMO: the kernel's arguments, filled at creation (smo_launch sets the iteration range and the history), its grid, the
// row source and the buffer of the computed rows
struct SmoSolver {
    SmoArgs a = {};
    int grid = 0;
    int rows = SMO_ROWS_RESIDENT;   // SMO_ROWS_RESIDENT, _SIGNED (svmb200_smo_create_signed) or _COMPUTED
    void* rows_buf = nullptr;  // |x|^2 | Q_ij slots | tags | stamps | stats | cache
    SmoShrink shrink = {};     // shrinking (svmb200_smo_set_shrinking): on, and its buffer at shrink.q
    bool started = false;      // a run has started
};

struct svmb200_pg {
    svmb200_ctx* ctx = nullptr;
    const double* dQ = nullptr;
    int64_t n = 0, ld = 0, row0 = 0, nrows = 0, nvars = 0, rows_per_rank = 0;
    int svr = 0;
    SolverKind solver = SOLVER_PG;
    ALArgs al = {};      // SOLVER_AL only
    SmoSolver smo;       // SOLVER_SMO only
    double fw_t = 0.0;   // Frank-Wolfe stabilisation parameter
    double eps = 1e-6;
    int64_t max_iter = 1000;
    int64_t hist_cap = 0;
    // device buffers
    double *x = nullptr, *g = nullptr, *d = nullptr, *u = nullptr, *w = nullptr;  // w: gathered [P][stride]
    int64_t stride = 0;  // rows_per_rank results + rows_per_rank / MV_GROUP shares of u'w
    bool p2p = false;           // fused exchange through the peer arena instead of ncclAllGather
    ProductPass pass = PASS_FULL;   // the pass of its products (product_pass)
    unsigned long long cur_seq = 0;  // sequence number of the product the next vector kernel consumes
    int nctas = 1;
    double *q = nullptr, *lb = nullptr, *ub = nullptr;
    double* sgn = nullptr;  // label signs (Q = (s s') o resident matrix), or null
    double *part = nullptr, *hist_f = nullptr, *hist_ng = nullptr;  // SMO: one allocation (smo_hist_reserve) at hist_f
    PGDeviceState* st = nullptr;
    PGDeviceState* st_host = nullptr;  // pinned; points at the slot of the most recent completed poll
    void* pinned = nullptr;            // 256 bytes: two poll slots of {PGDeviceState, fault flag}
    cudaEvent_t ev_poll[2] = {nullptr, nullptr};
    int64_t last_samples = 0;          // iterations of the last run that carried profiling events
    bool deferred_start = false;       // single-process group: first product + INIT are issued by svmb200_pg_start_group
    // host-side cursor
    int64_t k_next = 0;     // next iteration whose STEP kernel has not been enqueued
    bool finished = false;  // device reported done
    // stats of the last run
    float last_ms = 0.f, last_mv_ms = 0.f, last_comm_ms = 0.f, last_vec_ms = 0.f;
    int64_t last_passes = 0;
    bool profile = false;
    std::vector<cudaEvent_t> mv_ev;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // the context's solver pair (svmb200_timer_* has its own)
    void* slab = nullptr;        // all device buffers below live in this slab
    bool slab_private = false;   // true: allocated for this solver only (the context's slab was busy, or SMO)
};

constexpr size_t POLL_SLOT_BYTES = 128;  // {PGDeviceState, ..., int fault} per poll slot of the pinned block
constexpr int64_t PROFILE_STRIDE = 16;   // with profiling on, one iteration in this many carries CUDA events

static unsigned exchange_tag(unsigned long long seq) { return (unsigned)(seq % 0xfffffffful) + 1u; }  // never 0

static VecArgs make_vec_args(svmb200_pg* pg) {
    VecArgs a;
    a.x = pg->x;
    a.g = pg->g;
    a.d = pg->d;
    a.u = pg->u;
    a.q = pg->q;
    a.lb = pg->lb;
    a.ub = pg->ub;
    a.sgn = pg->sgn;
    a.gathered = pg->w;
    a.gathered_ll = nullptr;
    a.tag = 0;
    a.fault = nullptr;
    a.ll_pstride = 0;
    if (pg->p2p) {
        svmb200_ctx* ctx = pg->ctx;
        const size_t bufbytes = (size_t)pg->stride * ctx->nranks * sizeof(ulonglong2);
        a.gathered_ll = reinterpret_cast<const ulonglong2*>(ctx->arena + ARENA_DATA_OFF + (pg->cur_seq & 1) * bufbytes);
        a.tag = exchange_tag(pg->cur_seq);
        a.fault = exchange_fault(ctx);
    }
    a.rpr = pg->rows_per_rank;
    a.stride = pg->stride;
    a.part = pg->part;
    a.nctas = pg->nctas;
    a.hist_f = pg->hist_f;
    a.hist_ng = pg->hist_ng;
    a.hist_cap = pg->hist_cap;
    a.st = pg->st;
    a.n = pg->n;
    a.svr = pg->svr;
    a.eps = pg->eps;
    a.max_iter = pg->max_iter;
    a.fw_t = pg->fw_t;
    return a;
}

template <int MODE>
static int launch_vec(svmb200_pg* pg, long long k) {
    VecArgs a = make_vec_args(pg);
    const dim3 grid((unsigned)pg->nctas), block(VP_NT);
    cudaStream_t s = pg->ctx->stream;
    if (pg->solver == SOLVER_AL) SVM_CUDA(svm_launch_chained(al_vector_kernel<MODE>, grid, block, s, a, pg->al, (long long)(MODE == VP_INIT ? -1 : k)));
    else if (pg->solver == SOLVER_FW) SVM_CUDA(svm_launch_chained(fw_vector_kernel<MODE>, grid, block, s, a, k));
    else SVM_CUDA(svm_launch_chained(pg_vector_kernel<MODE>, grid, block, s, a, k));
    pg->ctx->launches++;
    return SVMB200_OK;
}

static cudaEvent_t pooled_event(svmb200_ctx* ctx);

// phase: 0 = the whole product; 1 / 2 = its two halves when a single host thread drives several ranks of a symmetric
// sharded solve (tile pass + sends for every rank first, then every rank's combine); for every other solver phase 1 is the
// whole product and phase 2 nothing
static int pg_product(svmb200_pg* pg, bool timed, int phase = 0) {
    // w[row0 : row0+nrows] = Q_shard u, then all ranks exchange their shards (K4)
    svmb200_ctx* ctx = pg->ctx;
    const bool split = pg->pass == PASS_SYMMETRIC && pg->p2p;
    if (phase == 2 && !split) return SVMB200_OK;
    if (phase == 1 && !split) phase = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    if (timed && phase != 2) {
        e0 = pooled_event(ctx);
        e1 = pooled_event(ctx);
        e2 = pooled_event(ctx);
        if (!e0 || !e1 || !e2) {
            svmb200_set_error("cannot create profiling events");
            return SVMB200_ERR_CUDA;
        }
        SVM_CUDA(cudaEventRecord(e0, ctx->stream));
        pg->mv_ev.push_back(e0);
        pg->mv_ev.push_back(e1);
        pg->mv_ev.push_back(e2);
    } else if (timed) {   // second half of a split product: the events of the first half
        e1 = pg->mv_ev[pg->mv_ev.size() - 2];
        e2 = pg->mv_ev[pg->mv_ev.size() - 1];
    }
    ProductOperands op;
    op.Q = pg->dQ;
    op.n = pg->n;
    op.nrows = pg->nrows;
    op.ld = pg->ld;
    op.rpr = pg->rows_per_rank;
    op.u = pg->u;
    op.u_rows = pg->u + pg->row0;
    op.done = &pg->st->done;
    op.phase = phase;
    ExchangeTargets xt;
    if (pg->p2p) {
        // K2 + K4 fused: results go straight into every rank's gathered buffer (parity = seq & 1)
        xt.nranks = ctx->nranks;
        const unsigned long long seq = phase == 2 ? pg->cur_seq : ++ctx->xseq;
        pg->cur_seq = seq;
        xt.tag = exchange_tag(seq);
        const size_t bufbytes = (size_t)pg->stride * ctx->nranks * sizeof(ulonglong2);
        const size_t slot = ARENA_DATA_OFF + (seq & 1) * bufbytes + (size_t)ctx->rank * pg->stride * sizeof(ulonglong2);
        for (int r = 0; r < ctx->nranks; ++r) xt.peer_w[r] = reinterpret_cast<ulonglong2*>(ctx->peer_arena[r] + slot);
        // the plain pointers only carry the slot geometry (w at [0, rpr), shares at [rpr, stride)) in this mode
        op.w = reinterpret_cast<double*>(ctx->arena);
        op.xt = &xt;
        op.seq = seq;
    } else {
        op.w = pg->w + (size_t)ctx->rank * pg->stride;   // this rank's shard, then the all-gather
    }
    op.denpart = op.w + pg->rows_per_rank;
    SVM_TRY(launch_product(ctx, pg->pass, op));
    if (e1 && phase != 1) SVM_CUDA(cudaEventRecord(e1, ctx->stream));
    if (!pg->p2p && ctx->nranks > 1) SVM_TRY(svm_comm_allgather(ctx, pg->w, pg->stride));
    if (e2 && phase != 1) SVM_CUDA(cudaEventRecord(e2, ctx->stream));
    if (phase != 2) pg->last_passes++;
    return SVMB200_OK;
}

static cudaEvent_t pooled_event(svmb200_ctx* ctx) {
    if (ctx->event_pool_used == ctx->event_pool.size()) {
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ctx->event_pool.push_back(e);
    }
    return ctx->event_pool[ctx->event_pool_used++];
}

void svm_release_solver_cache(svmb200_ctx* ctx) {
    for (cudaEvent_t e : ctx->event_pool) cudaEventDestroy(e);
    ctx->event_pool.clear();
    ctx->event_pool_used = 0;
    if (ctx->pg_ev0) cudaEventDestroy(ctx->pg_ev0);
    if (ctx->pg_ev1) cudaEventDestroy(ctx->pg_ev1);
    ctx->pg_ev0 = ctx->pg_ev1 = nullptr;
    for (cudaEvent_t& e : ctx->pg_ev_poll) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
    }
    if (ctx->pg_slab) cudaFree(ctx->pg_slab);
    ctx->pg_slab = nullptr;
    ctx->pg_slab_bytes = 0;
    if (ctx->pg_pinned) cudaFreeHost(ctx->pg_pinned);
    ctx->pg_pinned = nullptr;
}

extern "C" int svmb200_pg_destroy(svmb200_pg* pg) {
    if (!pg) return SVMB200_OK;
    if (pg->ctx) {
        cudaSetDevice(pg->ctx->device);
        cudaStreamSynchronize(pg->ctx->stream);
        if (pg->solver == SOLVER_SMO && pg->hist_f) cudaFree(pg->hist_f);
        if (pg->smo.rows_buf) cudaFree(pg->smo.rows_buf);
        if (pg->smo.shrink.q) cudaFree(const_cast<double*>(pg->smo.shrink.q));
        if (pg->slab_private) {
            if (pg->slab) cudaFree(pg->slab);
            if (pg->pinned) cudaFreeHost(pg->pinned);
            if (pg->ev0) cudaEventDestroy(pg->ev0);
            if (pg->ev1) cudaEventDestroy(pg->ev1);
            for (cudaEvent_t e : pg->ev_poll)
                if (e) cudaEventDestroy(e);
        } else if (pg->slab) {
            pg->ctx->pg_slab_busy = false;  // workspace, pinned block and events go back to the context
            pg->ctx->event_pool_used = 0;
        }
    }
    delete pg;
    return SVMB200_OK;
}

// a solver under construction: destroyed (whatever it holds so far) unless creation succeeds and releases it
struct PgDestroy {
    void operator()(svmb200_pg* pg) const { svmb200_pg_destroy(pg); }
};
using PgGuard = std::unique_ptr<svmb200_pg, PgDestroy>;

// Consecutive regions of one allocation, each rounded up to 256 bytes.  A layout is written once as a sequence of
// take() calls: run on a Carve without a base it sizes the allocation, run on one with the allocation as base it places
// the pointers.
struct Carve {
    unsigned char* base = nullptr;
    size_t bytes = 0;
    template <typename T>
    void take(T*& p, size_t size) {
        p = base ? reinterpret_cast<T*>(base + bytes) : nullptr;
        bytes += (size + 255) & ~size_t(255);
    }
};

// The solver's device slab of `bytes`, pinned poll block and event pair: the context's set, grown as needed, when
// `may_share` and no other solver holds it; else a private set.  svmb200_pg_destroy releases either, also after a
// failure part-way.
static int acquire_workspace(svmb200_pg* pg, size_t bytes, bool may_share) {
    svmb200_ctx* ctx = pg->ctx;
    const bool shared = may_share && !ctx->pg_slab_busy;
    pg->slab_private = !shared;
    if (shared && ctx->pg_slab_bytes < bytes) {
        SVM_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->pg_slab) cudaFree(ctx->pg_slab);
        ctx->pg_slab = nullptr;
        ctx->pg_slab_bytes = 0;
    }
    void*& slab = shared ? ctx->pg_slab : pg->slab;
    void*& pinned = shared ? ctx->pg_pinned : pg->pinned;
    cudaEvent_t& ev0 = shared ? ctx->pg_ev0 : pg->ev0;
    cudaEvent_t& ev1 = shared ? ctx->pg_ev1 : pg->ev1;
    cudaEvent_t* ev_poll = shared ? ctx->pg_ev_poll : pg->ev_poll;
    if (!slab) {
        SVM_CUDA(cudaMalloc(&slab, bytes));
        if (shared) ctx->pg_slab_bytes = bytes;
    }
    if (!pinned) SVM_CUDA(cudaMallocHost(&pinned, 256));
    if (!ev0) SVM_CUDA(cudaEventCreate(&ev0));
    if (!ev1) SVM_CUDA(cudaEventCreate(&ev1));
    for (int i = 0; i < 2; ++i)
        if (!ev_poll[i]) SVM_CUDA(cudaEventCreateWithFlags(&ev_poll[i], cudaEventDisableTiming));
    if (shared) {
        ctx->pg_slab_busy = true;
        ctx->event_pool_used = 0;
        pg->slab = ctx->pg_slab;
        pg->pinned = ctx->pg_pinned;
        pg->ev0 = ctx->pg_ev0;
        pg->ev1 = ctx->pg_ev1;
        pg->ev_poll[0] = ctx->pg_ev_poll[0];
        pg->ev_poll[1] = ctx->pg_ev_poll[1];
    }
    static_assert(sizeof(PGDeviceState) <= POLL_SLOT_BYTES - sizeof(int), "poll slot too small");
    pg->st_host = static_cast<PGDeviceState*>(pg->pinned);
    return SVMB200_OK;
}

// the checks every creator makes first, in this order; `fn` (the creator) prefixes the messages
static int check_create_args(const char* fn, svmb200_ctx* ctx, svmb200_pg** out, bool inputs, int64_t n,
                             const char* too_small, bool ld_ok, const char* ld_msg, int hessian) {
    SVM_TRY(svm_use(ctx));
    const char* msg = nullptr;
    if (out == nullptr) {
        msg = "out is null";
    } else {
        *out = nullptr;
        if (!inputs) msg = "null input";
        else if (n <= 1) msg = too_small;
        else if (!ld_ok) msg = ld_msg;
        else if (hessian != SVMB200_HESSIAN_PLAIN && hessian != SVMB200_HESSIAN_SVR) msg = "bad hessian layout";
    }
    if (msg) {
        svmb200_set_error("%s: %s", fn, msg);
        return SVMB200_ERR_ARG;
    }
    return SVMB200_OK;
}

// The pass of a solver's products, decided at creation and again by svmb200_pg_set_self_gram.  symmetric: the context
// asked for K2s when the solver was created; self_gram: the matrix is a self-Gram svmb200_gram built, exactly symmetric.
//   K2s  one rank holding the whole matrix, or the ranks of a fused peer exchange whose arena also holds the inboxes of
//        the column sums (two parities x P senders x rows_per_rank tagged entries in its upper half)
//   K2e  a self-Gram held whole by one rank, a solver with products (not SMO), a shape K2e covers and a 16-byte aligned
//        matrix; it reads ~60 % of K2's bytes at n = 50 000.  SVMB200_EXACT_SYMV=0 keeps K2 (A/B runs), and so does a
//        scratch for the column chains that cannot be allocated.
//   K2   every other solver.
// The persistent loop (K8) and lockstep batches (K2 x NB) are run modes of their own that bypass the pass.
static ProductPass product_pass(svmb200_pg* pg, bool symmetric, bool self_gram) {
    svmb200_ctx* ctx = pg->ctx;
    const int P = ctx->nranks;
    const bool whole = P == 1 && pg->row0 == 0 && pg->nrows == pg->n;
    const size_t inbox = symv_inbox_off(ctx);
    if (symmetric && (whole || (pg->p2p && ARENA_DATA_OFF + 2 * (size_t)pg->stride * P * sizeof(ulonglong2) <= inbox &&
                                inbox % 16 == 0 && 2 * symv_inbox_bytes(pg->rows_per_rank, P) <= ctx->arena_bytes - inbox)))
        return PASS_SYMMETRIC;
    if (!self_gram || pg->solver == SOLVER_SMO || !whole || !exact_shape_ok(pg->n, pg->ld) || !aligned16(pg->dQ))
        return PASS_FULL;
    const char* ev = getenv("SVMB200_EXACT_SYMV");
    if (ev != nullptr && atoi(ev) == 0) return PASS_FULL;
    if (exact_scratch_reserve(ctx, matvec_scratch(ctx), pg->n, pg->ld) != SVMB200_OK) {
        (void)cudaGetLastError();   // an out-of-memory error is not sticky
        return PASS_FULL;
    }
    return PASS_EXACT;
}

// host-side description of an augmented-Lagrangian solve (SOLVER_AL)
struct ALSpec {
    ALParams p;
    const double* a_host;      // equality row or null
    const double* lr_host;     // epochs step sizes
    const double* mom_host;    // epochs + 1 momenta, or null (= 0)
};

static int bcqp_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows, int hessian,
                       const double* q_host, const double* lb_host, const double* ub_host, const double* x0_host,
                       double eps, int64_t max_iter, SolverKind solver, double fw_t, svmb200_pg** out,
                       const ALSpec* al = nullptr, const double* sign_host = nullptr);

extern "C" int svmb200_pg_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                                 int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                                 const double* x0_host, double eps, int64_t max_iter, svmb200_pg** out) {
    return bcqp_create(ctx, dQ, n, ld, row0, nrows, hessian, q_host, lb_host, ub_host, x0_host, eps, max_iter, SOLVER_PG, 0.0, out);
}

extern "C" int svmb200_fw_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                                 int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                                 const double* x0_host, double eps, int64_t max_iter, double t, svmb200_pg** out) {
    SVM_CHECK_ARG(t >= 0.0 && t < 1.0, "t has to lie in [0, 1)");  // frank_wolfe.py:84-85
    return bcqp_create(ctx, dQ, n, ld, row0, nrows, hessian, q_host, lb_host, ub_host, x0_host, eps, max_iter, SOLVER_FW, t, out);
}

extern "C" int svmb200_pg_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                        int64_t nrows, int hessian, const double* sign_host, const double* q_host,
                                        const double* lb_host, const double* ub_host, const double* x0_host, double eps,
                                        int64_t max_iter, svmb200_pg** out) {
    return bcqp_create(ctx, dQ, n, ld, row0, nrows, hessian, q_host, lb_host, ub_host, x0_host, eps, max_iter, SOLVER_PG, 0.0, out,
                       nullptr, sign_host);
}

extern "C" int svmb200_fw_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                        int64_t nrows, int hessian, const double* sign_host, const double* q_host,
                                        const double* lb_host, const double* ub_host, const double* x0_host, double eps,
                                        int64_t max_iter, double t, svmb200_pg** out) {
    SVM_CHECK_ARG(t >= 0.0 && t < 1.0, "t has to lie in [0, 1)");  // frank_wolfe.py:84-85
    return bcqp_create(ctx, dQ, n, ld, row0, nrows, hessian, q_host, lb_host, ub_host, x0_host, eps, max_iter, SOLVER_FW, t, out,
                       nullptr, sign_host);
}

static int bcqp_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows, int hessian,
                       const double* q_host, const double* lb_host, const double* ub_host, const double* x0_host,
                       double eps, int64_t max_iter, SolverKind solver, double fw_t, svmb200_pg** out, const ALSpec* al,
                       const double* sign_host) {
    // n > 1: opti/_base.py:249-250
    SVM_TRY(check_create_args(__func__, ctx, out, dQ != nullptr && q_host != nullptr && ub_host != nullptr, n, "Q is too small",
                              ld >= n && ld % 2 == 0, "ld must be >= n and even", hessian));
    SVM_CHECK_ARG(max_iter > 0, "max_iter must be > 0");  // opti/_base.py:73-74
    SVM_CHECK_ARG(sign_host == nullptr || hessian == SVMB200_HESSIAN_PLAIN, "label signs need the plain layout");
    if (sign_host != nullptr) {
        for (int64_t i = 0; i < n; ++i) SVM_CHECK_ARG(sign_host[i] == 1.0 || sign_host[i] == -1.0, "signs must be +-1");
    }
    const int P = ctx->nranks;
    const int64_t rpr = rows_per_rank(n, P);
    {
        int64_t exp_row0 = 0, exp_rows = 0;
        SVM_TRY(svmb200_shard_rows(n, ctx->rank, P, &exp_row0, &exp_rows));
        SVM_CHECK_ARG(row0 == exp_row0 && nrows == exp_rows, "row shard does not match svmb200_shard_rows");
    }
    PgGuard guard(new svmb200_pg());
    svmb200_pg* pg = guard.get();
    pg->ctx = ctx;
    pg->dQ = dQ;
    pg->n = n;
    pg->ld = ld;
    pg->row0 = row0;
    pg->nrows = nrows;
    pg->svr = hessian == SVMB200_HESSIAN_SVR;
    pg->nvars = pg->svr ? 2 * n : n;
    pg->rows_per_rank = rpr;
    pg->stride = rpr + rpr / MV_GROUP;
    // The fused exchange double-buffers by sequence parity; that is safe because a rank's vector launch of product
    // s + 1 waits for EVERY peer's shard of s + 1, which a peer only publishes after its own vector launch of s -- so
    // nobody can overwrite a buffer that is still being read.  A rank with an EMPTY shard (the 64-row granularity leaves
    // the last ranks without rows when (P - 1) rows_per_rank >= n: small problems) publishes nothing, nobody waits for it, and it could be lapped and lose entries (found by the
    // multi-rank fuzz on the host emulation).  Such problems use the all-gather, which synchronises all ranks.
    const bool every_rank_owns_rows = (int64_t)(P - 1) * rpr < n;
    pg->p2p = ctx->p2p_enabled && P > 1 && every_rank_owns_rows &&
              ARENA_DATA_OFF + 2 * (size_t)pg->stride * P * sizeof(ulonglong2) <= ctx->arena_bytes;
    pg->nctas = (int)((n + VP_ELEMS - 1) / VP_ELEMS);
    if (pg->nctas > VP_MAXC) pg->nctas = VP_MAXC;
    if (pg->nctas < 1) pg->nctas = 1;
    pg->eps = eps;
    pg->solver = solver;
    pg->pass = product_pass(pg, ctx->symmetric, false);
    pg->fw_t = fw_t;
    pg->max_iter = max_iter;
    pg->hist_cap = max_iter + 1 < (1ll << 24) ? max_iter + 1 : (1ll << 24);
    const size_t nv = (size_t)pg->nvars * sizeof(double);
    const size_t sz_sched = (size_t)(max_iter + 1) * sizeof(double);
    double *sgn = nullptr, *arow = nullptr;
    auto layout = [&](Carve c) {
        // x g d q lb ub signs (nvars each) | u (ld) | gathered (stride*P) | partials | two histories | state
        for (double** v : {&pg->x, &pg->g, &pg->d, &pg->q, &pg->lb, &pg->ub, &sgn}) c.take(*v, nv);
        c.take(pg->u, (size_t)ld * sizeof(double));
        c.take(pg->w, (size_t)(pg->stride * P) * sizeof(double));
        c.take(pg->part, 2 * 3 * VP_MAXC * sizeof(double));
        c.take(pg->hist_f, (size_t)pg->hist_cap * sizeof(double));
        c.take(pg->hist_ng, (size_t)pg->hist_cap * sizeof(double));
        c.take(pg->st, sizeof(PGDeviceState));
        if (solver == SOLVER_AL) {
            // + multipliers, rule state, previous step, pre-jump point, equality row (nvars each), four per-iteration
            // scalar arrays (epochs + 1), double-buffered per-CTA sums, two slots of mu
            ALArgs& A = pg->al;
            for (double** v : {&A.lam_lb, &A.lam_ub, &A.s1, &A.s2, &A.s3, &A.step, &A.xpre, &arow}) c.take(*v, nv);
            for (const double** v : {&A.lr, &A.mom, &A.bc1, &A.bc2}) c.take(*v, sz_sched);
            c.take(A.part, 2 * AL_NSUMS * VP_MAXC * sizeof(double));
            c.take(A.mu, 2 * sizeof(double));
        }
        return c.bytes;
    };
    SVM_TRY(acquire_workspace(pg, layout(Carve{}), true));
    layout(Carve{static_cast<unsigned char*>(pg->slab)});
    pg->sgn = sign_host ? sgn : nullptr;
    if (solver == SOLVER_AL) {
        pg->al.p = al->p;
        pg->al.A = al->a_host ? arow : nullptr;
    }
    cudaStream_t s = ctx->stream;
    SVM_CUDA(cudaMemsetAsync(pg->st, 0, sizeof(PGDeviceState), s));
    SVM_CUDA(cudaMemsetAsync(pg->u, 0, (size_t)ld * sizeof(double), s));
    SVM_CUDA(cudaMemsetAsync(pg->w, 0, (size_t)(pg->stride * P) * sizeof(double), s));
    SVM_CUDA(cudaMemsetAsync(pg->part, 0, 2 * 3 * VP_MAXC * sizeof(double), s));
    SVM_CUDA(cudaMemsetAsync(pg->d, 0, nv, s));
    SVM_CUDA(cudaMemsetAsync(pg->g, 0, nv, s));
    // bounds / start point: opti/constrained/_base.py:61-65 (lb = 0, x0 = (lb+ub)/2)
    std::vector<double> lbv((size_t)pg->nvars, 0.0), x0v((size_t)pg->nvars), u0((size_t)n);
    if (lb_host) memcpy(lbv.data(), lb_host, nv);
    for (int64_t i = 0; i < pg->nvars; ++i) x0v[i] = x0_host ? x0_host[i] : (lbv[i] + ub_host[i]) / 2;
    for (int64_t j = 0; j < n; ++j) u0[j] = pg->svr ? x0v[j] - x0v[j + n] : (sign_host ? sign_host[j] * x0v[j] : x0v[j]);
    SVM_CUDA(cudaMemcpyAsync(pg->q, q_host, nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->ub, ub_host, nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->lb, lbv.data(), nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->x, x0v.data(), nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->u, u0.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, s));
    if (sign_host) SVM_CUDA(cudaMemcpyAsync(pg->sgn, sign_host, nv, cudaMemcpyHostToDevice, s));
    std::vector<double> sched;  // staging of the per-iteration scalars (augmented Lagrangian)
    if (solver == SOLVER_AL) {
        ALArgs& A = pg->al;
        // multipliers, rule state, previous step: zero (rmsprop.py:93 starts its moving mean of g^2 at one)
        SVM_CUDA(cudaMemsetAsync(A.lam_lb, 0, reinterpret_cast<unsigned char*>(arow) - reinterpret_cast<unsigned char*>(A.lam_lb), s));
        SVM_CUDA(cudaMemsetAsync(A.part, 0, 2 * AL_NSUMS * VP_MAXC * sizeof(double), s));
        SVM_CUDA(cudaMemsetAsync(A.mu, 0, 2 * sizeof(double), s));
        const size_t ne = (size_t)max_iter + 1;
        sched.assign(4 * ne, 0.0);
        for (size_t k = 0; k < ne; ++k) {
            sched[k] = al->lr_host[k < (size_t)max_iter ? k : (size_t)max_iter - 1];
            sched[ne + k] = al->mom_host ? al->mom_host[k] : 0.0;
            // adam.py / adamax.py: 1 - beta ** t with t = iter + 1, evaluated with the C library's pow like Python does
            sched[2 * ne + k] = 1.0 - pow(A.p.beta1, (double)(k + 1));
            sched[3 * ne + k] = 1.0 - pow(A.p.beta2, (double)(k + 1));
        }
        SVM_CUDA(cudaMemcpyAsync(const_cast<double*>(A.lr), sched.data(), ne * sizeof(double), cudaMemcpyHostToDevice, s));
        SVM_CUDA(cudaMemcpyAsync(const_cast<double*>(A.mom), sched.data() + ne, ne * sizeof(double), cudaMemcpyHostToDevice, s));
        SVM_CUDA(cudaMemcpyAsync(const_cast<double*>(A.bc1), sched.data() + 2 * ne, ne * sizeof(double), cudaMemcpyHostToDevice, s));
        SVM_CUDA(cudaMemcpyAsync(const_cast<double*>(A.bc2), sched.data() + 3 * ne, ne * sizeof(double), cudaMemcpyHostToDevice, s));
        if (al->a_host) SVM_CUDA(cudaMemcpyAsync(const_cast<double*>(A.A), al->a_host, nv, cudaMemcpyHostToDevice, s));
    }
    SVM_CUDA(cudaStreamSynchronize(s));  // staging vectors go out of scope
    if (solver == SOLVER_AL && pg->al.p.rule == AL_RMSPROP) {
        std::vector<double> ones((size_t)pg->nvars, 1.0);
        SVM_CUDA(cudaMemcpyAsync(pg->al.s1, ones.data(), nv, cudaMemcpyHostToDevice, s));
        SVM_CUDA(cudaStreamSynchronize(s));
    }
    pg->last_passes = 0;
    if (ctx->local_group && P > 1) {
        // one host thread drives every rank: it cannot issue a collective, and a vector launch that waits for a peer's
        // entries must not be enqueued before that peer's product exists in ITS stream order either (the host emulation
        // runs launches synchronously) -- so the first product and INIT are issued for all ranks together, iteration-major,
        // by svmb200_pg_start_group.  No creation barrier is needed: the host has seen every rank's previous solve end.
        if (!pg->p2p) {
            svmb200_set_error("a single-process group needs the fused exchange: every rank must own rows of the matrix "
                              "(n > %lld) and the gathered buffers must fit the arena", (long long)((P - 1) * rpr));
            return SVMB200_ERR_ARG;
        }
        pg->deferred_start = true;
        pg->k_next = 0;
        *out = guard.release();
        return SVMB200_OK;
    }
    if (pg->p2p) {
        // A one-double all-gather, in stream order, before the first fused product of this solver: it completes on a
        // rank only when EVERY rank has reached it, i.e. when every rank's previous solve -- whose last vector launch
        // may still be reading arena regions that this solve's layout overlaps -- has left the arena.  Without it the
        // fused exchange would be correct between two solves only by timing.  (SVMB200_P2P_CREATE_BARRIER=0 removes it
        // for A/B timing; ~30 us per solve.)
        const char* ev = getenv("SVMB200_P2P_CREATE_BARRIER");
        if (ev == nullptr || atoi(ev) != 0) SVM_TRY(svm_comm_allgather(ctx, pg->w, 1));
    }
    // augmented Lagrangian: sums of state 0 (no product needed: every launch of the loop is preceded by its own pass
    // w = Q xe); the others: g0 = Q x0 + q, first direction and its partial reductions
    if (solver != SOLVER_AL) SVM_TRY(pg_product(pg, false));
    SVM_TRY(launch_vec<VP_INIT>(pg, 0));
    pg->k_next = 0;
    *out = guard.release();
    return SVMB200_OK;
}

// A poll is a copy of the device state block (and of the exchange fault flag) into one of two pinned slots, followed by an
// event.  pg_run enqueues the NEXT batch of iterations before it waits for the poll of the previous one, so the stream
// never runs dry while the host looks at the stopping flags (a drained stream costs a launch latency per batch: 2.5 % of
// a C1-sized solve).
static int poll_enqueue(svmb200_pg* pg, int slot) {
    cudaStream_t s = pg->ctx->stream;
    unsigned char* dst = static_cast<unsigned char*>(pg->pinned) + (size_t)slot * POLL_SLOT_BYTES;
    SVM_CUDA(cudaMemcpyAsync(dst, pg->st, sizeof(PGDeviceState), cudaMemcpyDeviceToHost, s));
    int* fault = reinterpret_cast<int*>(dst + POLL_SLOT_BYTES - sizeof(int));
    *fault = 0;
    if (pg->p2p)
        SVM_CUDA(cudaMemcpyAsync(fault, exchange_fault(pg->ctx), sizeof(int), cudaMemcpyDeviceToHost, s));
    SVM_CUDA(cudaEventRecord(pg->ev_poll[slot], s));
    return SVMB200_OK;
}

static int poll_wait(svmb200_pg* pg, int slot) {
    SVM_CUDA(cudaEventSynchronize(pg->ev_poll[slot]));
    unsigned char* src = static_cast<unsigned char*>(pg->pinned) + (size_t)slot * POLL_SLOT_BYTES;
    pg->st_host = reinterpret_cast<PGDeviceState*>(src);
    if (pg->st_host->done) pg->finished = true;
    if (*reinterpret_cast<const int*>(src + POLL_SLOT_BYTES - sizeof(int))) {
        // sticky and context-fatal: the sequence numbers of the ranks can no longer be trusted to agree
        svmb200_set_error("peer exchange timed out: a rank stopped publishing its product shard (the context's "
                          "exchange is unusable from here on: destroy it and every peer's, then start over)");
        return SVMB200_ERR_STATE;
    }
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ persistent small-problem loop
// A projected-gradient solve on one GPU whose matrix fits the shared memory of the SMs (n <= 2 016 on a B200) runs as
// ONE cooperative launch (k_persistent.cuh) instead of two launches per iteration.  Same bits; SVMB200_PERSISTENT=0
// keeps the two-kernel loop (A/B), SVMB200_PERSISTENT_GRID overrides the grid size (tests on the host emulation).
// dynamic shared memory the cooperative kernels (this loop and SMO) may use: their static arrays take the rest of the 227 KB
constexpr size_t COOP_SMEM_MAX = 221 * 1024;

// Ready a cooperative launch of `kernel` on `grid` CTAs of `block` threads and `smem` bytes of dynamic shared memory: the
// opt-in to COOP_SMEM_MAX, the check that such a grid can be co-resident (it cannot on a partitioned GPU), and the
// context's grid barrier.  *fits tells whether the grid can run.
template <auto kernel>
static int cooperative_setup(svmb200_ctx* ctx, int grid, int block, size_t smem, bool* fits) {
    *fits = true;
#ifndef SVMB200_HOST_EMULATION
    SVM_TRY(svm_opt_in_smem<kernel>(ctx, (int)COOP_SMEM_MAX));
    int per_sm = 0;
    SVM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
    *fits = (long long)per_sm * ctx->sm_count >= grid;
#endif
    if (*fits && !ctx->gbar) {
        SVM_CUDA(cudaMalloc(&ctx->gbar, 256));
        SVM_CUDA(cudaMemsetAsync(ctx->gbar, 0, 256, ctx->stream));
    }
    return SVMB200_OK;
}

struct PersistPlan {
    int grid = 0, rows_per_cta = 0;
    size_t smem = 0;
};

static bool persistent_plan(const svmb200_pg* pg, int64_t budget, PersistPlan* plan) {
    static const int enabled = [] {
        const char* ev = getenv("SVMB200_PERSISTENT");
        return ev == nullptr ? 1 : atoi(ev);
    }();
    const svmb200_ctx* ctx = pg->ctx;
    if (!enabled || pg->solver != SOLVER_PG || ctx->nranks != 1 || pg->profile || budget < 8) return false;
    if (pg->svr || pg->sgn != nullptr) return false;  // plain layout, no label-sign view (k_persistent.cuh)
    if (pg->ld > 2 * PK_NT * PK_UMAX || pg->nrows != pg->n) return false;
    int grid = ctx->sm_count;
    if (const char* ev = getenv("SVMB200_PERSISTENT_GRID")) grid = atoi(ev);
    if (grid < 1 || grid < pg->nctas) return false;
    const int64_t rows = (pg->n + grid - 1) / grid;
    const size_t smem = (size_t)rows * pg->ld * sizeof(double);
    if (rows > PK_RMAX || smem > COOP_SMEM_MAX || pg->nctas > PK_VMAX) return false;
    plan->grid = grid;
    plan->rows_per_cta = (int)rows;
    plan->smem = smem;
    return true;
}

static int launch_persistent(svmb200_pg* pg, const PersistPlan& plan, int64_t niter) {
    svmb200_ctx* ctx = pg->ctx;
    // scratch: two w buffers, two product buffers, grid - 1 private copies of u (ld each)
    const size_t doubles = 4 * (size_t)pg->ld + (size_t)(plan.grid - 1) * (size_t)pg->ld;
    SVM_TRY(svm_scratch_reserve(ctx, &ctx->persist_buf, &ctx->persist_bytes, doubles * sizeof(double)));
    bool fits = false;
    SVM_TRY(cooperative_setup<pg_persistent_kernel>(ctx, plan.grid, PK_NT, plan.smem, &fits));
    if (!fits) {
        svmb200_set_error("persistent loop: %d CTAs cannot be co-resident", plan.grid);
        return SVMB200_ERR_STATE;
    }
    PersistArgs a;
    a.Q = pg->dQ;
    a.ld = pg->ld;
    a.n = pg->n;
    a.rows_per_cta = plan.rows_per_cta;
    a.wbuf = static_cast<double*>(ctx->persist_buf);
    a.prod = a.wbuf + 2 * pg->ld;
    a.priv = a.wbuf + 4 * pg->ld;
    a.gbar = ctx->gbar;
    a.v = make_vec_args(pg);
    a.k0 = pg->k_next;
    a.niter = niter;
    SVM_CUDA(svm_launch_cooperative(pg_persistent_kernel, dim3((unsigned)plan.grid), dim3(PK_NT), plan.smem, ctx->stream, a));
    ctx->launches++;
    return SVMB200_OK;
}

// statistics of the run about to start (pooled profiling events: reused, never destroyed per run)
static void reset_run_stats(svmb200_pg* pg) {
    pg->mv_ev.clear();
    pg->last_passes = 0;
    pg->last_samples = 0;
    pg->last_ms = pg->last_mv_ms = pg->last_comm_ms = pg->last_vec_ms = 0.f;
}

// The ranks of a single-process group (count > 1), or one solver (count == 1): `max_new` more iterations (< 0: to the
// end).  Launches are enqueued ITERATION-MAJOR over the ranks -- every rank's product k, then every rank's vector launch
// k -- so that in each stream a launch that waits for a peer's entries comes after that peer's product has been
// enqueued in its own stream; the ranks' state is replicated, so they stop together.
static int run_many(svmb200_pg* const* pgs, int count, int64_t max_new) {
    svmb200_pg* p0 = pgs[0];
    for (int r = 0; r < count; ++r) {
        svmb200_pg* pg = pgs[r];
        SVM_TRY(svm_use(pg->ctx));
        if (r == 0) pg->ctx->event_pool_used = 0;
        reset_run_stats(pg);
        SVM_CUDA(cudaEventRecord(pg->ev0, pg->ctx->stream));
    }
    if (!p0->finished) {
        const bool to_end = max_new < 0;
        int64_t budget = to_end ? (p0->max_iter - p0->k_next) : max_new;
        if (budget > p0->max_iter - p0->k_next) budget = p0->max_iter - p0->k_next;
        // enqueue in batches; the device-side done flag turns the remainder of a batch (and the batch enqueued behind it
        // before its poll came back) into no-ops
        const int64_t BATCH = 64;
        int pending = -1, slot = 0;
        int rc = SVMB200_OK;
        PersistPlan plan;
        if (count == 1 && persistent_plan(p0, budget, &plan)) {
            // one cooperative launch runs the whole budget (it leaves early when the stopping test fires)
            const int64_t k0 = p0->k_next;
            if (launch_persistent(p0, plan, budget) == SVMB200_OK) {
                rc = poll_enqueue(p0, 0);
                if (rc == SVMB200_OK) rc = poll_wait(p0, 0);
                SVM_TRY(rc);
                p0->k_next = p0->finished ? p0->st_host->iter : k0 + budget;
                p0->last_passes += p0->k_next - k0;
                budget = 0;
            } else {
                cudaGetLastError();  // the launch was refused (nothing ran): the two-kernel loop below takes over
            }
        }
        while (budget > 0 && !p0->finished && rc == SVMB200_OK) {
            const int64_t nb = budget < BATCH ? budget : BATCH;
            for (int64_t i = 0; i < nb && rc == SVMB200_OK; ++i) {
                // profiling events serialise the programmatic launches around them: sample one iteration in PROFILE_STRIDE
                // (rank 0 only)
                const bool sample = p0->profile && (p0->k_next % PROFILE_STRIDE) == 0;
                for (int ph = count > 1 ? 1 : 0; ph <= (count > 1 ? 2 : 0) && rc == SVMB200_OK; ++ph)
                    for (int r = 0; r < count && rc == SVMB200_OK; ++r) {
                        if (count > 1) rc = svm_use(pgs[r]->ctx);
                        if (rc == SVMB200_OK) rc = pg_product(pgs[r], sample && r == 0, ph);
                    }
                for (int r = 0; r < count && rc == SVMB200_OK; ++r) {
                    if (count > 1) rc = svm_use(pgs[r]->ctx);
                    if (rc == SVMB200_OK) rc = launch_vec<VP_STEP>(pgs[r], pgs[r]->k_next);
                    if (rc == SVMB200_OK && sample && r == 0) {
                        cudaEvent_t e3 = pooled_event(p0->ctx);
                        if (!e3) {
                            svmb200_set_error("cannot create profiling events");
                            rc = SVMB200_ERR_CUDA;
                        } else if (cudaEventRecord(e3, p0->ctx->stream) != cudaSuccess) {
                            svmb200_set_error("cudaEventRecord failed");
                            rc = SVMB200_ERR_CUDA;
                        } else {
                            p0->mv_ev.push_back(e3);
                            p0->last_samples++;
                        }
                    }
                    pgs[r]->k_next++;
                }
            }
            budget -= nb;
            for (int r = 0; r < count && rc == SVMB200_OK; ++r) {
                if (count > 1) rc = svm_use(pgs[r]->ctx);
                if (rc == SVMB200_OK) rc = poll_enqueue(pgs[r], slot);
            }
            if (pending >= 0)  // the batch BEFORE the one just enqueued
                for (int r = 0; r < count && rc == SVMB200_OK; ++r) rc = poll_wait(pgs[r], pending);
            pending = slot;
            slot ^= 1;
        }
        if (pending >= 0) {
            // the last poll is always collected: its copy targets pinned memory that outlives this call
            for (int r = 0; r < count; ++r) {
                const int rc2 = poll_wait(pgs[r], pending);
                if (rc == SVMB200_OK) rc = rc2;
            }
        }
        SVM_TRY(rc);
        for (int r = 0; r < count; ++r) {
            if (pgs[r]->finished != p0->finished) {
                svmb200_set_error("the ranks of a group disagree on the stopping test (replicated state diverged)");
                return SVMB200_ERR_STATE;
            }
            if (pgs[r]->finished) pgs[r]->k_next = pgs[r]->st_host->iter;
        }
        if (!p0->finished) {
            // make the state at callback point k_next visible (f, |d|, stopping tests); the augmented Lagrangian
            // needs w = Q xe for that (value and gradient at xe), the box-constrained solvers carry g along
            if (p0->solver == SOLVER_AL)
                for (int ph = count > 1 ? 1 : 0; ph <= (count > 1 ? 2 : 0); ++ph)
                    for (int r = 0; r < count; ++r) {
                        SVM_TRY(svm_use(pgs[r]->ctx));
                        SVM_TRY(pg_product(pgs[r], false, ph));
                    }
            for (int r = 0; r < count; ++r) {
                SVM_TRY(svm_use(pgs[r]->ctx));
                SVM_TRY(launch_vec<VP_FINALISE>(pgs[r], pgs[r]->k_next));
                SVM_TRY(poll_enqueue(pgs[r], 0));
            }
            for (int r = 0; r < count; ++r) SVM_TRY(poll_wait(pgs[r], 0));
        }
    }
    for (int r = 0; r < count; ++r) {
        svmb200_pg* pg = pgs[r];
        SVM_TRY(svm_use(pg->ctx));
        SVM_CUDA(cudaEventRecord(pg->ev1, pg->ctx->stream));
    }
    for (int r = 0; r < count; ++r) {
        svmb200_pg* pg = pgs[r];
        SVM_CUDA(cudaEventSynchronize(pg->ev1));
        SVM_CUDA(cudaEventElapsedTime(&pg->last_ms, pg->ev0, pg->ev1));
    }
    for (size_t i = 0; i + 3 < p0->mv_ev.size(); i += 4) {
        float ms = 0.f;
        SVM_CUDA(cudaEventElapsedTime(&ms, p0->mv_ev[i], p0->mv_ev[i + 1]));
        p0->last_mv_ms += ms;
        SVM_CUDA(cudaEventElapsedTime(&ms, p0->mv_ev[i + 1], p0->mv_ev[i + 2]));
        p0->last_comm_ms += ms;
        SVM_CUDA(cudaEventElapsedTime(&ms, p0->mv_ev[i + 2], p0->mv_ev[i + 3]));
        p0->last_vec_ms += ms;
    }
    return SVMB200_OK;
}

static int smo_run(svmb200_pg* pg, int64_t max_new);

extern "C" int svmb200_pg_run(svmb200_pg* pg, int64_t max_new, int64_t* iter, int* status) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    SVM_CHECK_ARG(!pg->deferred_start, "a solver of a single-process group runs through svmb200_pg_run_group");
    SVM_TRY(pg->solver == SOLVER_SMO ? smo_run(pg, max_new) : run_many(&pg, 1, max_new));
    if (iter) *iter = pg->st_host->iter;
    if (status) *status = pg->st_host->done ? pg->st_host->status : SVMB200_STATUS_UNKNOWN;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ single-process group
static int check_group(svmb200_pg* const* pgs, int count) {
    SVM_CHECK_ARG(pgs != nullptr && count >= 1 && count <= SVM_MAX_RANKS, "bad argument");
    for (int r = 0; r < count; ++r) {
        const svmb200_pg* p = pgs[r];
        SVM_CHECK_ARG(p != nullptr && p->ctx != nullptr, "null solver");
        SVM_CHECK_ARG(p->solver != SOLVER_SMO, "an SMO solver runs through svmb200_pg_run");
        SVM_CHECK_ARG(p->ctx->local_group && p->ctx->nranks == count && p->ctx->rank == r,
                      "pass one solver per rank of the single-process group, in rank order");
        SVM_CHECK_ARG(p->n == pgs[0]->n && p->solver == pgs[0]->solver && p->max_iter == pgs[0]->max_iter &&
                          p->svr == pgs[0]->svr && p->k_next == pgs[0]->k_next,
                      "the solvers of a group must pose the same problem and be in the same state");
    }
    return SVMB200_OK;
}

// first product (g0 = Q x0 + q) and INIT launch of solvers that were created on the ranks of a single-process group
extern "C" int svmb200_pg_start_group(svmb200_pg* const* pgs, int count) {
    SVM_TRY(check_group(pgs, count));
    for (int r = 0; r < count; ++r) SVM_CHECK_ARG(pgs[r]->deferred_start, "solver already started");
    if (pgs[0]->solver != SOLVER_AL)
        for (int ph = 1; ph <= 2; ++ph)
            for (int r = 0; r < count; ++r) {
                SVM_TRY(svm_use(pgs[r]->ctx));
                SVM_TRY(pg_product(pgs[r], false, ph));
            }
    for (int r = 0; r < count; ++r) {
        SVM_TRY(svm_use(pgs[r]->ctx));
        SVM_TRY(launch_vec<VP_INIT>(pgs[r], 0));
        pgs[r]->deferred_start = false;
    }
    return SVMB200_OK;
}

// svmb200_pg_run for every rank of a single-process group at once (one host thread, no collective): iter / status are
// those of the replicated state
extern "C" int svmb200_pg_run_group(svmb200_pg* const* pgs, int count, int64_t max_new, int64_t* iter, int* status) {
    SVM_TRY(check_group(pgs, count));
    for (int r = 0; r < count; ++r) SVM_CHECK_ARG(!pgs[r]->deferred_start, "call svmb200_pg_start_group first");
    SVM_TRY(run_many(pgs, count, max_new));
    if (iter) *iter = pgs[0]->st_host->iter;
    if (status) *status = pgs[0]->st_host->done ? pgs[0]->st_host->status : SVMB200_STATUS_UNKNOWN;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ batched driver
// `count` solvers of one kind that share the resident matrix (same context, shard, layout and iteration limit) run
// to termination in lockstep (SURVEY.md 8f-4): per iteration ceil(count / MV_MULTI_MAX) passes over the matrix
// instead of `count`, and one vector launch for all problems.  Every problem keeps its own state, histories and
// stopping tests -- one that finishes early ignores the remaining launches -- and, because the multi-vector pass
// reproduces the single-vector reductions bit for bit, ends exactly where its own svmb200_pg_run would have.
// Multi-GPU: the fused peer exchange of the single solves carries over -- K2 x NB stores every problem's shard into
// every rank's arena as tagged entries, the vector launch waits on the entries it reads; one sequence number (tag,
// buffer parity) per iteration for the whole batch.  The batch has its own arena region behind the two buffers of
// the single-solver layout (whose last reader, a member's INIT launch, may still be running on a slower rank when
// the first batched product of a faster rank arrives).  Without peer access: one ncclAllGather per problem.
struct BatchExchange {
    bool p2p = false;
    size_t base = 0;        // arena offset of the batch region
    size_t bufbytes = 0;    // one problem's gathered buffer (stride * nranks tagged entries)
    unsigned long long seq = 0;
};

static int batch_product(svmb200_ctx* ctx, svmb200_pg* const* pgs, int count, BatchExchange& bx) {
    const int nlaunch = (count + MV_MULTI_MAX - 1) / MV_MULTI_MAX;
    svmb200_pg* p0 = pgs[0];
    if (bx.p2p) bx.seq = ++ctx->xseq;
    for (int l = 0, b0 = 0; l < nlaunch; ++l) {
        const int nb = (count - b0 + (nlaunch - l) - 1) / (nlaunch - l);  // balanced split
        const double* du[MV_MULTI_MAX];
        double* dw[MV_MULTI_MAX];
        const double* dur[MV_MULTI_MAX];
        double* dden[MV_MULTI_MAX];
        const int* ddone[MV_MULTI_MAX];
        for (int i = 0; i < nb; ++i) {
            svmb200_pg* pg = pgs[b0 + i];
            double* wshard = pg->w + (size_t)ctx->rank * pg->stride;
            du[i] = pg->u;
            dw[i] = wshard;
            dur[i] = pg->u + pg->row0;
            dden[i] = wshard + pg->rows_per_rank;
            ddone[i] = &pg->st->done;
        }
        if (bx.p2p) {
            ExchangeTargets xt;
            xt.nranks = ctx->nranks;
            xt.tag = exchange_tag(bx.seq);
            // this rank's slot of problem b0 in the parity copy of the batch region, in every rank's arena
            const size_t slot = bx.base + (bx.seq & 1) * (size_t)count * bx.bufbytes + (size_t)b0 * bx.bufbytes +
                                (size_t)ctx->rank * p0->stride * sizeof(ulonglong2);
            for (int r = 0; r < ctx->nranks; ++r) xt.peer_w[r] = reinterpret_cast<ulonglong2*>(ctx->peer_arena[r] + slot);
            SVM_TRY(launch_matvec_multi(ctx, p0->dQ, p0->nrows, p0->ld, nb, du, dw, dur, dden, ddone, &xt,
                                        (long long)(bx.bufbytes / sizeof(ulonglong2)), (long long)p0->rows_per_rank));
        } else {
            SVM_TRY(launch_matvec_multi(ctx, p0->dQ, p0->nrows, p0->ld, nb, du, dw, dur, dden, ddone));
        }
        b0 += nb;
    }
    if (!bx.p2p && ctx->nranks > 1) {
        for (int b = 0; b < count; ++b) SVM_TRY(svm_comm_allgather(ctx, pgs[b]->w, pgs[b]->stride));
    }
    for (int b = 0; b < count; ++b) pgs[b]->last_passes += nlaunch;
    return SVMB200_OK;
}

template <int MODE>
static int launch_vec_batch(svmb200_ctx* ctx, SolverKind solver, int nctas, int count, const VecArgs* dva, const ALArgs* dal,
                            long long k, const BatchExchange& bx) {
    const dim3 grid((unsigned)nctas, (unsigned)count);
    const unsigned tag = bx.p2p ? exchange_tag(bx.seq) : 0u;
    const int parity = bx.p2p ? (int)(bx.seq & 1) : 0;
    const dim3 block(VP_NT);
    if (solver == SOLVER_AL) SVM_CUDA(svm_launch_chained(al_vector_batch_kernel<MODE>, grid, block, ctx->stream, dva, dal, k, tag, parity));
    else if (solver == SOLVER_FW) SVM_CUDA(svm_launch_chained(fw_vector_batch_kernel<MODE>, grid, block, ctx->stream, dva, k, tag, parity));
    else SVM_CUDA(svm_launch_chained(pg_vector_batch_kernel<MODE>, grid, block, ctx->stream, dva, k, tag, parity));
    ctx->launches++;
    return SVMB200_OK;
}

// one copy per problem, one synchronisation; returns the number of problems still running
static int batch_poll(svmb200_ctx* ctx, svmb200_pg* const* pgs, int count, int* running, const BatchExchange& bx) {
    for (int b = 0; b < count; ++b)
        SVM_CUDA(cudaMemcpyAsync(pgs[b]->st_host, pgs[b]->st, sizeof(PGDeviceState), cudaMemcpyDeviceToHost, ctx->stream));
    SVM_CUDA(cudaStreamSynchronize(ctx->stream));
    if (bx.p2p) {
        int fault = 0;
        SVM_CUDA(cudaMemcpy(&fault, exchange_fault(ctx), sizeof(int), cudaMemcpyDeviceToHost));
        if (fault) {
            svmb200_set_error("peer exchange timed out: a rank stopped publishing its product shards");
            return SVMB200_ERR_STATE;
        }
    }
    int r = 0;
    for (int b = 0; b < count; ++b) {
        if (pgs[b]->st_host->done) pgs[b]->finished = true;
        else ++r;
    }
    *running = r;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_run_batch(svmb200_pg* const* pgs, int count, int64_t* iters, int* statuses) {
    SVM_CHECK_ARG(pgs != nullptr && count >= 1 && count <= 65535, "bad argument");
    svmb200_pg* p0 = pgs[0];
    for (int b = 0; b < count; ++b) {
        const svmb200_pg* p = pgs[b];
        SVM_CHECK_ARG(p != nullptr, "null solver");
        SVM_CHECK_ARG(p->solver != SOLVER_SMO, "SMO solvers have no lockstep batch: run them one by one");
        SVM_CHECK_ARG(p->ctx == p0->ctx && p->dQ == p0->dQ && p->n == p0->n && p->ld == p0->ld && p->row0 == p0->row0 &&
                          p->nrows == p0->nrows && p->svr == p0->svr,
                      "the solvers of a batch must share the resident matrix, its shard and its layout");
        SVM_CHECK_ARG(p->solver == p0->solver && p->max_iter == p0->max_iter,
                      "the solvers of a batch must be of one kind and share the iteration limit");
        SVM_CHECK_ARG(p->k_next == 0 && !p->finished, "a batch takes solvers that have not run yet");
        SVM_CHECK_ARG(!p->deferred_start, "lockstep batches are not available on a single-process group");
        for (int c = 0; c < b; ++c) SVM_CHECK_ARG(pgs[c] != p, "a solver is listed twice");
    }
    svmb200_ctx* ctx = p0->ctx;
    SVM_TRY(svm_use(ctx));
    // fused peer exchange when every member was created with it and the batch region fits the arena (the same
    // decision on every rank: it depends on sizes only)
    BatchExchange bx;
    bx.bufbytes = (size_t)p0->stride * ctx->nranks * sizeof(ulonglong2);
    bx.base = ARENA_DATA_OFF + 2 * bx.bufbytes;
    bx.p2p = ctx->p2p_enabled && ctx->nranks > 1 && bx.base + 2 * (size_t)count * bx.bufbytes <= ctx->arena_bytes;
    for (int b = 0; b < count; ++b) bx.p2p = bx.p2p && pgs[b]->p2p;
    // per-problem slab pointers differ, so every problem needs its own pinned state block (the context owns one)
    for (int b = 0; b < count; ++b) {
        pgs[b]->p2p = false;  // the members' own (single-solver) exchange path is not used from here on
        for (int c = 0; c < b; ++c) SVM_CHECK_ARG(pgs[c]->st_host != pgs[b]->st_host, "solvers share a state block");
        reset_run_stats(pgs[b]);
    }
    // argument blocks of the vector kernels (constant over the run: only k changes from launch to launch)
    const SolverKind solver = p0->solver;
    const size_t va_bytes = ((size_t)count * sizeof(VecArgs) + 255) & ~size_t(255);
    const size_t al_bytes = solver == SOLVER_AL ? (((size_t)count * sizeof(ALArgs) + 255) & ~size_t(255)) : 0;
    SVM_TRY(svm_scratch_reserve(ctx, &ctx->batch_buf, &ctx->batch_bytes, va_bytes + al_bytes));
    VecArgs* dva = static_cast<VecArgs*>(ctx->batch_buf);
    ALArgs* dal = solver == SOLVER_AL ? reinterpret_cast<ALArgs*>(static_cast<unsigned char*>(ctx->batch_buf) + va_bytes) : nullptr;
    {
        std::vector<VecArgs> hv((size_t)count);
        for (int b = 0; b < count; ++b) {
            hv[b] = make_vec_args(pgs[b]);
            if (bx.p2p) {
                hv[b].gathered_ll = reinterpret_cast<const ulonglong2*>(ctx->arena + bx.base + (size_t)b * bx.bufbytes);
                hv[b].ll_pstride = (long long)((size_t)count * bx.bufbytes / sizeof(ulonglong2));
                hv[b].fault = exchange_fault(ctx);
            }
        }
        SVM_CUDA(cudaMemcpyAsync(dva, hv.data(), (size_t)count * sizeof(VecArgs), cudaMemcpyHostToDevice, ctx->stream));
        if (solver == SOLVER_AL) {
            std::vector<ALArgs> ha((size_t)count);
            for (int b = 0; b < count; ++b) ha[b] = pgs[b]->al;
            SVM_CUDA(cudaMemcpyAsync(dal, ha.data(), (size_t)count * sizeof(ALArgs), cudaMemcpyHostToDevice, ctx->stream));
        }
        SVM_CUDA(cudaStreamSynchronize(ctx->stream));  // staging vectors go out of scope
    }
    SVM_CUDA(cudaEventRecord(p0->ev0, ctx->stream));
    const int64_t max_iter = p0->max_iter;
    int64_t k = 0;
    int running = count;
    const int64_t BATCH = 64;  // iterations enqueued between two looks at the done flags
    while (k < max_iter && running > 0) {
        const int64_t nb = max_iter - k < BATCH ? max_iter - k : BATCH;
        for (int64_t i = 0; i < nb; ++i, ++k) {
            SVM_TRY(batch_product(ctx, pgs, count, bx));
            SVM_TRY(launch_vec_batch<VP_STEP>(ctx, solver, p0->nctas, count, dva, dal, k, bx));
        }
        SVM_TRY(batch_poll(ctx, pgs, count, &running, bx));
    }
    if (running > 0) {
        // state at callback point max_iter (see svmb200_pg_run): the epoch / iteration limit ends every problem left
        if (solver == SOLVER_AL) SVM_TRY(batch_product(ctx, pgs, count, bx));
        SVM_TRY(launch_vec_batch<VP_FINALISE>(ctx, solver, p0->nctas, count, dva, dal, k, bx));
        SVM_TRY(batch_poll(ctx, pgs, count, &running, bx));
    }
    SVM_CUDA(cudaEventRecord(p0->ev1, ctx->stream));
    SVM_CUDA(cudaEventSynchronize(p0->ev1));
    float ms = 0.f;
    SVM_CUDA(cudaEventElapsedTime(&ms, p0->ev0, p0->ev1));
    for (int b = 0; b < count; ++b) {
        svmb200_pg* pg = pgs[b];
        pg->last_ms = ms;  // device time of the whole batch
        pg->k_next = pg->finished ? pg->st_host->iter : k;
        if (iters) iters[b] = pg->st_host->iter;
        if (statuses) statuses[b] = pg->st_host->done ? pg->st_host->status : SVMB200_STATUS_UNKNOWN;
    }
    if (running > 0) {
        svmb200_set_error("batched solve: %d problem(s) did not reach a stopping test", running);
        return SVMB200_ERR_STATE;
    }
    return SVMB200_OK;
}

// the device state block into st_host, once the work enqueued so far is done
static int pull_state(svmb200_pg* pg) {
    SVM_TRY(svm_use(pg->ctx));
    SVM_CUDA(cudaMemcpyAsync(pg->st_host, pg->st, sizeof(PGDeviceState), cudaMemcpyDeviceToHost, pg->ctx->stream));
    SVM_CUDA(cudaStreamSynchronize(pg->ctx->stream));
    return SVMB200_OK;
}

extern "C" int svmb200_pg_state(svmb200_pg* pg, double* x_host, double* g_host, double* f, double* ng) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    SVM_TRY(pull_state(pg));
    cudaStream_t s = pg->ctx->stream;
    const size_t nv = (size_t)pg->nvars * sizeof(double);
    // augmented Lagrangian with Nesterov momentum: the device iterate is the next evaluation point (jump included);
    // when the optimality test ends the run the reference has not taken that jump yet
    const bool pre_jump = pg->solver == SOLVER_AL && pg->al.p.momentum_type == AL_MOM_NESTEROV && pg->st_host->done &&
                          pg->st_host->status == SVMB200_STATUS_OPTIMAL;
    if (x_host) SVM_CUDA(cudaMemcpyAsync(x_host, pre_jump ? pg->al.xpre : pg->x, nv, cudaMemcpyDeviceToHost, s));
    if (g_host) SVM_CUDA(cudaMemcpyAsync(g_host, pg->g, nv, cudaMemcpyDeviceToHost, s));
    SVM_CUDA(cudaStreamSynchronize(s));
    if (f) *f = pg->st_host->f;
    if (ng) *ng = pg->st_host->ng;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_scalars(svmb200_pg* pg, double* vals6) {
    SVM_CHECK_ARG(pg != nullptr && vals6 != nullptr, "null argument");
    SVM_TRY(pull_state(pg));
    vals6[0] = pg->st_host->f;
    vals6[1] = pg->st_host->ng;
    vals6[2] = pg->st_host->s;
    vals6[3] = pg->st_host->maxt;
    vals6[4] = pg->st_host->t;
    vals6[5] = pg->st_host->den;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_history(svmb200_pg* pg, double* f_hist_host, double* ng_hist_host, int64_t* count) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    SVM_TRY(pull_state(pg));
    cudaStream_t s = pg->ctx->stream;
    int64_t cnt = pg->st_host->iter + 1;
    if (cnt > pg->hist_cap) cnt = pg->hist_cap;
    if (f_hist_host) SVM_CUDA(cudaMemcpyAsync(f_hist_host, pg->hist_f, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (ng_hist_host) SVM_CUDA(cudaMemcpyAsync(ng_hist_host, pg->hist_ng, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, s));
    SVM_CUDA(cudaStreamSynchronize(s));
    if (count) *count = cnt;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_stats(svmb200_pg* pg, float* ms, int64_t* passes, float* matvec_ms) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    if (ms) *ms = pg->last_ms;
    if (passes) *passes = pg->last_passes;
    if (matvec_ms) *matvec_ms = pg->last_mv_ms;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_stats_ex(svmb200_pg* pg, float* matvec_ms, float* comm_ms, float* vector_ms) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    if (matvec_ms) *matvec_ms = pg->last_mv_ms;
    if (comm_ms) *comm_ms = pg->last_comm_ms;
    if (vector_ms) *vector_ms = pg->last_vec_ms;
    return SVMB200_OK;
}

// iterations of the last svmb200_pg_run whose launches were bracketed by CUDA events (profiling samples one iteration
// in 16: the events serialise the programmatic launches around them); the *_ms sums of svmb200_pg_stats_ex cover these
extern "C" int svmb200_pg_profile_samples(svmb200_pg* pg, int64_t* samples) {
    SVM_CHECK_ARG(pg != nullptr && samples != nullptr, "null argument");
    *samples = pg->last_samples;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_set_profile(svmb200_pg* pg, int on) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    pg->profile = on != 0;
    return SVMB200_OK;
}

// 1 when the solver's products come from the upper triangle alone (svmb200_ctx_set_symmetric was on at its creation and
// it holds the whole matrix on one rank, or exchanges its shard through the peer arena)
extern "C" int svmb200_pg_is_symmetric(svmb200_pg* pg, int* on) {
    SVM_CHECK_ARG(pg != nullptr && on != nullptr, "null argument");
    *on = pg->pass == PASS_SYMMETRIC ? 1 : 0;
    return SVMB200_OK;
}

// The solver's matrix is a self-Gram svmb200_gram built (same = 1): exactly symmetric, and the solver may take K2e
// (product_pass).  Products already taken by K2 (the first one, at creation) have the same bits.
extern "C" int svmb200_pg_set_self_gram(svmb200_pg* pg, int on) {
    SVM_CHECK_ARG(pg != nullptr, "null solver");
    SVM_TRY(svm_use(pg->ctx));
    pg->pass = product_pass(pg, pg->pass == PASS_SYMMETRIC, on != 0);
    return SVMB200_OK;
}

extern "C" int svmb200_pg_is_exact_symv(svmb200_pg* pg, int* on) {
    SVM_CHECK_ARG(pg != nullptr && on != nullptr, "null argument");
    *on = pg->pass == PASS_EXACT ? 1 : 0;
    return SVMB200_OK;
}

extern "C" int svmb200_pg_device_x(svmb200_pg* pg, double** dx) {
    SVM_CHECK_ARG(pg != nullptr && dx != nullptr, "null argument");
    *dx = pg->x;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ augmented Lagrangian API
extern "C" int svmb200_al_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                                 int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                                 const double* x0_host, const double* a_host, double b, double rho, int rule,
                                 int momentum_type, const double* step_sizes, const double* momenta, double decay,
                                 double beta1, double beta2, double offset, double tol, int64_t epochs, svmb200_pg** out) {
    return svmb200_al_create_signed(ctx, dQ, n, ld, row0, nrows, hessian, nullptr, q_host, lb_host, ub_host, x0_host, a_host,
                                    b, rho, rule, momentum_type, step_sizes, momenta, decay, beta1, beta2, offset, tol,
                                    epochs, out);
}

extern "C" int svmb200_al_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                        int64_t nrows, int hessian, const double* sign_host, const double* q_host,
                                        const double* lb_host, const double* ub_host, const double* x0_host,
                                        const double* a_host, double b, double rho, int rule, int momentum_type,
                                        const double* step_sizes, const double* momenta, double decay, double beta1,
                                        double beta2, double offset, double tol, int64_t epochs, svmb200_pg** out) {
    SVM_CHECK_ARG(x0_host != nullptr, "the start point is required (opti/_base.py:36-60 draws it on the host)");
    SVM_CHECK_ARG(step_sizes != nullptr, "step_sizes is null");
    SVM_CHECK_ARG(rho > 0.0, "rho must be must > 0");                       // constrained/_base.py:276-277
    SVM_CHECK_ARG(rule >= AL_ADAGRAD && rule <= AL_ADAMAX, "unknown update rule");
    SVM_CHECK_ARG(momentum_type >= AL_MOM_NONE && momentum_type <= AL_MOM_NESTEROV, "unknown momentum type");
    SVM_CHECK_ARG(momentum_type == AL_MOM_NONE || (rule != AL_ADAGRAD && rule != AL_ADADELTA),
                  "AdaGrad and AdaDelta take no momentum");
    SVM_CHECK_ARG(momentum_type == AL_MOM_NONE || momenta != nullptr, "momenta is null");
    SVM_CHECK_ARG(offset > 0.0, "offset must be > 0");                      // adagrad.py:80-81
    SVM_CHECK_ARG(decay >= 0.0 && decay < 1.0, "decay has to lie in [0, 1)");
    SVM_CHECK_ARG(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0, "beta has to lie in [0, 1)");
    SVM_CHECK_ARG(epochs > 0 && epochs < (1ll << 24), "epochs must lie in [1, 2^24)");
    ALSpec spec;
    spec.p.rule = rule;
    spec.p.momentum_type = momentum_type;
    spec.p.has_eq = a_host != nullptr;
    spec.p.b = b;
    spec.p.rho = rho;
    spec.p.offset = offset;
    spec.p.tol = tol;
    spec.p.decay = decay;
    spec.p.om_decay = 1.0 - decay;
    spec.p.beta1 = beta1;
    spec.p.om_beta1 = 1.0 - beta1;
    spec.p.beta2 = beta2;
    spec.p.om_beta2 = 1.0 - beta2;
    spec.a_host = a_host;
    spec.lr_host = step_sizes;
    spec.mom_host = momentum_type == AL_MOM_NONE ? nullptr : momenta;
    return bcqp_create(ctx, dQ, n, ld, row0, nrows, hessian, q_host, lb_host, ub_host, x0_host, 0.0, epochs, SOLVER_AL, 0.0, out,
                       &spec, sign_host);
}

extern "C" int svmb200_al_multipliers(svmb200_pg* pg, double* mu, double* lam_lb_host, double* lam_ub_host) {
    SVM_CHECK_ARG(pg != nullptr && pg->solver == SOLVER_AL, "not an augmented-Lagrangian solver");
    SVM_TRY(pull_state(pg));
    cudaStream_t s = pg->ctx->stream;
    const size_t nv = (size_t)pg->nvars * sizeof(double);
    if (lam_lb_host) SVM_CUDA(cudaMemcpyAsync(lam_lb_host, pg->al.lam_lb, nv, cudaMemcpyDeviceToHost, s));
    if (lam_ub_host) SVM_CUDA(cudaMemcpyAsync(lam_ub_host, pg->al.lam_ub, nv, cudaMemcpyDeviceToHost, s));
    SVM_CUDA(cudaStreamSynchronize(s));
    if (mu) *mu = pg->st_host->mu;
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ K11: SMO (k_smo.cuh)
// libsvm's problem  min a'Qa/2 + q'a  s.t.  y'a = 0, 0 <= a <= ub  on the resident matrix.  One cooperative launch runs up
// to SMO_CHUNK iterations with the variables in the shared memory of its CTAs; the host polls the state between launches.
// The grid is one CTA per SM, but no CTA takes fewer than SMO_MIN_SLICE variables: an iteration costs two grid barriers plus
// the slice's work, and a barrier over fewer CTAs is cheaper (profiles/smo_grid_sweep.jsonl, B200: C1, 2 000 variables,
// 8.63 us per iteration on 148 CTAs, 7.77 on 16; C4, 50 000 variables, 12.4 us on 148, 12.2 on 74, 16.2 on 37).
// SVMB200_SMO_GRID overrides it (sweeps; tests on the host emulation); the grid grows when the slices would not fit the
// shared memory.
constexpr int64_t SMO_CHUNK = 65536;
constexpr int64_t SMO_MIN_SLICE = 128;
constexpr int64_t SMO_SLICE_MAX = (int64_t)(COOP_SMEM_MAX / (SMO_ARRAYS * sizeof(double)));
static_assert(SMO_SLICE_MAX <= 32 * SMO_ACT_WORDS, "the shrinking flags of a slice do not fit SMO_ACT_WORDS");

static size_t smo_smem_bytes(const svmb200_pg* pg) { return (size_t)pg->smo.a.slice * SMO_ARRAYS * sizeof(double); }

// computed rows (K12): what svmb200_smo_create_rows adds to the resident solver
struct SmoRowsSpec {
    KernelFn kf;
    size_t cache_bytes;
};

extern "C" int64_t svmb200_smo_max_vars(int sm_count) { return SMO_SLICE_MAX * (int64_t)sm_count; }

// the kernel of a row source, and its launch set-up
static void (*smo_kernel(int rows))(SmoArgs) {
    return rows == SMO_ROWS_COMPUTED ? smo_persistent_kernel<SMO_ROWS_COMPUTED>
         : rows == SMO_ROWS_SIGNED   ? smo_persistent_kernel<SMO_ROWS_SIGNED>
                                     : smo_persistent_kernel<SMO_ROWS_RESIDENT>;
}

static int smo_setup(svmb200_ctx* ctx, int rows, int grid, size_t smem, bool* fits) {
    return rows == SMO_ROWS_COMPUTED ? cooperative_setup<smo_persistent_kernel<SMO_ROWS_COMPUTED>>(ctx, grid, SMO_NT, smem, fits)
         : rows == SMO_ROWS_SIGNED   ? cooperative_setup<smo_persistent_kernel<SMO_ROWS_SIGNED>>(ctx, grid, SMO_NT, smem, fits)
                                     : cooperative_setup<smo_persistent_kernel<SMO_ROWS_RESIDENT>>(ctx, grid, SMO_NT, smem, fits);
}

// the same with shrinking
static void (*smo_shrink_kernel_of(int rows))(SmoShrinkArgs) {
    return rows == SMO_ROWS_COMPUTED ? smo_shrink_kernel<SMO_ROWS_COMPUTED>
         : rows == SMO_ROWS_SIGNED   ? smo_shrink_kernel<SMO_ROWS_SIGNED>
                                     : smo_shrink_kernel<SMO_ROWS_RESIDENT>;
}

static int smo_shrink_setup(svmb200_ctx* ctx, int rows, int grid, size_t smem, bool* fits) {
    return rows == SMO_ROWS_COMPUTED ? cooperative_setup<smo_shrink_kernel<SMO_ROWS_COMPUTED>>(ctx, grid, SMO_NT, smem, fits)
         : rows == SMO_ROWS_SIGNED   ? cooperative_setup<smo_shrink_kernel<SMO_ROWS_SIGNED>>(ctx, grid, SMO_NT, smem, fits)
                                     : cooperative_setup<smo_shrink_kernel<SMO_ROWS_RESIDENT>>(ctx, grid, SMO_NT, smem, fits);
}

// rows: the computed form (K12), else null; signed_view: dQ is an unsigned M read with the signs (SMO_ROWS_SIGNED);
// active: null, or one byte per variable of a signed view (svmb200_smo_create_subset): 0 holds the variable at 0
static int smo_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int hessian, const double* sign_host,
                      const double* q_host, const double* ub_host, double tol, int64_t max_iter, const SmoRowsSpec* rows,
                      bool signed_view, const unsigned char* active, svmb200_pg** out) {
    SVM_CHECK_ARG(max_iter > 0, "max_iter must be > 0");
    SVM_CHECK_ARG(tol >= 0.0, "tol must be >= 0");
    const int64_t nvars = hessian == SVMB200_HESSIAN_SVR ? 2 * n : n;
    SVM_CHECK_ARG(nvars < (1ll << 31), "too many variables");
    if (rows) {
        const int64_t cap = svmb200_smo_max_vars(ctx->sm_count > 0 ? ctx->sm_count : 1);
        if (nvars > cap) {
            svmb200_set_error("SMO with computed rows holds at most %lld variables on this GPU (%lld per CTA x %d SMs, the "
                              "shared-memory slice): %lld requested", (long long)cap, (long long)SMO_SLICE_MAX, ctx->sm_count,
                              (long long)nvars);
            return SVMB200_ERR_ARG;
        }
    }
    // an inactive variable gets ub = 0 (and alpha = 0, as every variable): it is then in neither I_up nor I_low, so it is
    // never selected, never enters m or M, and the solve of the active variables is their own problem's solve
    std::vector<double> ub_active;
    bool side[2] = {false, false};
    if (active) ub_active.assign(ub_host, ub_host + nvars);
    for (int64_t t = 0; t < nvars; ++t) {
        SVM_CHECK_ARG(sign_host[t] == 1.0 || sign_host[t] == -1.0, "signs must be +-1");
        if (active && !active[t]) {
            ub_active[(size_t)t] = 0.0;
            continue;
        }
        SVM_CHECK_ARG(ub_host[t] > 0.0 && ub_host[t] < INFINITY, "upper bounds must be finite and > 0");
        side[sign_host[t] > 0.0] = true;
    }
    if (active) {
        SVM_CHECK_ARG(side[0] && side[1], "the active variables must hold both signs of the equality constraint");
        ub_host = ub_active.data();
    }
    int grid = ctx->sm_count > 0 ? ctx->sm_count : 1;
    if ((int64_t)grid * SMO_MIN_SLICE > nvars) grid = (int)((nvars + SMO_MIN_SLICE - 1) / SMO_MIN_SLICE);
    if (const char* ev = getenv("SVMB200_SMO_GRID")) grid = atoi(ev);
    SVM_CHECK_ARG(grid >= 1, "SVMB200_SMO_GRID must be >= 1");
    int64_t slice = (nvars + grid - 1) / grid;
    if (slice > SMO_SLICE_MAX) slice = SMO_SLICE_MAX;
    PgGuard guard(new svmb200_pg());
    svmb200_pg* pg = guard.get();
    pg->ctx = ctx;
    pg->dQ = dQ;
    pg->n = n;
    pg->ld = ld;
    pg->row0 = 0;
    pg->nrows = n;
    pg->svr = hessian == SVMB200_HESSIAN_SVR;
    pg->nvars = nvars;
    pg->rows_per_rank = n;
    pg->solver = SOLVER_SMO;
    pg->eps = tol;
    pg->max_iter = max_iter;
    SmoSolver& smo = pg->smo;
    SmoArgs& a = smo.a;
    a.slice = (int)slice;
    smo.grid = (int)((nvars + slice - 1) / slice);
    smo.rows = rows ? SMO_ROWS_COMPUTED : signed_view ? SMO_ROWS_SIGNED : SMO_ROWS_RESIDENT;
    bool fits = false;
    SVM_TRY(smo_setup(ctx, smo.rows, smo.grid, smo_smem_bytes(pg), &fits));
    if (!fits) {
        svmb200_set_error("SMO: %d CTAs of %zu bytes of shared memory cannot be co-resident", smo.grid, smo_smem_bytes(pg));
        return SVMB200_ERR_ARG;
    }
    // one private slab: alpha, G, signs, ub (nvars each) | candidate slots | state
    const size_t nv = (size_t)nvars * sizeof(double), cand_bytes = (size_t)4 * smo.grid * sizeof(SmoCand);
    auto layout = [&](Carve c) {
        for (double** v : {&pg->x, &pg->g, &pg->sgn, &pg->ub}) c.take(*v, nv);
        c.take(a.cand, cand_bytes);
        c.take(pg->st, sizeof(PGDeviceState));
        return c.bytes;
    };
    SVM_TRY(acquire_workspace(pg, layout(Carve{}), false));
    layout(Carve{static_cast<unsigned char*>(pg->slab)});
    // start: alpha = 0, G = q
    cudaStream_t s = ctx->stream;
    SVM_CUDA(cudaMemsetAsync(pg->x, 0, nv, s));
    SVM_CUDA(cudaMemcpyAsync(pg->g, q_host, nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->sgn, sign_host, nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(pg->ub, ub_host, nv, cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemsetAsync(a.cand, 0, cand_bytes, s));
    SVM_CUDA(cudaMemsetAsync(pg->st, 0, sizeof(PGDeviceState), s));
    if (rows) {
        // cache geometry: every sample its own slot when all n rows fit, else sets of SMO_CACHE_WAYS (fewer if the
        // cache has fewer slots); cache_bytes = 0: no cache, every row is computed
        int64_t slots = (int64_t)(rows->cache_bytes / (nv > 0 ? nv : 1));
        if (slots >= n) {
            a.sets = n;
            a.ways = 1;
        } else if (slots > 0) {
            a.ways = slots < SMO_CACHE_WAYS ? slots : SMO_CACHE_WAYS;
            a.sets = slots / a.ways;
        }
        slots = a.sets * a.ways;
        // kernel of X, |x|^2, Q_ij slots, private tags and stamps per CTA, hit / miss count, row cache (sets x ways slots)
        a.kf = rows->kf;
        double* sqn = nullptr;
        auto rows_layout = [&](Carve c) {
            c.take(sqn, (size_t)n * sizeof(double));
            c.take(a.qij, (size_t)2 * smo.grid * sizeof(double));
            c.take(a.tags, (size_t)smo.grid * slots * sizeof(int));
            c.take(a.stamps, (size_t)smo.grid * slots * sizeof(long long));
            c.take(a.stats, 2 * sizeof(unsigned long long));
            c.take(a.cache, (size_t)slots * nv);
            return c.bytes;
        };
        SVM_CUDA(cudaMalloc(&smo.rows_buf, rows_layout(Carve{})));
        rows_layout(Carve{static_cast<unsigned char*>(smo.rows_buf)});
        if (slots == 0) a.cache = nullptr;
        SVM_CUDA(cudaMemsetAsync(a.qij, 0, (size_t)2 * smo.grid * sizeof(double), s));
        SVM_CUDA(cudaMemsetAsync(a.tags, 0xff, reinterpret_cast<unsigned char*>(a.stats) - reinterpret_cast<unsigned char*>(a.tags),
                                 s));   // tag -1 (empty), stamp -1
        SVM_CUDA(cudaMemsetAsync(a.stats, 0, 2 * sizeof(unsigned long long), s));
        if (a.kf.kernel == SVMB200_KERNEL_GAUSSIAN) {
            SVM_TRY(svm_row_sqnorms(ctx, a.kf.X, n, a.kf.ldx, a.kf.d, sqn));
            a.kf.sqn = sqn;
        }
    }
    SVM_CUDA(cudaStreamSynchronize(s));   // the host arrays belong to the caller
    a.Q = dQ;
    a.ld = ld;
    a.n = n;
    a.nvars = nvars;
    a.svr = pg->svr;
    a.x = pg->x;
    a.g = pg->g;
    a.sgn = pg->sgn;
    a.ub = pg->ub;
    a.gbar = ctx->gbar;
    a.st = pg->st;
    a.tol = tol;
    a.max_iter = max_iter;
    pg->k_next = 0;
    *out = guard.release();
    return SVMB200_OK;
}

extern "C" int svmb200_smo_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                                  int hessian, const double* sign_host, const double* q_host, const double* ub_host,
                                  double tol, int64_t max_iter, svmb200_pg** out) {
    SVM_TRY(check_create_args(__func__, ctx, out, dQ != nullptr && sign_host != nullptr && q_host != nullptr && ub_host != nullptr,
                              n, "Q is too small", ld >= n && ld % 2 == 0, "ld must be >= n and even", hessian));
    SVM_CHECK_ARG(row0 == 0 && nrows == n, "SMO needs the whole matrix on this rank (row0 = 0, nrows = n): it has no sharded form");
    return smo_create(ctx, dQ, n, ld, hessian, sign_host, q_host, ub_host, tol, max_iter, nullptr, false, nullptr, out);
}

extern "C" int svmb200_smo_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                         int64_t nrows, int hessian, const double* sign_host, const double* q_host,
                                         const double* ub_host, double tol, int64_t max_iter, svmb200_pg** out) {
    SVM_TRY(check_create_args(__func__, ctx, out, dQ != nullptr && sign_host != nullptr && q_host != nullptr && ub_host != nullptr,
                              n, "M is too small", ld >= n && ld % 2 == 0, "ld must be >= n and even", hessian));
    SVM_CHECK_ARG(row0 == 0 && nrows == n, "SMO needs the whole matrix on this rank (row0 = 0, nrows = n): it has no sharded form");
    return smo_create(ctx, dQ, n, ld, hessian, sign_host, q_host, ub_host, tol, max_iter, nullptr, true, nullptr, out);
}

extern "C" int svmb200_smo_create_subset(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                         int64_t nrows, int hessian, const double* sign_host, const double* q_host,
                                         const double* ub_host, const unsigned char* active, double tol, int64_t max_iter,
                                         svmb200_pg** out) {
    SVM_TRY(check_create_args(__func__, ctx, out,
                              dQ != nullptr && sign_host != nullptr && q_host != nullptr && ub_host != nullptr && active != nullptr,
                              n, "M is too small", ld >= n && ld % 2 == 0, "ld must be >= n and even", hessian));
    SVM_CHECK_ARG(row0 == 0 && nrows == n, "SMO needs the whole matrix on this rank (row0 = 0, nrows = n): it has no sharded form");
    return smo_create(ctx, dQ, n, ld, hessian, sign_host, q_host, ub_host, tol, max_iter, nullptr, true, active, out);
}

extern "C" int svmb200_smo_create_rows(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ldx, int64_t d, int kernel,
                                       double gamma, double coef0, double degree, int hessian, const double* sign_host,
                                       const double* q_host, const double* ub_host, double tol, int64_t max_iter,
                                       size_t cache_bytes, svmb200_pg** out) {
    SVM_TRY(check_create_args(__func__, ctx, out, dX != nullptr && sign_host != nullptr && q_host != nullptr && ub_host != nullptr,
                              n, "X is too small",
                              d > 0 && ldx >= d && ldx % 2 == 0 && (reinterpret_cast<uintptr_t>(dX) & 15) == 0,
                              "ldx must be even and >= d, X 16-byte aligned", hessian));
    SVM_CHECK_ARG(kernel >= SVMB200_KERNEL_LINEAR && kernel <= SVMB200_KERNEL_LAPLACIAN, "unknown kernel id");
    SVM_CHECK_ARG((kernel != SVMB200_KERNEL_GAUSSIAN && kernel != SVMB200_KERNEL_LAPLACIAN) || gamma >= 0.0,
                  "gamma must be >= 0 for the gaussian / laplacian kernels");
    SVM_CHECK_ARG(d < (1ll << 31), "dimension too large");
    SmoRowsSpec rows;
    rows.kf.X = dX;
    rows.kf.ldx = ldx;
    rows.kf.d = d;
    rows.kf.sqn = nullptr;
    rows.kf.kernel = kernel;
    rows.kf.gamma = gamma;
    rows.kf.coef0 = coef0;
    rows.kf.degree = degree;
    rows.kf.int_degree = svm_gram_int_degree(degree);
    rows.cache_bytes = cache_bytes;
    return smo_create(ctx, nullptr, n, 0, hessian, sign_host, q_host, ub_host, tol, max_iter, &rows, false, nullptr, out);
}

// Shrinking: q (nvars), the state, the active flags (nvars bytes) in one allocation at shrink.q.  Flags start set for
// every variable that is not held (ub > 0); the counter at min(l, 1000) + 1 puts the first check at state min(l, 1000).
extern "C" int svmb200_smo_set_shrinking(svmb200_pg* pg, int on) {
    SVM_CHECK_ARG(pg != nullptr && pg->solver == SOLVER_SMO, "not an SMO solver");
    SVM_CHECK_ARG(!pg->smo.started, "svmb200_smo_set_shrinking: the solver has already run");
    SVM_TRY(svm_use(pg->ctx));
    SmoShrink& sh = pg->smo.shrink;
    if (!on) {
        if (sh.q) SVM_CUDA(cudaFree(const_cast<double*>(sh.q)));
        sh = {};
        return SVMB200_OK;
    }
    if (sh.on) return SVMB200_OK;
    bool fits = false;
    SVM_TRY(smo_shrink_setup(pg->ctx, pg->smo.rows, pg->smo.grid, smo_smem_bytes(pg), &fits));
    if (!fits) {
        svmb200_set_error("SMO: %d CTAs of %zu bytes of shared memory cannot be co-resident", pg->smo.grid, smo_smem_bytes(pg));
        return SVMB200_ERR_ARG;
    }
    const size_t nv = (size_t)pg->nvars * sizeof(double);
    std::vector<double> ub((size_t)pg->nvars);
    std::vector<unsigned char> act((size_t)pg->nvars);
    cudaStream_t s = pg->ctx->stream;
    SVM_CUDA(cudaMemcpyAsync(ub.data(), pg->ub, nv, cudaMemcpyDeviceToHost, s));
    SVM_CUDA(cudaStreamSynchronize(s));
    long long l = 0;
    for (size_t t = 0; t < act.size(); ++t) l += act[t] = ub[t] > 0.0;
    SmoShrinkState st = {};
    st.counter = (l < SMO_SHRINK_EVERY ? l : SMO_SHRINK_EVERY) + 1;
    st.active = l;
    st.prepared = -1;
    const size_t st_off = nv, act_off = st_off + ((sizeof(SmoShrinkState) + 255) & ~size_t(255));
    unsigned char* buf = nullptr;
    SVM_CUDA(cudaMalloc(&buf, act_off + (size_t)pg->nvars));
    sh.q = reinterpret_cast<double*>(buf);
    sh.st = reinterpret_cast<SmoShrinkState*>(buf + st_off);
    sh.act = buf + act_off;
    sh.l = l;
    sh.on = 1;
    // before the first run G = q
    SVM_CUDA(cudaMemcpyAsync(buf, pg->g, nv, cudaMemcpyDeviceToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(sh.st, &st, sizeof(st), cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaMemcpyAsync(sh.act, act.data(), act.size(), cudaMemcpyHostToDevice, s));
    SVM_CUDA(cudaStreamSynchronize(s));
    return SVMB200_OK;
}

extern "C" int svmb200_smo_shrink_stats(svmb200_pg* pg, int64_t* active, int64_t* checks, int64_t* reconstructions) {
    SVM_CHECK_ARG(pg != nullptr && pg->solver == SOLVER_SMO, "not an SMO solver");
    SVM_TRY(svm_use(pg->ctx));
    SmoShrinkState st = {};
    if (pg->smo.shrink.on) {
        SVM_CUDA(cudaMemcpyAsync(&st, pg->smo.shrink.st, sizeof(st), cudaMemcpyDeviceToHost, pg->ctx->stream));
        SVM_CUDA(cudaStreamSynchronize(pg->ctx->stream));
    } else {
        st.active = pg->nvars;
    }
    if (active) *active = st.active;
    if (checks) *checks = st.checks;
    if (reconstructions) *reconstructions = st.reconstructions;
    return SVMB200_OK;
}

extern "C" int svmb200_smo_cache_stats(svmb200_pg* pg, int* computed, int64_t* slots, int64_t* hits, int64_t* misses) {
    SVM_CHECK_ARG(pg != nullptr && pg->solver == SOLVER_SMO, "not an SMO solver");
    SVM_TRY(svm_use(pg->ctx));
    const SmoArgs& a = pg->smo.a;
    unsigned long long hm[2] = {0, 0};
    if (pg->smo.rows == SMO_ROWS_COMPUTED) {
        SVM_CUDA(cudaMemcpyAsync(hm, a.stats, sizeof(hm), cudaMemcpyDeviceToHost, pg->ctx->stream));
        SVM_CUDA(cudaStreamSynchronize(pg->ctx->stream));
    }
    if (computed) *computed = pg->smo.rows == SMO_ROWS_COMPUTED;
    if (slots) *slots = a.sets * a.ways;
    if (hits) *hits = (int64_t)hm[0];
    if (misses) *misses = (int64_t)hm[1];
    return SVMB200_OK;
}

// history buffers for states 0 .. need - 1, one allocation (hist_f | hist_ng, hist_cap each): grown geometrically with the
// iterations actually run (max_iter may be 10^7)
static int smo_hist_reserve(svmb200_pg* pg, int64_t need) {
    if (need <= pg->hist_cap) return SVMB200_OK;
    int64_t cap = pg->hist_cap * 2 > need ? pg->hist_cap * 2 : need;
    if (cap < 1024) cap = 1024;
    if (cap > pg->max_iter + 1) cap = pg->max_iter + 1;
    cudaStream_t s = pg->ctx->stream;
    double* h = nullptr;
    SVM_CUDA(cudaMalloc(&h, 2 * (size_t)cap * sizeof(double)));
    if (pg->hist_f) {
        SVM_CUDA(cudaMemcpyAsync(h, pg->hist_f, (size_t)pg->hist_cap * sizeof(double), cudaMemcpyDeviceToDevice, s));
        SVM_CUDA(cudaMemcpyAsync(h + cap, pg->hist_ng, (size_t)pg->hist_cap * sizeof(double), cudaMemcpyDeviceToDevice, s));
        SVM_CUDA(cudaStreamSynchronize(s));
        SVM_CUDA(cudaFree(pg->hist_f));
    }
    pg->hist_f = h;
    pg->hist_ng = h + cap;
    pg->hist_cap = cap;
    return SVMB200_OK;
}

// evaluate states k_next .. k_next + niter, stepping between them, unless the stopping test fires first
static int smo_launch(svmb200_pg* pg, int64_t niter) {
    SmoArgs& a = pg->smo.a;
    a.hist_f = pg->hist_f;
    a.hist_gap = pg->hist_ng;
    a.hist_cap = pg->hist_cap;
    a.k0 = pg->k_next;
    a.niter = niter;
    if (pg->smo.shrink.on)
        SVM_CUDA(svm_launch_cooperative(smo_shrink_kernel_of(pg->smo.rows), dim3((unsigned)pg->smo.grid), dim3(SMO_NT),
                                        smo_smem_bytes(pg), pg->ctx->stream, SmoShrinkArgs{a, pg->smo.shrink}));
    else
        SVM_CUDA(svm_launch_cooperative(smo_kernel(pg->smo.rows), dim3((unsigned)pg->smo.grid), dim3(SMO_NT), smo_smem_bytes(pg),
                                        pg->ctx->stream, a));
    pg->ctx->launches++;
    return SVMB200_OK;
}

static int smo_run(svmb200_pg* pg, int64_t max_new) {
    svmb200_ctx* ctx = pg->ctx;
    SVM_TRY(svm_use(ctx));
    reset_run_stats(pg);   // last_passes stays 0: an iteration reads two rows, never a full pass over Q
    pg->smo.started = true;
    SVM_CUDA(cudaEventRecord(pg->ev0, ctx->stream));
    if (!pg->finished) {
        int64_t budget = pg->max_iter - pg->k_next;
        if (max_new >= 0 && max_new < budget) budget = max_new;
        do {   // at least one launch: max_new = 0 evaluates the current state
            const int64_t nb = budget < SMO_CHUNK ? budget : SMO_CHUNK;
            SVM_TRY(smo_hist_reserve(pg, pg->k_next + nb + 1));
            SVM_TRY(smo_launch(pg, nb));
            SVM_TRY(poll_enqueue(pg, 0));
            SVM_TRY(poll_wait(pg, 0));
            pg->k_next = pg->finished ? pg->st_host->iter : pg->k_next + nb;
            budget -= nb;
        } while (budget > 0 && !pg->finished);
    }
    SVM_CUDA(cudaEventRecord(pg->ev1, ctx->stream));
    SVM_CUDA(cudaEventSynchronize(pg->ev1));
    SVM_CUDA(cudaEventElapsedTime(&pg->last_ms, pg->ev0, pg->ev1));
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ K14: SMO batch (k_smo.cuh)
// Several resident or signed-view SMO problems (subsets included) on one matrix share the GPU: an SMO iteration is bound
// by the latency of two grid barriers, not by bandwidth, and a smaller grid costs a problem little (profiles/smo_grid_sweep.jsonl).  So
// problems run side by side on disjoint ranges of CTAs, at most one CTA per SM, in one cooperative launch of at most
// SMO_BATCH_CHUNK iterations per problem.  Before every launch the scheduler admits unfinished problems in index order
// while their minimum grids (slices of at most SMO_SLICE_MAX variables) fit the SMs, and splits the SMs evenly among
// them, no problem above its own single-fit grid; after it, one synchronisation reads every admitted problem's state.
// Problems that finished give their SMs to the others at the next launch and waiting problems are admitted.  A solve
// does not depend on its grid, so each problem ends bit for bit where its own svmb200_pg_run would.
// SVMB200_SMO_BATCH_SMS caps the SMs a batch uses and SVMB200_SMO_BATCH_CHUNK sets the chunk (sweeps; tests on the host
// emulation, which reports 148 SMs).
constexpr int64_t SMO_BATCH_CHUNK = 4096;

static int env_positive(const char* name, int64_t* value) {
    if (const char* ev = getenv(name)) {
        const long long v = atoll(ev);
        if (v < 1) {
            svmb200_set_error("%s must be >= 1", name);
            return SVMB200_ERR_ARG;
        }
        *value = v;
    }
    return SVMB200_OK;
}

extern "C" int svmb200_smo_run_batch(svmb200_pg* const* pgs, int count, int64_t* iters, int* statuses) {
    SVM_CHECK_ARG(pgs != nullptr && count >= 1 && count <= 65535, "bad argument");
    svmb200_pg* p0 = pgs[0];
    for (int b = 0; b < count; ++b) {
        const svmb200_pg* p = pgs[b];
        SVM_CHECK_ARG(p != nullptr && p0 != nullptr, "null solver");
        SVM_CHECK_ARG(p->solver == SOLVER_SMO, "svmb200_smo_run_batch takes SMO solvers only");
        SVM_CHECK_ARG(p->smo.rows != SMO_ROWS_COMPUTED, "an SMO solver with computed rows has no batch: run it alone");
        SVM_CHECK_ARG(p->ctx == p0->ctx && p->dQ == p0->dQ && p->n == p0->n && p->ld == p0->ld && p->svr == p0->svr &&
                          p->smo.rows == p0->smo.rows,
                      "the solvers of a batch must share the resident matrix and its layout");
        SVM_CHECK_ARG(p->k_next == 0 && !p->finished, "a batch takes solvers that have not run yet");
        for (int c = 0; c < b; ++c) SVM_CHECK_ARG(pgs[c] != p, "a solver is listed twice");
    }
    svmb200_ctx* ctx = p0->ctx;
    SVM_TRY(svm_use(ctx));
    int64_t sms = ctx->sm_count > 0 ? ctx->sm_count : 1, chunk = SMO_BATCH_CHUNK;
    int64_t cap = sms;
    SVM_TRY(env_positive("SVMB200_SMO_BATCH_SMS", &cap));
    SVM_TRY(env_positive("SVMB200_SMO_BATCH_CHUNK", &chunk));
    if (cap < sms) sms = cap;
    const int64_t nvars = p0->nvars, g_min = (nvars + SMO_SLICE_MAX - 1) / SMO_SLICE_MAX;
    if (sms < g_min) sms = g_min;   // a cap below one problem's minimum grid still runs one problem at a time
    const int64_t slots = std::min<int64_t>(count, sms / g_min);
    // per launch: the problems' arguments, and one grid barrier (256 bytes) per admitted problem
    const size_t probs_bytes = ((size_t)slots * sizeof(SmoBatchProblem) + 255) & ~size_t(255);
    SVM_TRY(svm_scratch_reserve(ctx, &ctx->batch_buf, &ctx->batch_bytes, probs_bytes + (size_t)slots * 256));
    SmoBatchProblem* dprobs = static_cast<SmoBatchProblem*>(ctx->batch_buf);
    unsigned* bars = reinterpret_cast<unsigned*>(static_cast<unsigned char*>(ctx->batch_buf) + probs_bytes);
    SVM_CUDA(cudaMemsetAsync(bars, 0, (size_t)slots * 256, ctx->stream));
    bool shrink = false;   // one problem shrinks: the launches take smo_batch_shrink_kernel (a flag per problem)
    for (int b = 0; b < count; ++b) {
        reset_run_stats(pgs[b]);
        pgs[b]->smo.started = true;
        shrink = shrink || pgs[b]->smo.shrink.on;
    }
    SVM_CUDA(cudaEventRecord(p0->ev0, ctx->stream));
    std::vector<SmoBatchProblem> hp((size_t)slots);
    std::vector<int> admitted((size_t)slots);
    std::vector<int64_t> nb((size_t)slots);
    for (int next = 0;;) {
        while (next < count && pgs[next]->finished) ++next;
        int k = 0;
        for (int b = next; b < count && k < slots; ++b)
            if (!pgs[b]->finished) admitted[k++] = b;
        if (k == 0) break;
        int cta0 = 0;
        size_t smem = 0;
        for (int r = 0; r < k; ++r) {
            svmb200_pg* pg = pgs[admitted[r]];
            int64_t g = sms / k + (r < sms % k ? 1 : 0);
            if (g > pg->smo.grid) g = pg->smo.grid;
            const int64_t slice = (nvars + g - 1) / g;
            const int64_t left = pg->max_iter - pg->k_next;
            nb[r] = left < chunk ? left : chunk;
            SVM_TRY(smo_hist_reserve(pg, pg->k_next + nb[r] + 1));
            SmoBatchProblem& p = hp[r];
            p.a = pg->smo.a;
            p.a.slice = (int)slice;
            p.a.gbar = bars + (size_t)r * 64;
            p.a.hist_f = pg->hist_f;
            p.a.hist_gap = pg->hist_ng;
            p.a.hist_cap = pg->hist_cap;
            p.a.k0 = pg->k_next;
            p.a.niter = nb[r];
            p.s = pg->smo.shrink;
            p.cta0 = cta0;
            p.grid = (int)((nvars + slice - 1) / slice);
            cta0 += p.grid;
            smem = std::max(smem, (size_t)slice * SMO_ARRAYS * sizeof(double));
        }
        bool fits = false;
        const bool sgn = p0->smo.rows == SMO_ROWS_SIGNED;
        void (*kernel)(SmoBatchArgs) = shrink ? (sgn ? smo_batch_shrink_kernel<SMO_ROWS_SIGNED> : smo_batch_shrink_kernel<SMO_ROWS_RESIDENT>)
                                              : (sgn ? smo_batch_kernel<SMO_ROWS_SIGNED> : smo_batch_kernel<SMO_ROWS_RESIDENT>);
        SVM_TRY(shrink ? (sgn ? cooperative_setup<smo_batch_shrink_kernel<SMO_ROWS_SIGNED>>(ctx, cta0, SMO_NT, smem, &fits)
                              : cooperative_setup<smo_batch_shrink_kernel<SMO_ROWS_RESIDENT>>(ctx, cta0, SMO_NT, smem, &fits))
                       : (sgn ? cooperative_setup<smo_batch_kernel<SMO_ROWS_SIGNED>>(ctx, cta0, SMO_NT, smem, &fits)
                              : cooperative_setup<smo_batch_kernel<SMO_ROWS_RESIDENT>>(ctx, cta0, SMO_NT, smem, &fits)));
        if (!fits) {
            svmb200_set_error("SMO batch: %d CTAs of %zu bytes of shared memory cannot be co-resident", cta0, smem);
            return SVMB200_ERR_STATE;
        }
        SVM_CUDA(cudaMemcpyAsync(dprobs, hp.data(), (size_t)k * sizeof(SmoBatchProblem), cudaMemcpyHostToDevice, ctx->stream));
        SmoBatchArgs ba;
        ba.probs = dprobs;
        ba.count = k;
        SVM_CUDA(svm_launch_cooperative(kernel, dim3((unsigned)cta0), dim3(SMO_NT), smem, ctx->stream, ba));
        ctx->launches++;
        for (int r = 0; r < k; ++r) {
            svmb200_pg* pg = pgs[admitted[r]];
            SVM_CUDA(cudaMemcpyAsync(pg->st_host, pg->st, sizeof(PGDeviceState), cudaMemcpyDeviceToHost, ctx->stream));
        }
        SVM_CUDA(cudaStreamSynchronize(ctx->stream));
        for (int r = 0; r < k; ++r) {
            svmb200_pg* pg = pgs[admitted[r]];
            if (pg->st_host->done) pg->finished = true;
            pg->k_next = pg->finished ? pg->st_host->iter : pg->k_next + nb[r];
        }
    }
    SVM_CUDA(cudaEventRecord(p0->ev1, ctx->stream));
    SVM_CUDA(cudaEventSynchronize(p0->ev1));
    float ms = 0.f;
    SVM_CUDA(cudaEventElapsedTime(&ms, p0->ev0, p0->ev1));
    for (int b = 0; b < count; ++b) {
        svmb200_pg* pg = pgs[b];
        pg->last_ms = ms;  // device time of the whole batch
        if (iters) iters[b] = pg->st_host->iter;
        if (statuses) statuses[b] = pg->st_host->status;
    }
    return SVMB200_OK;
}

// ------------------------------------------------------------------------------------------ K5
extern "C" int svmb200_masked_product(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                                      int64_t nrows, const double* beta_host, double* v_host) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dQ && beta_host && v_host, "null argument");
    SVM_CHECK_ARG(ld >= n && ld % 2 == 0, "ld must be >= n and even");
    const int P = ctx->nranks;
    const int64_t rpr = rows_per_rank(n, P);
    {
        int64_t exp_row0 = 0, exp_rows = 0;
        SVM_TRY(svmb200_shard_rows(n, ctx->rank, P, &exp_row0, &exp_rows));
        SVM_CHECK_ARG(row0 == exp_row0 && nrows == exp_rows, "row shard does not match svmb200_shard_rows");
    }
    SVM_TRY(svm_scratch_reserve(ctx, &ctx->mp_buf, &ctx->mp_bytes, (size_t)(ld + rpr * P) * sizeof(double)));
    double* du = static_cast<double*>(ctx->mp_buf);
    double* dw = du + ld;
    int rc = SVMB200_OK;
    cudaStream_t s = ctx->stream;
    cudaMemsetAsync(du, 0, (size_t)ld * sizeof(double), s);
    cudaMemsetAsync(dw, 0, (size_t)(rpr * P) * sizeof(double), s);
    cudaMemcpyAsync(du, beta_host, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, s);
    rc = svm_launch_matvec(ctx, dQ, nrows, ld, du, dw + (size_t)ctx->rank * rpr, nullptr);
    if (rc == SVMB200_OK && P > 1 && !ctx->local_group) rc = svm_comm_allgather(ctx, dw, rpr);
    if (rc == SVMB200_OK && ctx->local_group && P > 1) {
        // single-process group: no collective -- this call fills rows [row0, row0 + nrows) of v_host, the caller makes it
        // once per rank with the same v_host
        if (nrows > 0)
            cudaMemcpyAsync(v_host + row0, dw + (size_t)ctx->rank * rpr, (size_t)nrows * sizeof(double), cudaMemcpyDeviceToHost, s);
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) {
            svmb200_set_error("masked_product: %s", cudaGetErrorString(e));
            rc = SVMB200_ERR_CUDA;
        }
        return rc;
    }
    if (rc == SVMB200_OK) {
        cudaMemcpyAsync(v_host, dw, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s);
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) {
            svmb200_set_error("masked_product: %s", cudaGetErrorString(e));
            rc = SVMB200_ERR_CUDA;
        }
    }
    return rc;
}

// The same for every rank of a single-process group at once: count contexts (rank order) with their shards dQ[r];
// all products run concurrently, v_host receives the n results.
extern "C" int svmb200_masked_product_group(svmb200_ctx* const* ctxs, const double* const* dQ, int count, int64_t n, int64_t ld,
                                            const double* beta_host, double* v_host) {
    SVM_CHECK_ARG(ctxs != nullptr && dQ != nullptr && count >= 1 && count <= SVM_MAX_RANKS && beta_host && v_host, "bad argument");
    SVM_CHECK_ARG(ld >= n && ld % 2 == 0, "ld must be >= n and even");
    const int64_t rpr = rows_per_rank(n, count);
    for (int r = 0; r < count; ++r) {
        svmb200_ctx* ctx = ctxs[r];
        SVM_CHECK_ARG(ctx != nullptr && ctx->nranks == count && ctx->rank == r && (count == 1 || ctx->local_group),
                      "pass the contexts of the single-process group in rank order");
        SVM_TRY(svm_use(ctx));
        int64_t row0 = 0, nrows = 0;
        SVM_TRY(svmb200_shard_rows(n, r, count, &row0, &nrows));
        SVM_CHECK_ARG(nrows == 0 || dQ[r] != nullptr, "null shard");
        SVM_TRY(svm_scratch_reserve(ctx, &ctx->mp_buf, &ctx->mp_bytes, (size_t)(ld + rpr * count) * sizeof(double)));
        double* du = static_cast<double*>(ctx->mp_buf);
        double* dw = du + ld;
        cudaStream_t s = ctx->stream;
        SVM_CUDA(cudaMemsetAsync(du, 0, (size_t)ld * sizeof(double), s));
        SVM_CUDA(cudaMemcpyAsync(du, beta_host, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, s));
        SVM_TRY(svm_launch_matvec(ctx, dQ[r], nrows, ld, du, dw, nullptr));
        if (nrows > 0) SVM_CUDA(cudaMemcpyAsync(v_host + row0, dw, (size_t)nrows * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    for (int r = 0; r < count; ++r) {
        SVM_TRY(svm_use(ctxs[r]));
        SVM_CUDA(cudaStreamSynchronize(ctxs[r]->stream));
    }
    return SVMB200_OK;
}
