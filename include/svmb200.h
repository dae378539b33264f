/*
 * svmb200.h -- C ABI of the B200-native kernel-SVM dual training path.
 *
 * This is the drop-in boundary for ONE hot path of dmeoli/optiml (a pure-Python/NumPy library):
 *   SVC/SVR(dual=True, reg_intercept=True, optimizer=ProjectedGradient).fit / decision_function
 * with LinearKernel / PolyKernel / GaussianKernel.  The reference has no FFI seam of its own; the
 * seam is the NumPy call sites listed beside each entry point (paths relative to the reference
 * repository root).  A binding only needs ctypes/cffi: plain pointers, sizes and doubles, no
 * framework types.  INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *   - every function returns 0 on success and a non-zero code on failure; svmb200_last_error()
 *     then returns a thread-local, NUL-terminated description (CUDA / NCCL error text included);
 *   - there is NO CPU fallback: without a CUDA device (or with a non-sm_100 device) the compute
 *     entry points fail with SVMB200_ERR_CUDA;
 *   - "dptr" arguments are device pointers obtained from svmb200_malloc on the same context;
 *     "host" arguments are ordinary host pointers (pinned or pageable);
 *   - all matrices are FP64, row-major; "ld" is the row stride in elements;
 *   - one context == one GPU == one CUDA stream; multi-GPU runs use one process (context) per GPU
 *     and exchange the per-iteration product shards with one NCCL all-gather (svmb200_comm_*).
 */
#ifndef SVMB200_H
#define SVMB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVMB200_OK 0
#define SVMB200_ERR_ARG 1     /* invalid argument */
#define SVMB200_ERR_CUDA 2    /* CUDA runtime / driver error, or no usable device */
#define SVMB200_ERR_NCCL 3    /* NCCL error or libnccl not loadable */
#define SVMB200_ERR_STATE 4   /* call sequence error */

/* kernel ids: optiml/ml/svm/kernels.py:40 (LinearKernel), :54 (PolyKernel), :98 (GaussianKernel) */
#define SVMB200_KERNEL_LINEAR 0
#define SVMB200_KERNEL_POLY 1
#define SVMB200_KERNEL_GAUSSIAN 2
/* widening (SURVEY.md 8f-2): kernels.py:166 (SigmoidKernel), :132 (LaplacianKernel) */
#define SVMB200_KERNEL_SIGMOID 3
#define SVMB200_KERNEL_LAPLACIAN 4

/* Hessian layouts understood by the solver */
#define SVMB200_HESSIAN_PLAIN 0 /* Q is the n x n matrix itself, nvars = n (SVC; generic BCQP)      */
#define SVMB200_HESSIAN_SVR 1   /* resident matrix is M = K+1 (n x n); Q = [[M,-M],[-M,M]], nvars=2n */

/* solver status, optiml/opti/_base.py:76 and projected_gradient.py:100-106 */
#define SVMB200_STATUS_UNKNOWN 0
#define SVMB200_STATUS_OPTIMAL 1
#define SVMB200_STATUS_STOPPED 2

typedef struct svmb200_ctx svmb200_ctx;
typedef struct svmb200_pg svmb200_pg;

const char* svmb200_last_error(void);
const char* svmb200_version(void);

/* ---- context, memory, multi-GPU plumbing ------------------------------------------------- */
int svmb200_device_count(int* count);
int svmb200_ctx_create(int device, svmb200_ctx** out);
int svmb200_ctx_destroy(svmb200_ctx* ctx);
int svmb200_ctx_info(svmb200_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* free_bytes,
                     size_t* total_bytes);
int svmb200_malloc(svmb200_ctx* ctx, size_t bytes, void** dptr);
int svmb200_free(svmb200_ctx* ctx, void* dptr);
int svmb200_memset(svmb200_ctx* ctx, void* dptr, int value, size_t bytes);
int svmb200_h2d(svmb200_ctx* ctx, void* dptr, const void* host, size_t bytes);
int svmb200_d2h(svmb200_ctx* ctx, void* host, const void* dptr, size_t bytes);
int svmb200_d2d(svmb200_ctx* ctx, void* dst, const void* src, size_t bytes);
int svmb200_sync(svmb200_ctx* ctx);
int svmb200_host_alloc_pinned(size_t bytes, void** host);
int svmb200_host_free_pinned(void* host);
/* CUDA-event timing on the context's stream (used by bench.py; torch events do not see this stream) */
int svmb200_timer_start(svmb200_ctx* ctx);
int svmb200_timer_stop_ms(svmb200_ctx* ctx, float* ms); /* records, synchronises, returns elapsed */
/* number of kernels this library launched on the context since creation */
int svmb200_launch_count(svmb200_ctx* ctx, uint64_t* launches);

/* NCCL: rank 0 calls svmb200_comm_unique_id and broadcasts the 128 bytes by any means
 * (the Python host uses torch.distributed); every rank then calls svmb200_comm_init. */
int svmb200_comm_unique_id(void* id128);
int svmb200_comm_init(svmb200_ctx* ctx, const void* id128, int rank, int nranks);
int svmb200_comm_destroy(svmb200_ctx* ctx);
/* Optional fused exchange over NVLink peer memory (replaces the per-iteration ncclAllGather of the
 * solver): every rank exports an arena (svmb200_comm_p2p_export returns its 64-byte CUDA IPC handle),
 * the handles of all ranks, concatenated in rank order, are passed to svmb200_comm_p2p_attach.  The
 * matvec kernel then stores its results directly into every peer's arena as self-validating tagged
 * 16-byte entries (no fence, no flag); the vector kernel spins on the entries it reads.  Without it
 * (or if IPC mapping fails, or for a problem so small that the 64-row shard granularity leaves a rank
 * without rows) NCCL is used. */
int svmb200_comm_p2p_export(svmb200_ctx* ctx, size_t arena_bytes, void* handle64);
int svmb200_comm_p2p_attach(svmb200_ctx* ctx, const void* handles, int nranks);
int svmb200_comm_p2p_enabled(svmb200_ctx* ctx, int* enabled);
int svmb200_comm_p2p_disable(svmb200_ctx* ctx); /* all ranks must agree: call it everywhere if any rank failed to attach */
/* Row partition used by every sharded entry point: rank r owns rows [row0, row0+nrows) of an n-row
 * matrix, ceil(n/nranks) rounded up to a multiple of 64 rows per rank (the last ranks may get fewer,
 * possibly none).  Aligned shard boundaries keep every reduction shape independent of nranks. */
int svmb200_shard_rows(int64_t n, int rank, int nranks, int64_t* row0, int64_t* nrows);

/* ---- K1: Gram / Hessian build ------------------------------------------------------------
 * Replaces  kernels.py:49-51 (linear), :91-95 (poly), :125-129 (gaussian, via sklearn
 * euclidean_distances) fused with  ml/svm/_base.py:554,628 (SVC: Q = K o yy^T + yy^T) or
 * :1098-1099,1178 (SVR: M = K + 1; the 2x2 sign pattern is applied by the solver).
 *
 * out[i - row0][j] = s_i s_j ( k(A_i, B_j) + bias ),  i in [row0, row0+nrows), j in [0, nb)
 *   k = <a,b>                              (LINEAR)
 *     = (gamma <a,b> + coef0) ^ degree     (POLY)
 *     = exp(-gamma max(0, |a|^2+|b|^2-2<a,b>)), distance forced to 0 where i == j if `same` (GAUSSIAN)
 *     = tanh(gamma <a,b> + coef0)                                                              (SIGMOID)
 *     = exp(-gamma sum_k |a_k - b_k|)   (LAPLACIAN; CUDA-core pairwise kernel, not a contraction)
 * dA: na x d (ld = lda), dB: nb x d (ld = ldb); pass dB = dA and same = 1 for the training Gram.
 * dsign_a / dsign_b: +-1.0 per row, or NULL (= +1).  Columns [nb, ldo) of `out` are zero-filled
 * (the solver streams whole padded rows).  ldo must be a multiple of 2.
 * Tiled FP64 tensor-core contraction (mma.sync DMMA), operands staged by TMA.                 */
int svmb200_gram(svmb200_ctx* ctx, const double* dA, int64_t na, int64_t lda, const double* dB, int64_t nb,
                 int64_t ldb, int64_t d, int same, int kernel, double gamma, double coef0, double degree,
                 const double* dsign_a, const double* dsign_b, double bias, int64_t row0, int64_t nrows,
                 double* dout, int64_t ldo);
/* helper: leading dimension the library wants for an n-column streamed matrix */
int64_t svmb200_padded_ld(int64_t ncols);

/* ---- K2: streaming matrix-vector product ---------------------------------------------------
 * dw[row0 + i] = sum_j dQ[i][j] * du[j], i in [0, nrows).  du must hold ld elements (pad = 0).
 * Replaces the three products of projected_gradient.py:82,121 (opti/_base.py:282,291).          */
int svmb200_matvec(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, const double* du, double* dw);

/* ---- K2s: the same product from the UPPER TRIANGLE of a symmetric matrix (opt-in) -----------
 * dw[i] = sum_j dQ[i][j] * du[j] for a symmetric n x n matrix, streaming 4 n^2 bytes instead of 8 n^2: every element
 * above the diagonal blocks is used for its row and, transposed, for its column.  The lower triangle is never read.
 * Replaces the same `Q.dot(d)` (projected_gradient.py:113) for the Hessians of the SVM dual, which are symmetric by
 * construction (ml/svm/_base.py:554, 1098-1099).  Reproducible run to run; NOT bit-identical to svmb200_matvec
 * (another summation order), which is why solvers use it only on request:
 *   svmb200_ctx_set_symmetric(ctx, 1)  (initial value: environment variable SVMB200_SYMMETRIC)  makes every solver
 *   created afterwards that holds the WHOLE matrix on one rank take its products this way; sharded solvers and
 *   lockstep batches keep the full pass.  svmb200_pg_is_symmetric reports what a solver does.                      */
int svmb200_symv(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, const double* du, double* dw);
int svmb200_ctx_set_symmetric(svmb200_ctx* ctx, int on);
int svmb200_ctx_get_symmetric(svmb200_ctx* ctx, int* on);
/* what one symmetric pass over an n x n matrix streams (bytes: diagonal blocks in full + everything to their right) and
 * its tile geometry (rows per band, columns per panel, work items) -- for rooflines; any output pointer may be NULL */
int svmb200_symv_geometry(int64_t n, int64_t ld, int64_t* streamed_bytes, int64_t* band_rows, int64_t* panel_cols,
                          int64_t* items);
/* the work plan of rank `rank` of `nranks` row blocks on a GPU with sm_count SMs: bands (the last ones of a shard may be
 * short ones, a quarter of the height, so that the grid ends on small items), how many of them are short, work items, and
 * the simulated finish time of the grid over a perfectly balanced one -- for tests and tuning                        */
int svmb200_symv_plan_info(int64_t n, int64_t ld, int rank, int nranks, int sm_count, int64_t* bands, int64_t* short_bands,
                           int64_t* items, double* finish_over_ideal);
/* the work items of that plan: seven ints each {first local row, rows, band, first column, columns, row-sum slot, 1 if the
 * item also feeds column sums}; *count items (items7 may be NULL to ask for the count), *row0 = first row of the block   */
int svmb200_symv_plan_items(int64_t n, int64_t ld, int rank, int nranks, int sm_count, int32_t* items7, int64_t capacity,
                            int64_t* count, int64_t* row0);

/* ---- K2e: svmb200_matvec's product, BIT FOR BIT, from the upper triangle of an EXACTLY symmetric matrix ----------
 * dw[i] = sum_j dQ[i][j] * du[j] for an n x n matrix with dQ[i][j] == dQ[j][i] bitwise (every self-Gram svmb200_gram
 * builds, same = 1), in svmb200_matvec's summation order.  Needs at least two column segments of 8192 and the last one
 * holding real rows (ld < n + 8192).  The lower triangle off the 8192 x 8192 diagonal blocks is never read.
 *   svmb200_pg_set_self_gram(pg, 1) tells a solver that its matrix is such a self-Gram: on one rank, without the
 *   opt-in symmetric pass, its products then take this pass (SVMB200_EXACT_SYMV=0 keeps svmb200_matvec's).
 *   svmb200_pg_is_exact_symv reports what a solver does.                                                          */
int svmb200_matvec_exact(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, const double* du, double* dw);
/* bytes one such pass moves: matrix elements read (diagonal blocks in full + the blocks to their right) and the column
 * chains written and read back; *items = work items of the tile pass.  Any output pointer may be NULL. */
int svmb200_exact_symv_geometry(int64_t n, int64_t ld, int64_t* matrix_bytes, int64_t* scratch_bytes, int64_t* items);

/* ---- K2+K3(+K4): projected-gradient solve of the box-constrained QP -------------------------
 * Replaces  BoxConstrainedQuadraticOptimizer.__init__ (opti/constrained/_base.py:59-73) +
 * ProjectedGradient.minimize (opti/constrained/projected_gradient.py:76-143).
 *
 * The context's rank owns rows [row0, row0+nrows) of the n x n resident matrix dQ (ld).  With a
 * communicator attached every rank must call the same sequence; row shards must be the ones
 * svmb200_shard_rows returns.
 * Host vectors q, lb, ub, x0 have nvars = n (PLAIN) or 2n (SVR) elements; lb may be NULL (= 0),
 * x0 may be NULL (= (lb+ub)/2).                                                               */
int svmb200_pg_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                      int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                      const double* x0_host, double eps, int64_t max_iter, svmb200_pg** out);
/* Frank-Wolfe on the same problem / same handle type (widening, SURVEY.md 8f-1): replaces FrankWolfe.minimize
 * (opti/constrained/frank_wolfe.py:88-165).  `t` in [0,1) is the stabilisation parameter.  The second history
 * array of svmb200_pg_history then holds the relative gap, svmb200_pg_state's `ng` the last gap. */
int svmb200_fw_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                      int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                      const double* x0_host, double eps, int64_t max_iter, double t, svmb200_pg** out);
/* K11: SMO on the same handle type -- libsvm's solver without shrinking (working-set selection WSS2; Fan, Chen & Lin
 * 2005) for the SVM dual WITH its equality constraint (an unregularised intercept, sklearn's SVC / SVR):
 *     min a'Qa/2 + q'a   s.t.  sign'a = 0,  0 <= a <= ub
 * Replaces optiml/ml/svm/smo.py (SMOClassifier, SMORegression; selection rules restated, not copied).  Starts at a = 0,
 * stops with OPTIMAL when the maximal violating pair's gap m - M is below `tol` (or no pair is left), with STOPPED at
 * max_iter.  sign_host: nvars values of +-1 (SVC: the labels; SVR: e = [1 (n times), -1 (n times)]); with the PLAIN
 * layout dQ holds Q itself (SVC: y_s y_t K_st), with SVR it holds K and Q = [[K,-K],[-K,K]].  The matrix must be the
 * whole problem on this rank (row0 = 0, nrows = n; otherwise SVMB200_ERR_ARG): there is no sharded SMO.  Then
 * svmb200_pg_run (chunks of at most 65 536 iterations per launch, history storage grown with the iterations run),
 * _state (x = a, g = G = Qa + q, f = objective tracked per step, ng = gap), _history (f and gap per state), _scalars
 * ({f, gap, 0, 0, 0, 0}), _stats (passes = 0: an iteration reads two rows of Q) and _destroy apply; lockstep batches
 * of svmb200_pg_run_batch and single-process groups do not (svmb200_smo_run_batch below is SMO's batch).           */
int svmb200_smo_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                       int hessian, const double* sign_host, const double* q_host, const double* ub_host, double tol,
                       int64_t max_iter, svmb200_pg** out);
/* The same solver on a signed view of a shared, unsigned M (svmb200_gram with bias 0 and no signs): dQ holds M (n x n)
 * and Q_st = (sign_s == sign_t ? M_st : -M_st) with s, t taken mod n, the signs being sign_host (SVC: the labels; SVR:
 * e, which is the SVR read of svmb200_smo_create).  The diagonal is read unsigned.  svmb200_gram signs a matrix by
 * flipping the sign bit of fl(K + bias), the same operation, so the solve is BIT-IDENTICAL to svmb200_smo_create on
 * the signed Q svmb200_gram builds with these signs.  Arguments and answers as for svmb200_smo_create.             */
int svmb200_smo_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                              int hessian, const double* sign_host, const double* q_host, const double* ub_host,
                              double tol, int64_t max_iter, svmb200_pg** out);
/* The signed-view solver on a subset of the variables: active_host holds one byte per variable, and a variable whose
 * byte is 0 is held at 0 (the solver sets its upper bound to 0; its ub_host and q_host entries are not used).  Such a
 * variable is never selected and never changes m or M, and ties go to the larger index, so the active variables follow
 * BIT FOR BIT the trajectory of the problem on them alone: with M from svmb200_gram over a subset of rows kept in index
 * order, the problem of a cross-validation fold, whose training rows are some of M's rows.  Active variables must have
 * finite upper bounds > 0, and both signs must occur among them (SVMB200_ERR_ARG otherwise).  Answers as for
 * svmb200_smo_create_signed; svmb200_pg_state returns all n (SVR: 2n) variables, the inactive ones at alpha = 0.
 * svmb200_smo_run_batch takes these solvers next to the plain signed-view ones on the same M. */
int svmb200_smo_create_subset(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                              int hessian, const double* sign_host, const double* q_host, const double* ub_host,
                              const unsigned char* active_host, double tol, int64_t max_iter, svmb200_pg** out);
/* K14: `count` fresh resident or signed-view SMO solvers (svmb200_smo_create / _create_signed / _create_subset, not run
 * yet, none twice) on the same context, matrix, n, ld and layout, run to termination side by side: each problem gets its
 * own range of CTAs of one cooperative launch (at most one CTA per SM), keeps its own tol, max_iter, state and history, and ends
 * BIT-IDENTICAL to its own svmb200_pg_run.  Before every launch unfinished problems are admitted in index order while
 * their minimum grids (slices of at most 4 714 variables) fit the SMs, and the SMs are split evenly among them (no
 * problem above its own single-fit grid); a launch runs at most 4 096 iterations per problem; problems that finished give
 * their SMs to the others at the next launch.  Afterwards every solver answers svmb200_pg_state / _history / _scalars
 * / _stats (ms = the whole batch) as after svmb200_pg_run.  SVMB200_ERR_ARG for solvers of another kind, computed
 * rows, mixed matrices or layouts, a solver listed twice or one that has run.  SVMB200_SMO_BATCH_SMS caps the SMs the
 * batch uses, SVMB200_SMO_BATCH_CHUNK sets the iterations per launch (sweeps, tests).  iters / statuses: `count`
 * entries each (may be NULL).                                                                                      */
int svmb200_smo_run_batch(svmb200_pg* const* pgs, int count, int64_t* iters, int* statuses);
/* K12: the same SMO solver for problems whose Hessian does not fit in HBM.  No matrix is stored: every row of Q the
 * solver needs is computed from X on the device, Q_st = sign_s sign_t k(x_{s mod n}, x_{t mod n}) (PLAIN: nvars = n,
 * SVC with sign = the labels; SVR: nvars = 2n, sign = e), with K1's arithmetic for the kernel value (svmb200_gram with
 * dA = dB = X, same = 1, bias 0, no signs).  dX: n x d, row stride ldx (even, 16-byte aligned), kept alive by the caller
 * until svmb200_pg_destroy.  A row cache of cache_bytes (rounded down to whole rows of nvars doubles; 0: no cache) is
 * owned by the solver.  Hits and misses never change a bit of the trajectory.  At most svmb200_smo_max_vars(SMs)
 * variables (the shared-memory slice: 4 714 per SM); more is SVMB200_ERR_ARG.  Then svmb200_pg_run / _state / _history
 * / _scalars / _stats / _destroy as for svmb200_smo_create. */
int svmb200_smo_create_rows(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ldx, int64_t d, int kernel,
                            double gamma, double coef0, double degree, int hessian, const double* sign_host,
                            const double* q_host, const double* ub_host, double tol, int64_t max_iter, size_t cache_bytes,
                            svmb200_pg** out);
int64_t svmb200_smo_max_vars(int sm_count);
/* row source of an SMO solver (computed = 1: svmb200_smo_create_rows), cache slots, hits and misses so far (every row
 * computed without a cache counts as a miss); any output pointer may be NULL */
int svmb200_smo_cache_stats(svmb200_pg* pg, int* computed, int64_t* slots, int64_t* hits, int64_t* misses);
/* Shrinking (libsvm's, on by default in libsvm and sklearn) for any SMO solver (all row sources, subsets, batches),
 * before its first run; SVMB200_ERR_ARG once a run has started.  on = 0 turns it off again.  Variables at a bound that
 * cannot enter the maximal violating pair are set aside every min(l, 1000) states (l: the variables not held at 0);
 * their G is rebuilt from q and alpha before the solver stops, so svmb200_pg_state returns the full G.  A run with
 * shrinking follows its own trajectory (k_smo.cuh documents the rule); it does not depend on the grid or the batch. */
int svmb200_smo_set_shrinking(svmb200_pg* pg, int on);
/* active variables after the last shrink check (all variables without shrinking), shrink checks and gradient
 * reconstructions so far; any output pointer may be NULL */
int svmb200_smo_shrink_stats(svmb200_pg* pg, int64_t* active, int64_t* checks, int64_t* reconstructions);
/* dout[r][t] = k(X_{rows[r]}, X_t) for t < n (0 for t in [n, ldo)), unsigned, no bias: the values SMO's computed rows use */
int svmb200_kernel_rows(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ldx, int64_t d, int kernel, double gamma,
                        double coef0, double degree, const int64_t* rows_host, int64_t nrows, double* dout, int64_t ldo);
/* Advance by at most `max_new` iterations (< 0: run to termination; 0: only evaluate the state at
 * the current callback point, i.e. f, |d| and the stopping tests).  The callback point of the
 * reference (projected_gradient.py:95-98) is reached once per iteration; the state visible after
 * svmb200_pg_run returns is the state AT a callback point: x, f(x), g(x), |projected gradient|.  */
int svmb200_pg_run(svmb200_pg* pg, int64_t max_new, int64_t* iter, int* status);
int svmb200_pg_state(svmb200_pg* pg, double* x_host, double* g_host, double* f, double* ng);
/* scalars of the last evaluated state: {f, |d| (PG) or gap (FW), |d|^2 (PG) or best lower bound (FW), max_t,
 * last step, last d'Qd} */
int svmb200_pg_scalars(svmb200_pg* pg, double* vals6);
/* f and |d| at every callback point so far: (iter+1) values each (train_loss_history, ml/svm/_base.py:289-293) */
int svmb200_pg_history(svmb200_pg* pg, double* f_hist_host, double* ng_hist_host, int64_t* count);
/* timing of the last svmb200_pg_run: device milliseconds and number of Q passes (matvec launches) */
int svmb200_pg_stats(svmb200_pg* pg, float* ms, int64_t* passes, float* matvec_ms);
/* when on, ONE ITERATION IN 16 of svmb200_pg_run is bracketed by CUDA events: K2 (matvec_ms above), the all-gather
 * and K3 (events serialise the programmatic launches around them, so they are sampled); svmb200_pg_stats_ex returns
 * the three sums over the sampled iterations of the last run, svmb200_pg_profile_samples how many those were */
int svmb200_pg_set_profile(svmb200_pg* pg, int on);
int svmb200_pg_stats_ex(svmb200_pg* pg, float* matvec_ms, float* comm_ms, float* vector_ms);
int svmb200_pg_profile_samples(svmb200_pg* pg, int64_t* samples);
int svmb200_pg_is_symmetric(svmb200_pg* pg, int* on);   /* 1: products from the upper triangle (K2s above) */
int svmb200_pg_set_self_gram(svmb200_pg* pg, int on);    /* the matrix is a self-Gram of svmb200_gram (K2e above) */
int svmb200_pg_is_exact_symv(svmb200_pg* pg, int* on);   /* 1: products from the upper triangle with K2's bits (K2e) */
int svmb200_pg_device_x(svmb200_pg* pg, double** dx); /* device pointer of the iterate (nvars)     */
int svmb200_pg_destroy(svmb200_pg* pg);

/* ---- widening (SURVEY.md 8f-3): augmented-Lagrangian dual driven by a full-batch stochastic optimiser -----------
 * Replaces  AugmentedLagrangianQuadratic.function_jacobian (opti/constrained/_base.py:395-407), the Lagrangian
 * branches of Optimizer.callback / check_lagrangian_dual_optimality (opti/_base.py:94-149) and the loops of
 * opti/unconstrained/stochastic/{adagrad,gradient_descent,rmsprop,adadelta,adam,amsgrad,adamax}.py, i.e. what
 * SVC/SVR(dual=True, optimizer=AdaGrad, ...) runs for reg_intercept in {True, False} (ml/svm/_base.py:638-725,
 * 1188-1270):   min x'Qx/2 + q'x  s.t.  a'x = b (optional),  lb <= x <= ub,   relaxed with multipliers
 * (mu, lambda_lb, lambda_ub) and the penalty rho/2 |violations|^2; one optimiser step and one multiplier update per
 * iteration.  Same resident matrix, same one streaming pass per iteration (K2) as the box-constrained solvers; the
 * handle type and svmb200_pg_run / _state / _history / _stats / _destroy are shared.  With this solver
 * svmb200_pg_history's second array holds the primal cost x'Qx/2 + q'x (ml/svm/_base.py:289-291 stores that) and
 * svmb200_pg_state's `ng` the last one.
 *   a_host      equality row (nvars) or NULL;  x0_host is required (the reference draws it with NumPy on the host)
 *   step_sizes  `epochs` values (a constant learning rate repeated, or a schedule drawn in advance)
 *   momenta     epochs + 1 values, ignored (may be NULL) when momentum_type is NONE
 *   decay / beta1 / beta2 / offset: the rule's constants (ignored where the rule has none)                        */
#define SVMB200_RULE_ADAGRAD 0
#define SVMB200_RULE_SGD 1
#define SVMB200_RULE_RMSPROP 2
#define SVMB200_RULE_ADADELTA 3
#define SVMB200_RULE_ADAM 4
#define SVMB200_RULE_AMSGRAD 5
#define SVMB200_RULE_ADAMAX 6
#define SVMB200_MOMENTUM_NONE 0
#define SVMB200_MOMENTUM_POLYAK 1
#define SVMB200_MOMENTUM_NESTEROV 2
int svmb200_al_create(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                      int hessian, const double* q_host, const double* lb_host, const double* ub_host,
                      const double* x0_host, const double* a_host, double b, double rho, int rule, int momentum_type,
                      const double* step_sizes, const double* momenta, double decay, double beta1, double beta2,
                      double offset, double tol, int64_t epochs, svmb200_pg** out);
/* multipliers after (or during) a run: mu of the equality row (0 without one), lambda of  -x <= -lb  and  x <= ub */
int svmb200_al_multipliers(svmb200_pg* pg, double* mu, double* lam_lb_host, double* lam_ub_host);

/* ---- widening (SURVEY.md 8f-4): problems that share one resident matrix -- one-vs-rest, multi-target -------------
 * sklearn's OneVsRestClassifier(SVC(...)) (the pattern of ml/tests/test_svc.py:101-147) clones the estimator per class
 * and every clone rebuilds the same Gram matrix and streams its own Q = (y_c y_c') o (K + 1) -- the classes differ in
 * the label signs only.  Here M = K + bias is built ONCE without signs (svmb200_gram with NULL signs) and
 *   - a `_signed` solver poses its problem on Q = (s s') o M for a host vector s of +-1 (hessian must be PLAIN;
 *     sign_host NULL = the unsigned entry point): the vector kernels apply s to the operand and to the product,
 *     both exact, so the iterates are BIT-IDENTICAL to a solve on a materialised Q;
 *   - svmb200_pg_run_batch runs `count` fresh solvers of one kind (all PG, all FW or all AL, same max_iter) that
 *     share the matrix, shard and layout to termination in lockstep: per iteration ceil(count/4) passes over M
 *     (K2 with up to four vector operands per pass, per-vector results bit-identical to svmb200_matvec) and one
 *     vector launch for all problems.  Each solver keeps its own state / history / stopping test and afterwards
 *     answers svmb200_pg_state / _history / _scalars / _al_multipliers as after svmb200_pg_run.  Multi-GPU batches use
 *     the fused peer exchange (own arena region, one tag per iteration for all problems) when it is enabled and the
 *     region fits the arena, ncclAllGather per problem otherwise.  iters / statuses: `count` entries each (may be NULL).
 * Also usable without signs (SVR layout included): several right-hand sides q against one matrix
 * (sklearn MultiOutputRegressor(SVR(...))).                                                                         */
int svmb200_pg_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                             int hessian, const double* sign_host, const double* q_host, const double* lb_host,
                             const double* ub_host, const double* x0_host, double eps, int64_t max_iter, svmb200_pg** out);
int svmb200_fw_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                             int hessian, const double* sign_host, const double* q_host, const double* lb_host,
                             const double* ub_host, const double* x0_host, double eps, int64_t max_iter, double t,
                             svmb200_pg** out);
int svmb200_al_create_signed(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0, int64_t nrows,
                             int hessian, const double* sign_host, const double* q_host, const double* lb_host,
                             const double* ub_host, const double* x0_host, const double* a_host, double b, double rho,
                             int rule, int momentum_type, const double* step_sizes, const double* momenta, double decay,
                             double beta1, double beta2, double offset, double tol, int64_t epochs, svmb200_pg** out);
int svmb200_pg_run_batch(svmb200_pg* const* pgs, int count, int64_t* iters, int* statuses);
/* dw[b][i] = sum_j dQ[i][j] * du[b][j] for `count` device vectors against one pass (per four vectors) over dQ;
 * every dw[b] is bit-identical to svmb200_matvec(dQ, du[b]).  du / dw: host arrays of device pointers.             */
int svmb200_matvec_multi(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, const double* const* du,
                         double* const* dw, int count);

/* ---- one process, N GPUs ----------------------------------------------------------------------------------------
 * The reference's API is ONE Python process calling SVC.fit (ml/svm/_base.py:631-636).  svmb200_comm_local_group turns
 * n contexts of the calling thread (one per device) into ranks 0..n-1 whose exchange arenas are mapped by plain peer
 * access (no torchrun, no NCCL, no IPC).  Solvers created on such contexts (svmb200_{pg,fw,al}_create*, one per rank
 * with that rank's shard) defer their first product; svmb200_pg_start_group issues it for all ranks, and
 * svmb200_pg_run_group advances all of them, enqueuing iteration-major over the ranks.  State, history and statistics
 * are read from the rank-0 solver with the calls above (the state is replicated).                                    */
int svmb200_comm_local_group(svmb200_ctx** ctxs, int n, size_t arena_bytes);
/* device-to-device copy between two contexts of this process (replicates X over the ranks of the group) */
int svmb200_copy_peer(svmb200_ctx* dst_ctx, void* dst, svmb200_ctx* src_ctx, const void* src, size_t bytes);
int svmb200_pg_start_group(svmb200_pg* const* pgs, int count);
int svmb200_pg_run_group(svmb200_pg* const* pgs, int count, int64_t max_new, int64_t* iter, int* status);
/* svmb200_masked_product for all ranks of the group at once (dQ[r]: rank r's shard); v_host receives all n rows */
int svmb200_masked_product_group(svmb200_ctx* const* ctxs, const double* const* dQ, int count, int64_t n, int64_t ld,
                                 const double* beta_host, double* v_host);

/* ---- K5: masked product for the intercept ---------------------------------------------------
 * Replaces the Python loop  ml/svm/_base.py:877-880 / :1433-1437:
 * v[i] = sum_m M[i][m] * beta[m] over the rank's rows (all-gathered when a communicator is attached),
 * beta = host vector of n coefficients (alpha masked to the support set; SVR: alpha+ - alpha-).
 * The caller finishes b = mean_n (y_n - (s_n v_n - sum(beta s))) on the host (O(n)).           */
int svmb200_masked_product(svmb200_ctx* ctx, const double* dQ, int64_t n, int64_t ld, int64_t row0,
                           int64_t nrows, const double* beta_host, double* v_host);

/* ---- K6: decision function --------------------------------------------------------------------
 * Replaces  ml/svm/_base.py:284-287:  out[j] = sum_i dual_coef[i] k(SV_i, X_j) + b, computed in
 * column chunks without materialising the nsv x m kernel matrix on the host.                    */
int svmb200_decision(svmb200_ctx* ctx, const double* sv_host, int64_t nsv, const double* dual_coef_host,
                     const double* x_host, int64_t m, int64_t d, int kernel, double gamma, double coef0,
                     double degree, double intercept, double* out_host);

/* The same with the support vectors already in HBM (dsv: nsv x d doubles, leading dimension ldsv, even): what fit
 * leaves behind (svmb200_gather_rows), so that predict does not upload them again on every call.                */
int svmb200_decision_device(svmb200_ctx* ctx, const double* dsv, int64_t nsv, int64_t ldsv,
                            const double* dual_coef_host, const double* x_host, int64_t m, int64_t d, int kernel,
                            double gamma, double coef0, double degree, double intercept, double* out_host);

/* ---- device-side replacements of the O(n d) host steps of fit (csrc/devmath.cu) -------------------------------
 * X.var() of kernels.py:93, 127 (gamma='scale') over the rows x cols logical elements of a device matrix,
 * BIT-IDENTICAL to NumPy (same pairwise-summation tree), and the all-finite test of the input validation
 * (sklearn check_pairwise_arrays, kernels.py:50, 92, 126) in the same pass: *nonfinite = 1 if any element is NaN or
 * +-inf.  want_variance = 0: finite test only.                                                                      */
int svmb200_device_variance(svmb200_ctx* ctx, const double* dX, int64_t rows, int64_t cols, int64_t ld,
                            int want_variance, double* var, int* nonfinite);
/* support_vectors_ = X[sv] (ml/svm/_base.py:869, 1425) gathered in HBM: dOut[i][:] = dX[idx_host[i]][:], pad columns
 * zero.  Asynchronous on the context's stream.                                                                      */
int svmb200_gather_rows(svmb200_ctx* ctx, const double* dX, int64_t nrows_src, int64_t ld_src, int64_t d,
                        const int64_t* idx_host, int64_t nidx, double* dOut, int64_t ld_out);

/* ---- host-pointer convenience entry points (what a reference-side binding would call) ------- */
/* kernels.py Kernel.__call__(X, Y=None): out is nx x ny row-major on the host. y_host NULL => Y is X */
int svmb200_kernel_matrix_host(svmb200_ctx* ctx, const double* x_host, int64_t nx, const double* y_host,
                               int64_t ny, int64_t d, int kernel, double gamma, double coef0, double degree,
                               double* out_host);
/* ProjectedGradient(quad=Quadratic(Q,q), ub, lb, x).minimize() on a host-resident Q (n x n, ld = n) */
int svmb200_bcqp_pg_host(svmb200_ctx* ctx, const double* Q_host, const double* q_host, const double* lb_host,
                         const double* ub_host, const double* x0_host, int64_t n, double eps, int64_t max_iter,
                         double* x_out, double* g_out, double* f_hist, double* ng_hist, int64_t* iter,
                         int* status);

/* ---- host-side helpers of the fit path (no device involved; every rank of a sharded fit repeats them) ---------- */
/* Population variance of `count` contiguous doubles, BIT-IDENTICAL to NumPy's x.var() (pairwise summation of
 * numpy/_core/src/umath/loops_utils.h.src, two passes of numpy/_core/_methods.py _var), fused and spread over
 * `threads` host threads.  Replaces the X.var() of kernels.py:93, 127 (gamma='scale').                          */
int svmb200_host_variance(const double* x_host, int64_t count, int threads, double* var);
/* out[i][:] = x[idx[i]][:] for rows of d doubles: support_vectors_ = X[sv] (ml/svm/_base.py:869, 1425)          */
int svmb200_host_gather_rows(const double* x_host, int64_t d, const int64_t* idx, int64_t nidx, double* out, int threads);

#ifdef __cplusplus
}
#endif
#endif /* SVMB200_H */
