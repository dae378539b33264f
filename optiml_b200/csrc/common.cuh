// Shared declarations for the svmb200 library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <vector>

#include "../../include/svmb200.h"

constexpr int SVM_MAX_RANKS = 16;

struct svmb200_ctx {
    int device = -1;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint64_t launches = 0;
    // NCCL (loaded lazily through dlopen, see comm.cu)
    void* nccl_comm = nullptr;
    int rank = 0, nranks = 1;
    // cached TMA encoder (driver entry point fetched at run time: no link-time libcuda dependency)
    void* encode_tiled = nullptr;
    // segment partials / tickets of the streaming matvec (grown on demand, pg.cu)
    void* matvec_scratch = nullptr;
    // fused exchange over NVLink peer memory (comm.cu): every rank owns an arena that all peers map
    // through CUDA IPC; K2 stores self-validating tagged entries straight into every peer's arena (pg.cu)
    bool p2p_enabled = false;
    unsigned char* arena = nullptr;               // local arena
    size_t arena_bytes = 0;
    unsigned char* peer_arena[SVM_MAX_RANKS] = {};  // peer_arena[r] = rank r's arena as mapped here (self: local)
    unsigned long long xseq = 0;                  // number of fused exchanges issued so far (same on all ranks)
    // single-process group (svmb200_comm_local_group): the ranks are contexts of ONE host thread, the arenas are plain
    // peer pointers (cudaDeviceEnablePeerAccess, no IPC, no NCCL).  Solvers are then created with a deferred first
    // product and advanced by svmb200_pg_run_group, which enqueues iteration-major over the ranks.
    bool local_group = false;
    // solver workspace recycled between solves (pg.cu): one device slab, one pinned state block, an event pool.
    // cudaMalloc / cudaMallocHost / cudaEventCreate / cudaFree are slow and jittery (tens to hundreds of ms when
    // the host is busy); a fit issues none of them after the first one of its size.
    void* pg_slab = nullptr;
    size_t pg_slab_bytes = 0;
    bool pg_slab_busy = false;
    void* pg_pinned = nullptr;
    cudaEvent_t pg_ev0 = nullptr, pg_ev1 = nullptr, pg_ev_poll[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> event_pool;
    size_t event_pool_used = 0;
    // small per-call scratch, grown on demand and reused in stream order: row norms of K1, operands of K5
    void* norm_buf = nullptr;
    size_t norm_bytes = 0;
    void* mp_buf = nullptr;
    size_t mp_bytes = 0;
    // argument blocks of a batched solve (one VecArgs / ALArgs per problem, read by the batch vector kernels)
    void* batch_buf = nullptr;
    size_t batch_bytes = 0;
    // device-side X.var() (devmath.cu): leaf table of NumPy's pairwise tree, leaf sums, pinned staging -- cached per size
    void* var_cache = nullptr;
    // grid barrier of the persistent small-problem kernel (k_persistent.cuh): 256 zeroed bytes
    unsigned* gbar = nullptr;
    void* persist_buf = nullptr;   // w / product double buffers and the CTAs' private iterates
    size_t persist_bytes = 0;
    // opt-in: solvers created on this context take their products from the upper triangle of the (symmetric) matrix
    // (K2s, k2_symv.cuh); svmb200_ctx_set_symmetric, initial value from SVMB200_SYMMETRIC
    bool symmetric = false;
    // row indices of a device gather (support vectors)
    void* idx_buf = nullptr;
    size_t idx_bytes = 0;
};

// grow-only device scratch; safe to reuse without a sync because every user runs on ctx->stream
int svm_scratch_reserve(svmb200_ctx* ctx, void** buf, size_t* have, size_t need);

void svm_release_solver_cache(svmb200_ctx* ctx);
void svm_release_variance_cache(svmb200_ctx* ctx);

// arena layout
constexpr size_t ARENA_LOCAL_OFF = 256;    // [+8] int fault: set by a reader whose bounded spin expired
constexpr size_t ARENA_DATA_OFF = 1024;    // two gathered buffers of tagged 16-byte entries (double-buffered by sequence parity)

void svmb200_set_error(const char* fmt, ...);

#define SVM_CHECK_ARG(cond, msg)                                   \
    do {                                                           \
        if (!(cond)) {                                             \
            svmb200_set_error("%s: %s", __func__, msg);            \
            return SVMB200_ERR_ARG;                                \
        }                                                          \
    } while (0)

#define SVM_CUDA(call)                                                                                 \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            svmb200_set_error("%s:%d %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return SVMB200_ERR_CUDA;                                                                   \
        }                                                                                              \
    } while (0)

#define SVM_TRY(call)              \
    do {                           \
        int rc__ = (call);         \
        if (rc__ != SVMB200_OK) return rc__; \
    } while (0)

static inline int svm_use(svmb200_ctx* ctx) {
    if (!ctx) {
        svmb200_set_error("null context");
        return SVMB200_ERR_ARG;
    }
    SVM_CUDA(cudaSetDevice(ctx->device));
    return SVMB200_OK;
}

static inline int64_t round_up64(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

// Opt `kernel` in to `bytes` of dynamic shared memory, above the default 48 KB.  The attribute belongs to the device (a
// single-process device group launches one kernel on every GPU of the box from one process): set once per device index
// below 64, and on every call for any other index.
template <auto kernel>
static inline int svm_opt_in_smem(const svmb200_ctx* ctx, int bytes) {
    static bool done[64] = {};
    const bool tracked = ctx->device >= 0 && ctx->device < 64;
    if (tracked && done[ctx->device]) return SVMB200_OK;
    SVM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (tracked) done[ctx->device] = true;
    return SVMB200_OK;
}

// ---- programmatic dependent launch (PDL): the kernels of the solver loop form a strict chain (K2 -> K3 -> K2 ...), each
// a few hundred microseconds or less at 8 GPUs, so the 2-3 us between the end of one grid and the first instruction of the
// next are paid twice per iteration.  A kernel launched with the programmatic-serialisation attribute may be SCHEDULED
// while its predecessor is still running (as soon as every CTA of the predecessor has passed pdl_launch_dependents());
// its CTAs sit in pdl_wait() until the predecessor grid has completed and its memory is visible.  Correctness is that of
// the plain stream order: nothing is read or written before pdl_wait().
#ifndef SVMB200_HOST_EMULATION
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline cudaError_t svm_launch_chained_smem(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t svm_launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
    return svm_launch_chained_smem(kernel, grid, block, 0, stream, args...);
}
template <typename Arg>
static inline cudaError_t svm_launch_cooperative(void (*kernel)(Arg), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Arg arg) {
    void* params[] = {&arg};
    return cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), grid, block, params, smem, stream);
}
#else
template <typename Arg>
static inline cudaError_t svm_launch_cooperative(void (*kernel)(Arg), dim3 grid, dim3 block, size_t smem, cudaStream_t, Arg arg) {
    emu::launch_cooperative(grid, block, smem, [=]() { kernel(arg); });
    return cudaSuccess;
}
static inline void pdl_wait() {}
static inline void pdl_launch_dependents() {}
template <typename... KArgs, typename... Args>
static inline cudaError_t svm_launch_chained_smem(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t, Args... args) {
    emu::launch(grid, block, smem, [=]() { kernel(KArgs(args)...); });
    return cudaSuccess;
}
template <typename... KArgs, typename... Args>
static inline cudaError_t svm_launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
    return svm_launch_chained_smem(kernel, grid, block, 0, stream, args...);
}
#endif

// internal cross-file entry points
int svm_comm_allgather(svmb200_ctx* ctx, double* dbuf, int64_t count_per_rank);  // in place, on ctx->stream
void svm_release_matvec_scratch(svmb200_ctx* ctx);
int svm_launch_matvec(svmb200_ctx* ctx, const double* dQ, int64_t nrows, int64_t ld, const double* du, double* dw,
                      const int* d_done);
