// Exploration harness for K2s (the symmetric pass, optiml_b200/csrc/k2_symv.cuh): times the PRODUCT kernels themselves
// (tile pass + combine) for several tile shapes on the C4-sized matrix (n = 50 000, 20 GB resident, 10 GB streamed),
// next to the full pass (K2) on the same matrix, and checks every shape against K2's product.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -o symv_sweep symv_sweep.cu
// Run:   ./symv_sweep [n]
#include "../optiml_b200/csrc/k2_symv.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <functional>

void svmb200_set_error(const char*, ...) {}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

// a symmetric matrix without storing a second copy: Q[i][j] = h(min(i,j), max(i,j))
__global__ void fill_sym(double* Q, long long n, long long ld) {
    const long long total = n * ld;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / ld, j = e % ld;
        double v = 0.0;
        if (j < n) {
            const unsigned long long a = (unsigned long long)(i < j ? i : j), b = (unsigned long long)(i < j ? j : i);
            unsigned long long h = a * 0x9E3779B97F4A7C15ull ^ (b + 0x632BE59BD9B4E019ull) * 0xC2B2AE3D27D4EB4Full;
            h ^= h >> 29;
            h *= 0xBF58476D1CE4E5B9ull;
            h ^= h >> 32;
            v = (double)(h >> 11) * (1.0 / 9007199254740992.0) - 0.5;
        }
        Q[e] = v;
    }
}
__global__ void fill_vec(double* u, long long n, long long ld) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < ld; i += (long long)gridDim.x * blockDim.x)
        u[i] = i < n ? 0.25 + 1e-3 * (double)(i % 997) - 0.4 * (double)(i % 3) : 0.0;
}

struct Bufs {
    double *Q, *u, *w, *wref, *wpart, *rowpart, *colpart, *den;
    unsigned* tickets;
    SymvItem* items;
    int* tables;
    long long n, ld;
};

static float time_launches(int reps, const std::function<void()>& f) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) f();
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) f();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaGetLastError());
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    return ms / reps;
}

template <class S>
void run_shape(const Bufs& b, int reps) {
    SymvPlan plan;
    symv_build_plan<S>(b.n, b.ld, 0, 1, b.n, plan, 2 * 148);
    const std::vector<SymvItem>& items = plan.items;
    CK(cudaMemcpy(b.items, items.data(), items.size() * sizeof(SymvItem), cudaMemcpyHostToDevice));
    std::vector<int> tables = plan.nseg;
    tables.insert(tables.end(), plan.band_of_unit.begin(), plan.band_of_unit.end());
    CK(cudaMemcpy(b.tables, tables.data(), tables.size() * sizeof(int), cudaMemcpyHostToDevice));
    const long long n_pad = (b.n + 15) / 16 * 16;
    SymvArgs a{b.Q, b.ld, b.n, 0, n_pad, b.u, b.rowpart, b.colpart, b.items, nullptr, nullptr};
    SymvCombineArgs c = {};
    c.rowpart = b.rowpart;
    c.colpart = b.colpart;
    c.ld = b.ld;
    c.nrows = b.n;
    c.row0 = 0;
    c.n_pad = n_pad;
    c.unit = plan.unit;
    c.nseg = b.tables;
    c.band_of_unit = b.tables + plan.nseg.size();
    c.u_rows = b.u;
    c.w = b.w;
    c.denpart = b.den;
    const unsigned ngroups = (unsigned)((b.n + MV_GROUP - 1) / MV_GROUP);
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, symv_tile_kernel<S>));
    int occ = 0;
    CK(cudaFuncSetAttribute(symv_tile_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::RING_BYTES));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, symv_tile_kernel<S>, SY_NT, S::RING_BYTES));
    CK(cudaMemset(b.w, 0xFF, b.n * 8));
    auto both = [&]() {
        CK(svm_launch_chained_smem(symv_tile_kernel<S>, dim3((unsigned)items.size()), dim3(SY_NT), (size_t)S::RING_BYTES, (cudaStream_t)0, a));
        CK(svm_launch_chained(symv_combine_kernel, dim3(ngroups), dim3(MV_GROUP * SY_CPARTS), (cudaStream_t)0, c));
    };
    const float ms_both = time_launches(reps, both);
    const float ms_tile = time_launches(reps, [&]() { CK(svm_launch_chained_smem(symv_tile_kernel<S>, dim3((unsigned)items.size()), dim3(SY_NT), (size_t)S::RING_BYTES, (cudaStream_t)0, a)); });
    const float ms_comb = time_launches(reps, [&]() { CK(svm_launch_chained(symv_combine_kernel, dim3(ngroups), dim3(MV_GROUP * SY_CPARTS), (cudaStream_t)0, c)); });
    // correctness against the full pass
    std::vector<double> w(b.n), wr(b.n);
    CK(cudaMemcpy(w.data(), b.w, b.n * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(wr.data(), b.wref, b.n * 8, cudaMemcpyDeviceToHost));
    double maxd = 0, maxw = 0;
    for (long long i = 0; i < b.n; ++i) {
        maxd = std::max(maxd, std::fabs(w[i] - wr[i]));
        maxw = std::max(maxw, std::fabs(wr[i]));
    }
    const double elems = (double)plan.streamed_elems;   // the upper triangle in band geometry
    printf("TR%-2d NRB%-2d NCH%d LB%-2d mb%d st%d BH%-3d BW%-4d items %5zu regs %3d occ %d | pass+combine %8.4f ms  tile %8.4f ms (%7.1f GB/s streamed)  "
           "combine %7.4f ms | vs full-pass bytes: %7.1f GB/s-equivalent | max|dw| %.2e (|w| %.1e)\n",
           S::TR, S::NRB, S::NCH, S::LB, S::MINB, S::STAGES, S::BH, S::BW, items.size(), fa.numRegs, occ, ms_both, ms_tile, 8.0 * elems / ms_tile / 1e6,
           ms_comb, 8.0 * (double)b.n * (double)b.ld / ms_both / 1e6, maxd, maxw);
    fflush(stdout);
}

// the tile pass of ONE rank of a P-rank solve, timed alone on this GPU (the plan, the shard's rows, no peers needed)
template <class S>
void run_rank(const Bufs& b, int reps, int P, int r, int slots) {
    const long long rpr = ((b.n + P - 1) / P + 63) / 64 * 64;
    SymvPlan plan;
    symv_build_plan<S>(b.n, b.ld, r, P, rpr, plan, slots);
    CK(cudaMemcpy(b.items, plan.items.data(), plan.items.size() * sizeof(SymvItem), cudaMemcpyHostToDevice));
    const long long n_pad = (plan.nrows + 15) / 16 * 16;
    SymvArgs a{b.Q + plan.row0 * b.ld, b.ld, plan.nrows, plan.row0, n_pad, b.u, b.rowpart, b.colpart, b.items, nullptr, nullptr};
    CK(cudaFuncSetAttribute(symv_tile_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::RING_BYTES));
    const float ms = time_launches(reps, [&]() { CK(svm_launch_chained_smem(symv_tile_kernel<S>, dim3((unsigned)plan.items.size()), dim3(SY_NT), (size_t)S::RING_BYTES, (cudaStream_t)0, a)); });
    int nshort = 0;
    for (long long I = 0; I + 1 < plan.nbands; ++I) nshort += plan.band_lr0[I + 1] - plan.band_lr0[I] < S::BH;
    printf("rank %d of %d (planned for %d slots): bands %lld (%d short) items %zu streamed %.4f GB | tile %8.4f ms = %7.1f GB/s\n", r, P, slots,
           plan.nbands, nshort, plan.items.size(), 8.0 * plan.streamed_elems / 1e9, ms, 8.0 * plan.streamed_elems / ms / 1e6);
    fflush(stdout);
}

int main(int argc, char** argv) {
    const long long n = argc > 1 ? atoll(argv[1]) : 50000;
    const int reps = argc > 2 ? atoi(argv[2]) : 100;
    const long long ld = (n + 15) / 16 * 16;
    Bufs b;
    b.n = n;
    b.ld = ld;
    const long long n_pad = (n + 15) / 16 * 16;
    CK(cudaMalloc(&b.Q, (size_t)n * ld * 8));
    CK(cudaMalloc(&b.u, ld * 8));
    CK(cudaMalloc(&b.w, n * 8));
    CK(cudaMalloc(&b.wref, n * 8));
    CK(cudaMalloc(&b.den, (n / MV_GROUP + 1) * 8));
    const int nseg = (int)((ld + MV_SEG - 1) / MV_SEG);
    CK(cudaMalloc(&b.wpart, (size_t)nseg * n_pad * 8));
    CK(cudaMalloc(&b.tickets, (n / MV_GROUP + 1) * 4));
    CK(cudaMemset(b.tickets, 0, (n / MV_GROUP + 1) * 4));
    CK(cudaMalloc(&b.rowpart, (size_t)(4 + 2 * ld / SY_CHUNK) * n_pad * 8));   // enough for BW >= 512, cut panels included
    CK(cudaMalloc(&b.colpart, (size_t)((n + 31) / 32 + 64) * ld * 8));      // enough for BH >= 32 and the short bands
    CK(cudaMalloc(&b.items, (size_t)((n + 31) / 32) * (2 + ld / SY_CHUNK) * sizeof(SymvItem)));
    CK(cudaMalloc(&b.tables, (size_t)(n + 64) * sizeof(int)));
    fill_sym<<<148 * 8, 256>>>(b.Q, n, ld);
    fill_vec<<<148, 256>>>(b.u, n, ld);
    CK(cudaDeviceSynchronize());
    // the full pass (K2) on the same matrix: reference product and reference time
    MatvecArgs m = {};
    m.Q = b.Q;
    m.ld = ld;
    m.nrows = n;
    m.u = b.u;
    m.w = b.wref;
    m.wpart = b.wpart;
    m.nrows_pad = n_pad;
    m.tickets = b.tickets;
    m.nseg = nseg;
    const long long ngroups = (n + MV_GROUP - 1) / MV_GROUP;
    const unsigned nitems = (unsigned)(ngroups * MV_BPG * nseg);
    const float ms_full = time_launches(reps / 2 + 1, [&]() { CK(svm_launch_chained(matvec_seg_kernel, dim3(nitems), dim3(MV_NT), (cudaStream_t)0, m)); });
    printf("n = %lld  ld = %lld   full pass (K2): %8.4f ms  %7.1f GB/s\n", n, ld, ms_full, 8.0 * n * ld / ms_full / 1e6);
    run_shape<SymvDefault>(b, reps);
    if (argc > 3 && strcmp(argv[3], "one") == 0) return 0;   // profiling runs: the shipped shape only
    if (argc > 3 && strcmp(argv[3], "bands") == 0) {          // band height / ring depth around the shipped shape
        run_shape<SymvShape<16, 8, 4, 8, 2, 2>>(b, reps);
        run_shape<SymvShape<16, 16, 4, 8, 2, 2>>(b, reps);
        run_shape<SymvShape<16, 12, 4, 8, 2, 2>>(b, reps);
        run_shape<SymvShape<16, 16, 4, 4, 2, 4>>(b, reps);
        run_shape<SymvDefault>(b, reps);
        run_shape<SymvShape<16, 16, 4, 8, 2, 2>>(b, reps);
        return 0;
    }
    if (argc > 3 && strcmp(argv[3], "bands2") == 0) {         // batch size / ring depth / band height, full matrix and shards
#define BOTH(...)                                         \
    run_shape<SymvShape<__VA_ARGS__>>(b, reps);           \
    run_rank<SymvShape<__VA_ARGS__>>(b, 2 * reps, 8, 0, 296); \
    run_rank<SymvShape<__VA_ARGS__>>(b, 2 * reps, 4, 0, 296);
        BOTH(16, 8, 4, 8, 2, 3)
        BOTH(16, 16, 4, 4, 2, 4)
        BOTH(16, 16, 4, 4, 2, 5)
        BOTH(16, 16, 4, 2, 2, 8)
        BOTH(16, 16, 4, 2, 2, 10)
        BOTH(16, 8, 4, 4, 2, 6)
        BOTH(16, 8, 4, 4, 2, 4)
        BOTH(16, 24, 4, 4, 2, 4)
        BOTH(16, 16, 4, 4, 2, 4)
        BOTH(16, 8, 4, 8, 2, 3)
#undef BOTH
        return 0;
    }
    if (argc > 4 && strcmp(argv[3], "shard") == 0) {         // the tile pass of single ranks of a P-rank solve
        const int P = atoi(argv[4]);
        for (int r : {0, P / 2, P - 1}) {
            run_rank<SymvDefault>(b, reps, P, r, 296);        // the graded plan
            run_rank<SymvDefault>(b, reps, P, r, 1 << 20);    // everything in "one wave": no grading (whole panels, tall bands)
        }
        return 0;
    }
    run_shape<SymvShape<16, 8, 4, 8, 2, 2>>(b, reps);
    run_shape<SymvShape<16, 8, 4, 4, 3, 4>>(b, reps);
    run_shape<SymvShape<16, 8, 4, 8, 3, 2>>(b, reps);
    run_shape<SymvShape<16, 8, 4, 4, 2, 6>>(b, reps);
    run_shape<SymvShape<16, 8, 4, 8, 1, 6>>(b, reps);
    run_shape<SymvShape<8, 16, 4, 8, 3, 2>>(b, reps);
    run_shape<SymvShape<16, 16, 4, 8, 2, 3>>(b, reps);
    run_shape<SymvShape<16, 8, 2, 8, 2, 3>>(b, reps);
    run_shape<SymvShape<32, 4, 4, 8, 2, 3>>(b, reps);
    run_shape<SymvShape<32, 8, 4, 8, 2, 3>>(b, reps);
    run_shape<SymvShape<16, 8, 8, 8, 2, 3>>(b, reps);
    run_shape<SymvShape<16, 8, 4, 8, 2, 3>>(b, reps);
    return 0;
}
