// K1: Gram / Hessian build.  out = s_a s_b^T o (k(A, B) + bias), FP64.
//
// Restates  optiml/ml/svm/kernels.py:49-51 (linear), :91-95 (poly), :125-129 (gaussian through
// sklearn euclidean_distances: D = -2AB' + |a|^2 + |b|^2, max(D,0), diag = 0 when B is A) fused with
// optiml/ml/svm/_base.py:554,628 (Q = K o yy' + yy') / :1098-1099,1178 (M = K + 1).
//
// Structure (sm_100a): persistent CTAs of three warpgroups, 128x64 output tiles.
//   warpgroup 2 : TMA producers -- warp 8 / warp 9 (one elected lane each) feed one 4-stage ring per
//                 consumer group with cp.async.bulk.tensor 2D boxes (A: 128 rows x 16 doubles, B: 64 x 16,
//                 128 B inner extent, SWIZZLE_128B), mbarrier full/empty; registers handed back with
//                 setmaxnreg.dec.
//   warpgroups 0,1 : two consumer groups, one 128x64 tile each: FP64 tensor-core contraction
//                 (mma.sync.m8n8k4 -> DMMA; tcgen05 has no f64 kind; 64x32 accumulator block per warp,
//                 setmaxnreg.inc to 232 registers) followed by the fused exp/pow/sign/bias epilogue.
//                 DMMA and vector FP64 share ONE execution unit on B200 (scripts/fp64_probe.cu), so the
//                 epilogue cannot hide behind the other group's contraction; by default the two groups
//                 change phase together (named barrier), ping-pong and free-running are kept as measured
//                 alternatives (SVMB200_GRAM_EXCLUSIVE=1/0).
// Shared-memory reads are bank-conflict free: with the 128B swizzle the 16-byte chunk c of row r
// lives at chunk c^(r&7); the four k-slots of an m8n8k4 fragment are mapped to chunks {s, s+4}
// (s = k-step), so the 16 lanes of a half-warp hit 16 distinct 8-byte bank pairs.
#include "common.cuh"
#include "kernel_fn.cuh"   // exp8, ipow_rn, pow / tanh out of line (shared with K12)
#include <cudaTypedefs.h>
#include <math.h>
#include <stdlib.h>

namespace {

constexpr int BM = 128, BN = 64, BK = 16, STAGES = 4;
constexpr int GROUP_WARPS = 4;                      // warps per consumer group
constexpr int GRAM_THREADS = 384;                   // 2 consumer warpgroups + 1 producer warpgroup
constexpr int A_BYTES = BM * BK * 8;                // 16 KB
constexpr int B_BYTES = BN * BK * 8;                // 8 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;      // 24 KB
constexpr int RING_BYTES = STAGES * STAGE_BYTES;    // 96 KB per consumer group
constexpr int OPND_DOUBLES = 2 * BM + 2 * BN;         // per group: |a|^2, s_a for 128 rows; |b|^2, s_b for 64 columns
constexpr int GRAM_SMEM = 2 * RING_BYTES + 1024 + 4 * STAGES * 8 + 2 * OPND_DOUBLES * 8;
constexpr int BAR_GROUP0 = 1;                       // named barriers 1,2: "group g may use the tensor pipe"
constexpr int BAR_PHASE = 5;                        // named barrier 5: both groups change phase together (lockstep)
constexpr int BAR_LOCAL0 = 3;                       // named barriers 3,4: group-local sync around the operand staging

struct GramArgs {
    const double* norm_a;  // |a_i|^2 per row of A (gaussian) or null
    const double* norm_b;
    const double* sign_a;  // +-1 per row or null
    const double* sign_b;
    double* out;
    long long ldo;
    long long row0, nrows;  // rows of A handled by this launch
    long long nb;           // valid columns (rows of B)
    int kchunks;
    int tiles_m, tiles_n;
    int same;
    int exclusive;  // 0: groups run free; 1: ping-pong on the tensor pipe; 2: lockstep phases (see kernel)
    int backoff;    // 1: the producers sleep between polls of a full ring (default); 0: they spin (A/B: SVMB200_GRAM_BACKOFF)
    double gamma, coef0, degree, bias;
    int int_degree;  // degree when it is an integer in [1, 64] (poly: binary powering instead of pow()), else 0
};

#ifndef SVMB200_HOST_EMULATION
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// Producer-side wait: a producer whose ring is full has nothing to do until a consumer frees a stage (one k chunk of
// contraction, ~1 us; never during an epilogue phase).  Spinning on try_wait it issued 3.7e9 of the kernel's 9.5e9
// warp-instructions (profiles/r1_gram_kernel_sass_stalls.txt) in the two schedulers it shares with consumer warps,
// whose epilogue is issue-bound -- so it sleeps between polls (the ring is four stages deep: ~3 us of slack).
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) return;
        __nanosleep(128);
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
// The n x n output is written once and never read by this kernel; X (51 MB at C4) is re-read by every row of tiles.
// With default stores the 20 GB output stream evicted X from the 126 MB L2 again and again: 10.8 GB of DRAM reads for
// 51 MB of operands (profiles/r1_gram_kernel_ncu.txt).  Output stores carry an evict-first L2 policy instead.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void st_evict_first_f64x2(double* ptr, double2 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(ptr), "d"(v.x), "d"(v.y), "l"(pol) : "memory");
}
#define SVM_PTX(...) asm volatile(__VA_ARGS__)
#else
// tests/cuda_emu compiles this file for the host: the PTX wrappers map onto the emulation's shared-memory offsets,
// mbarriers (arrival count + transaction bytes + phase), tiled copies with the 128-byte swizzle, and a warp-collective
// m8n8k4 product; fences, register re-allocation and prefetches have no counterpart there
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return emu::smem_offset(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { emu::mbar_init(bar, count); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) { emu::mbar_arrive(bar, bytes); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { emu::mbar_arrive(bar, 0); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) { emu::mbar_wait(bar, parity); }
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) { emu::mbar_wait(bar, parity); }
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    emu::tma_load_2d(dst, map, bar, c0, c1);
}
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) { emu::dmma_m8n8k4(c0, c1, a, b); }
__device__ __forceinline__ uint64_t l2_evict_first_policy() { return 0; }
__device__ __forceinline__ void st_evict_first_f64x2(double* ptr, double2 v, uint64_t) { *reinterpret_cast<double2*>(ptr) = v; }
#define SVM_PTX(...) ((void)0)
#endif

#ifndef SVMB200_HOST_EMULATION
__device__ __forceinline__ void cp_async_8(double* smem_dst, const double* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
#else
__device__ __forceinline__ void cp_async_8(double* smem_dst, const double* gmem_src) { *smem_dst = *gmem_src; }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { emu::named_barrier(id, nthreads, true); }
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) { emu::named_barrier(id, nthreads, false); }
#endif

// Tile order.  A tile needs one 128-row A panel and one 64-row B panel; with the plain row-major order a B panel is
// re-read once per tile ROW, i.e. after a full sweep over X plus as many bytes of output stores: at C4 that thrashed the L2
// (10.8 GB of DRAM reads for 51 MB of operands, profiles/r1_gram_kernel_ncu.txt; 7.6 GB with evict-first stores).  Tiles
// are therefore enumerated in BANDS of GRAM_BAND tile rows, column by column inside a band: the ~300 tiles in flight
// share a handful of B panels and the band's A panels (4 MB), and X comes from DRAM once per band (tiles_m / 32 times).
constexpr int GRAM_BAND = 32;
__device__ __forceinline__ void tile_coords(int tile, int tiles_m, int tiles_n, int& tm, int& tn) {
    const int per_band = GRAM_BAND * tiles_n;
    const int band = tile / per_band, within = tile - band * per_band;
    const int rows = (tiles_m - band * GRAM_BAND) < GRAM_BAND ? (tiles_m - band * GRAM_BAND) : GRAM_BAND;
    tn = within / rows;
    tm = band * GRAM_BAND + (within - tn * rows);
}

template <bool V>
struct EdgeTile {
    static constexpr bool value = V;
};

template <int KERNEL>
__global__ void __launch_bounds__(GRAM_THREADS, 1)
gram_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const GramArgs p) {
#ifndef SVMB200_HOST_EMULATION
    extern __shared__ unsigned char smem_raw[];
#else
    unsigned char* smem_raw = emu::dynamic_smem();
#endif
    // 1024-byte alignment required by the 128B swizzle pattern -- as an OFFSET from the shared array, so that the compiler
    // keeps the address space and the fragment / operand loads below are LDS (an integer round-up of the generic address
    // turned all of them into generic LD: profiles/r1_gram_kernel_sass_stalls.txt)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * RING_BYTES);  // [group][full x STAGES | empty x STAGES]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int gq = 0; gq < 2; ++gq)
            for (int s = 0; s < STAGES; ++s) {
                mbar_init(smem_u32(bars + gq * 2 * STAGES + s), 1);
                mbar_init(smem_u32(bars + gq * 2 * STAGES + STAGES + s), GROUP_WARPS);
            }
        SVM_PTX("fence.mbarrier_init.release.cluster;" ::: "memory");
        SVM_PTX("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    const int ntiles = p.tiles_m * p.tiles_n;

    if (warp >= 2 * GROUP_WARPS) {
        // ===================== TMA producers: warp 8 -> ring 0, warp 9 -> ring 1 =====================
        SVM_PTX("setmaxnreg.dec.sync.aligned.u32 40;");
        const int grp = warp - 2 * GROUP_WARPS;
        if (grp < 2 && lane == 0) {
            SVM_PTX("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
            SVM_PTX("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
            const uint32_t ring = smem_u32(smem) + grp * RING_BYTES;
            const uint32_t full0 = smem_u32(bars + grp * 2 * STAGES), empty0 = full0 + 8 * STAGES;
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x + grp * gridDim.x; tile < ntiles; tile += 2 * gridDim.x) {
                int tm, tn;
                tile_coords(tile, p.tiles_m, p.tiles_n, tm, tn);
                const int arow = (int)p.row0 + tm * BM;
                const int brow = tn * BN;
                for (int kc = 0; kc < p.kchunks; ++kc) {
                    if (p.backoff) mbar_wait_backoff(empty0 + 8 * stage, phase ^ 1);
                    else mbar_wait(empty0 + 8 * stage, phase ^ 1);
                    const uint32_t fb = full0 + 8 * stage;
                    mbar_expect_tx(fb, STAGE_BYTES);
                    const uint32_t dst = ring + stage * STAGE_BYTES;
                    tma_load_2d(dst, &map_a, fb, kc * BK, arow);
                    tma_load_2d(dst + A_BYTES, &map_b, fb, kc * BK, brow);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
        return;
    }

    // ===================== consumer groups (ping-pong) =====================
    SVM_PTX("setmaxnreg.inc.sync.aligned.u32 232;");
    const int grp = warp / GROUP_WARPS;           // 0 or 1
    const int wg = warp % GROUP_WARPS;
    const int wm = wg >> 1, wn = wg & 1;          // 2 x 2 warps -> 64 x 32 per warp
    const int g = lane >> 2, t = lane & 3;
    // byte offset of this lane's k-slot inside a 128-byte row, before the per-step XOR
    const int hi = (t >> 1) * 4, sub = (t & 1) * 8;
    const unsigned char* ring = smem + grp * RING_BYTES;
    const uint32_t full0 = smem_u32(bars + grp * 2 * STAGES), empty0 = full0 + 8 * STAGES;
    // per-tile epilogue operands, staged with cp.async while the contraction runs
    double* opnd = reinterpret_cast<double*>(smem + 2 * RING_BYTES + 4 * STAGES * 8) + grp * OPND_DOUBLES;
    double* sm_na = opnd;
    double* sm_sa = opnd + BM;
    double* sm_nb = opnd + 2 * BM;
    double* sm_sb = opnd + 2 * BM + BN;
    const int gt = threadIdx.x - grp * GROUP_WARPS * 32;  // thread index inside the group
    int stage = 0;
    uint32_t phase = 0;
    // group 1 lets group 0 go first
    if (p.exclusive == 1 && grp == 1) named_bar_arrive(BAR_GROUP0 + 0, 2 * GROUP_WARPS * 32);

    // exclusive == 2: LOCKSTEP -- both groups contract together, then run their epilogues together.  DMMA and
    // vector FP64 share one execution unit on this part (scripts/fp64_probe.cu: mixed = sum of both), and a DMMA
    // holds it for 16 cycles, so an epilogue that runs beside the other group's contraction gets one FP64 issue
    // per DMMA and crawls; phases of the same kind must run together.
    const bool lockstep = p.exclusive == 2;
    const bool pingpong = p.exclusive == 1;
    const int rounds = (ntiles - (int)blockIdx.x + 2 * (int)gridDim.x - 1) / (2 * (int)gridDim.x);  // tiles of group 0
    for (int round = 0; round < rounds; ++round) {
        const int tile = blockIdx.x + (2 * round + grp) * gridDim.x;
        const bool has_tile = tile < ntiles;
        int tm = 0, tn = 0;
        if (has_tile) tile_coords(tile, p.tiles_m, p.tiles_n, tm, tn);
        double acc[8][4][2];
        if (has_tile) {
#pragma unroll
        for (int mi = 0; mi < 8; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
        // stage |a|^2, s_a (128 rows) and |b|^2, s_b (64 columns) of this tile: asynchronous 8-byte copies
        {
            const long long i = p.row0 + (long long)tm * BM + gt;
            const bool rok = i < p.row0 + p.nrows;
            if (KERNEL == SVMB200_KERNEL_GAUSSIAN && rok) cp_async_8(sm_na + gt, p.norm_a + i);
            else sm_na[gt] = 0.0;
            if (p.sign_a != nullptr && rok) cp_async_8(sm_sa + gt, p.sign_a + i);
            else sm_sa[gt] = 1.0;
            if (gt < BN) {
                const long long c = (long long)tn * BN + gt;
                const bool cok = c < p.nb;
                if (KERNEL == SVMB200_KERNEL_GAUSSIAN && cok) cp_async_8(sm_nb + gt, p.norm_b + c);
                else sm_nb[gt] = 0.0;
                if (p.sign_b != nullptr && cok) cp_async_8(sm_sb + gt, p.sign_b + c);
                else sm_sb[gt] = 1.0;
            }
            SVM_PTX("cp.async.commit_group;" ::: "memory");
        }
        // wait for the tensor pipe (the other group has finished its contraction)
        if (pingpong) named_bar_sync(BAR_GROUP0 + grp, 2 * GROUP_WARPS * 32);
        for (int kc = 0; kc < p.kchunks; ++kc) {
            mbar_wait(full0 + 8 * stage, phase);
            const unsigned char* sa = ring + stage * STAGE_BYTES + (wm * 64 + g) * 128;
            const unsigned char* sb = ring + stage * STAGE_BYTES + A_BYTES + (wn * 32 + g) * 128;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int off = (((s + hi) ^ g) << 4) + sub;
                double a[8], b[4];
#pragma unroll
                for (int mi = 0; mi < 8; ++mi) a[mi] = *reinterpret_cast<const double*>(sa + mi * 8 * 128 + off);
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) b[ni] = *reinterpret_cast<const double*>(sb + ni * 8 * 128 + off);
#pragma unroll
                for (int mi = 0; mi < 8; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty0 + 8 * stage);
            if (++stage == STAGES) {
                stage = 0;
                phase ^= 1;
            }
        }
        // hand the tensor pipe to the other group if it still has a tile to contract
        // (contractions alternate: this CTA's tile list is split even/odd between the groups, so the other
        // group's next contraction is the tile one grid stride after ours)
        if (pingpong && tile + (int)gridDim.x < ntiles) named_bar_arrive(BAR_GROUP0 + (grp ^ 1), 2 * GROUP_WARPS * 32);
        }  // has_tile (contraction)
        if (lockstep) named_bar_sync(BAR_PHASE, 2 * GROUP_WARPS * 32);
        if (has_tile) {

        // ---- fused epilogue: kernel function, bias, label signs, 128-bit stores
        const long long col_base = (long long)tn * BN + wn * 32 + 2 * t;
        SVM_PTX("cp.async.wait_all;" ::: "memory");
        named_bar_sync(BAR_LOCAL0 + grp, GROUP_WARPS * 32);  // every thread's staged operands are visible
        double nbv[4][2];
        unsigned sbh[4][2];  // sign bit of s_b
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int cl = wn * 32 + 2 * t + ni * 8 + e;
                nbv[ni][e] = sm_nb[cl];
                sbh[ni][e] = (unsigned)__double2hiint(sm_sb[cl]) & 0x80000000u;
            }
        }
        // Interior tiles -- every row inside the shard, every column a real column, no diagonal element (all but
        // O(n / 64) of the n^2 / 8192 tiles) -- take a copy of the epilogue with the per-element range and diagonal
        // tests compiled out: the ncu source view put ~45 of the ~70 instructions per output on the integer /
        // select side, and the epilogue is issue-bound (two warps per scheduler), not FP64-bound.
        const long long tile_r0 = p.row0 + (long long)tm * BM, tile_c0 = (long long)tn * BN;
        const bool edge = tile_r0 + BM > p.row0 + p.nrows || tile_c0 + BN > p.nb ||
                          (p.same && tile_r0 < tile_c0 + BN && tile_c0 < tile_r0 + BM);
        const bool tile_lower = tile_r0 >= tile_c0 + BN;   // an interior tile of a self-Gram lies wholly below the diagonal
        const uint64_t out_policy = l2_evict_first_policy();
        auto epilogue = [&](auto edge_tag) {
            constexpr bool EDGE = decltype(edge_tag)::value;
#pragma unroll
            for (int mi = 0; mi < 8; ++mi) {
                const long long i = p.row0 + (long long)tm * BM + wm * 64 + mi * 8 + g;  // row of A
                if (EDGE && i >= p.row0 + p.nrows) continue;
                const int rl = wm * 64 + mi * 8 + g;
                const unsigned sah = (unsigned)__double2hiint(sm_sa[rl]) & 0x80000000u;
                double* orow = p.out + (i - p.row0) * p.ldo;
                double val[8];
                if (KERNEL == SVMB200_KERNEL_GAUSSIAN) {
                    // D = (-2<a,b> + |a|^2) + |b|^2 ; clamp ; exact zero on the diagonal of a self-Gram.  In a self-Gram
                    // the norm of the smaller global index goes inside the fma, so out[t][s] == out[s][t] bit for bit
                    // (the upper triangle is sklearn's order; the lower one is its mirror)
                    const double na = sm_na[rl];
                    double x[8];
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const bool lower = p.same && (EDGE ? i > col_base + ni * 8 + e : tile_lower);
                            const double nlo = lower ? nbv[ni][e] : na, nhi = lower ? na : nbv[ni][e];
                            double dist = __dadd_rn(fma(-2.0, acc[mi][ni][e], nlo), nhi);  // -2<a,b> is exact
                            dist = dist < 0.0 ? 0.0 : dist;  // np.maximum(D, 0); select instead of fmax(), see exp8
                            if (EDGE && p.same && (i == col_base + ni * 8 + e)) dist = 0.0;
                            x[ni * 2 + e] = __dmul_rn(-p.gamma, dist);
                        }
                    exp8(x, val);
                } else if (KERNEL == SVMB200_KERNEL_POLY) {
                    if (p.int_degree > 0) {
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                            for (int e = 0; e < 2; ++e)  // separately rounded product and sum (NumPy semantics)
                                val[ni * 2 + e] = ipow_rn(__dadd_rn(__dmul_rn(p.gamma, acc[mi][ni][e]), p.coef0), p.int_degree);
                    } else {
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                            for (int e = 0; e < 2; ++e)
                                val[ni * 2 + e] = pow_outofline(__dadd_rn(__dmul_rn(p.gamma, acc[mi][ni][e]), p.coef0), p.degree);
                    }
                } else if (KERNEL == SVMB200_KERNEL_SIGMOID) {
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int e = 0; e < 2; ++e)  // kernels.py:197-201
                            val[ni * 2 + e] = tanh_outofline(__dadd_rn(__dmul_rn(p.gamma, acc[mi][ni][e]), p.coef0));
                } else {
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int e = 0; e < 2; ++e) val[ni * 2 + e] = acc[mi][ni][e];
                }
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    const long long c = col_base + ni * 8;
                    if (EDGE && c >= p.ldo) continue;
                    double2 v;
                    double* ve = reinterpret_cast<double*>(&v);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        double o = 0.0;
                        if (!EDGE || c + e < p.nb) {
                            o = val[ni * 2 + e];
                            if (p.bias != 0.0) o = __dadd_rn(o, p.bias);
                            // times s_a s_b = +-1: flip the sign bit (integer pipe, not the shared FP64 unit)
                            o = __hiloint2double(__double2hiint(o) ^ (int)(sah ^ sbh[ni][e]), __double2loint(o));
                        }
                        ve[e] = o;
                    }
                    st_evict_first_f64x2(orow + c, v, out_policy);
                }
            }
        };
        if (edge) epilogue(EdgeTile<true>());
        else epilogue(EdgeTile<false>());
        named_bar_sync(BAR_LOCAL0 + grp, GROUP_WARPS * 32);  // operands free for the next tile's staging
        }  // has_tile (epilogue)
        if (lockstep) named_bar_sync(BAR_PHASE, 2 * GROUP_WARPS * 32);
    }
}


// ------------------------------------------------------------------------------------------------
// Laplacian kernel (widening, SURVEY.md 8f-2): k(a,b) = exp(-gamma * sum_k |a_k - b_k|)
// (optiml/ml/svm/kernels.py:159-163 -> sklearn manhattan_distances -> scipy cdist 'cityblock': a sequential
// sum over k).  Not a contraction: CUDA-core tile kernel, 128x128 outputs per CTA, 8x8 per thread, operands
// staged (transposed) in shared memory 16 features at a time, the same k order as the reference so the
// distances are bit-identical; exp8 epilogue, bias, label signs, zero pad columns as in gram_kernel.
constexpr int LT = 128, LKC = 16, LPAD = 2, LAP_THREADS = 256;

struct LapArgs {
    const double *A, *B;
    long long lda, ldb, na, nb, d;
    const double *sign_a, *sign_b;
    double* out;
    long long ldo, row0, nrows;
    double gamma, bias;
};

__global__ void __launch_bounds__(LAP_THREADS) laplacian_kernel(const LapArgs p) {
    __shared__ __align__(16) double As[LKC][LT + LPAD];
    __shared__ __align__(16) double Bs[LKC][LT + LPAD];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const long long i0 = p.row0 + (long long)blockIdx.y * LT;   // first row of A in this tile
    const long long j0 = (long long)blockIdx.x * LT;            // first row of B (= output column)
    double acc[8][8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[r][c] = 0.0;
    double ra[8], rb[8];
    auto fetch = [&](long long kc) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int e = tid + j * LAP_THREADS, row = e >> 4, k = e & 15;
            const long long ia = i0 + row, jb = j0 + row, kk = kc + k;
            ra[j] = (ia < p.row0 + p.nrows && kk < p.d) ? p.A[ia * p.lda + kk] : 0.0;
            rb[j] = (jb < p.nb && kk < p.d) ? p.B[jb * p.ldb + kk] : 0.0;
        }
    };
    fetch(0);
    for (long long kc = 0; kc < p.d; kc += LKC) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int e = tid + j * LAP_THREADS, row = e >> 4, k = e & 15;
            As[k][row] = ra[j];
            Bs[k][row] = rb[j];
        }
        __syncthreads();
        if (kc + LKC < p.d) fetch(kc + LKC);  // next chunk's global loads overlap the arithmetic below
#pragma unroll 4
        for (int k = 0; k < LKC; ++k) {
            double a[8], b[8];
#pragma unroll
            for (int r = 0; r < 8; r += 2) {
                const double2 v = *reinterpret_cast<const double2*>(&As[k][ty * 8 + r]);
                a[r] = v.x;
                a[r + 1] = v.y;
                const double2 w = *reinterpret_cast<const double2*>(&Bs[k][tx * 8 + r]);
                b[r] = w.x;
                b[r + 1] = w.y;
            }
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = __dadd_rn(acc[r][c], fabs(__dsub_rn(a[r], b[c])));
        }
    }
    // epilogue
    unsigned sbh[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const long long col = j0 + tx * 8 + c;
        sbh[c] = (p.sign_b != nullptr && col < p.nb) ? ((unsigned)__double2hiint(p.sign_b[col]) & 0x80000000u) : 0u;
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const long long i = i0 + ty * 8 + r;
        if (i >= p.row0 + p.nrows) continue;
        const unsigned sah = (p.sign_a != nullptr) ? ((unsigned)__double2hiint(p.sign_a[i]) & 0x80000000u) : 0u;
        double x[8], val[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) x[c] = __dmul_rn(-p.gamma, acc[r][c]);
        exp8(x, val);
        double* orow = p.out + (i - p.row0) * p.ldo;
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            const long long col = j0 + tx * 8 + c;
            if (col >= p.ldo) continue;
            double2 v;
            double* ve = reinterpret_cast<double*>(&v);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                double o = 0.0;
                if (col + e < p.nb) {
                    o = val[c + e];
                    if (p.bias != 0.0) o = __dadd_rn(o, p.bias);
                    o = __hiloint2double(__double2hiint(o) ^ (int)(sah ^ sbh[c + e]), __double2loint(o));
                }
                ve[e] = o;
            }
            *reinterpret_cast<double2*>(orow + col) = v;
        }
    }
}

// |x_i|^2 per row: one warp per row, fixed lane-strided order + butterfly
__global__ void row_sqnorm_kernel(const double* __restrict__ X, long long n, long long ld, long long d,
                                  double* __restrict__ out) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const int lane = threadIdx.x & 31;
    const double* x = X + row * ld;
    double s = 0.0;
    for (long long k = lane; k < d; k += 32) s = fma(x[k], x[k], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row] = s;
}

int make_tensor_map(svmb200_ctx* ctx, CUtensorMap* map, const double* base, int64_t rows, int64_t d, int64_t ld,
                    int box_rows) {
    if (!ctx->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        SVM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || fn == nullptr) {
            svmb200_set_error("cuTensorMapEncodeTiled is not available from this driver");
            return SVMB200_ERR_CUDA;
        }
        ctx->encode_tiled = fn;
    }
    auto encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ctx->encode_tiled);
    cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(double)};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        svmb200_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld d=%lld ld=%lld)", (int)r,
                          (long long)rows, (long long)d, (long long)ld);
        return SVMB200_ERR_CUDA;
    }
    return SVMB200_OK;
}

template <int KERNEL>
int launch_gram(svmb200_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb, const GramArgs& args) {
    SVM_TRY(svm_opt_in_smem<gram_kernel<KERNEL>>(ctx, GRAM_SMEM));
    const int ntiles = args.tiles_m * args.tiles_n;
    const int grid = ntiles < ctx->sm_count ? ntiles : ctx->sm_count;
    gram_kernel<KERNEL><<<grid, GRAM_THREADS, GRAM_SMEM, ctx->stream>>>(ma, mb, args);
    ctx->launches++;
    SVM_CUDA(cudaGetLastError());
    return SVMB200_OK;
}

// K12: the listed rows of the unsigned kernel matrix, one thread per element, through kfn_value (kernel_fn.cuh)
__global__ void kernel_rows_kernel(const KernelFn p, long long n, const long long* __restrict__ rows, long long nrows,
                                   double* __restrict__ out, long long ldo) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ldo) return;
    for (long long r = blockIdx.y; r < nrows; r += gridDim.y) out[r * ldo + t] = t < n ? kfn_value(p, rows[r], t) : 0.0;
}

}  // namespace

extern "C" int64_t svmb200_padded_ld(int64_t ncols) { return round_up64(ncols < 1 ? 1 : ncols, 16); }

extern "C" int svmb200_gram(svmb200_ctx* ctx, const double* dA, int64_t na, int64_t lda, const double* dB, int64_t nb,
                            int64_t ldb, int64_t d, int same, int kernel, double gamma, double coef0, double degree,
                            const double* dsign_a, const double* dsign_b, double bias, int64_t row0, int64_t nrows,
                            double* dout, int64_t ldo) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dA && dB && dout, "null matrix");
    SVM_CHECK_ARG(na > 0 && nb > 0 && d > 0, "empty operand");
    SVM_CHECK_ARG(lda >= d && ldb >= d && lda % 2 == 0 && ldb % 2 == 0, "lda/ldb must be even and >= d (16-byte row stride for TMA)");
    SVM_CHECK_ARG((reinterpret_cast<uintptr_t>(dA) & 15) == 0 && (reinterpret_cast<uintptr_t>(dB) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(dout) & 15) == 0, "matrices must be 16-byte aligned");
    SVM_CHECK_ARG(ldo >= nb && ldo % 2 == 0, "ldo must be even and >= nb");
    SVM_CHECK_ARG(row0 >= 0 && nrows >= 0 && row0 + nrows <= na, "row range outside A");
    SVM_CHECK_ARG(kernel >= SVMB200_KERNEL_LINEAR && kernel <= SVMB200_KERNEL_LAPLACIAN, "unknown kernel id");
    SVM_CHECK_ARG((kernel != SVMB200_KERNEL_GAUSSIAN && kernel != SVMB200_KERNEL_LAPLACIAN) || gamma >= 0.0,
                  "gamma must be >= 0 for the gaussian / laplacian kernels");
    SVM_CHECK_ARG(na < (1ll << 31) && nb < (1ll << 31) && d < (1ll << 31), "dimension too large");
    if (nrows == 0) return SVMB200_OK;

    if (kernel == SVMB200_KERNEL_LAPLACIAN) {
        LapArgs a;
        a.A = dA;
        a.B = dB;
        a.lda = lda;
        a.ldb = ldb;
        a.na = na;
        a.nb = nb;
        a.d = d;
        a.sign_a = dsign_a;
        a.sign_b = dsign_b;
        a.out = dout;
        a.ldo = ldo;
        a.row0 = row0;
        a.nrows = nrows;
        a.gamma = gamma;
        a.bias = bias;
        dim3 grid((unsigned)((ldo + LT - 1) / LT), (unsigned)((nrows + LT - 1) / LT));
        SVM_CHECK_ARG(grid.y <= 65535, "row range too large for one launch");
        laplacian_kernel<<<grid, LAP_THREADS, 0, ctx->stream>>>(a);
        ctx->launches++;
        SVM_CUDA(cudaGetLastError());
        return SVMB200_OK;
    }

    double *norm_a = nullptr, *norm_b = nullptr;
    if (kernel == SVMB200_KERNEL_GAUSSIAN) {
        const bool shared_norms = (dB == dA && nb == na);
        SVM_TRY(svm_scratch_reserve(ctx, &ctx->norm_buf, &ctx->norm_bytes, (size_t)(na + (shared_norms ? 0 : nb)) * sizeof(double)));
        norm_a = static_cast<double*>(ctx->norm_buf);
        const int wpb = 8;
        row_sqnorm_kernel<<<(unsigned)((na + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(dA, na, lda, d, norm_a);
        ctx->launches++;
        if (shared_norms) {
            norm_b = norm_a;
        } else {
            norm_b = norm_a + na;
            row_sqnorm_kernel<<<(unsigned)((nb + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(dB, nb, ldb, d, norm_b);
            ctx->launches++;
        }
    }
    int rc = SVMB200_OK;
    CUtensorMap ma, mb;
    rc = make_tensor_map(ctx, &ma, dA, na, d, lda, BM);
    if (rc == SVMB200_OK) rc = make_tensor_map(ctx, &mb, dB, nb, d, ldb, BN);
    if (rc == SVMB200_OK) {
        GramArgs a;
        a.norm_a = norm_a;
        a.norm_b = norm_b;
        a.sign_a = dsign_a;
        a.sign_b = dsign_b;
        a.out = dout;
        a.ldo = ldo;
        a.row0 = row0;
        a.nrows = nrows;
        a.nb = nb;
        a.kchunks = (int)((d + BK - 1) / BK);
        a.tiles_m = (int)((nrows + BM - 1) / BM);
        a.tiles_n = (int)((ldo + BN - 1) / BN);
        a.same = same;
        {
            // phase lock-step when there is an epilogue (see kernel comment); SVMB200_GRAM_EXCLUSIVE=0/1/2 overrides
            const char* ev = getenv("SVMB200_GRAM_EXCLUSIVE");
            a.exclusive = ev ? atoi(ev) : (kernel != SVMB200_KERNEL_LINEAR ? 2 : 0);
            const char* bo = getenv("SVMB200_GRAM_BACKOFF");
            a.backoff = bo ? atoi(bo) : 1;
        }
        a.gamma = gamma;
        a.coef0 = coef0;
        a.degree = degree;
        a.bias = bias;
        a.int_degree = svm_gram_int_degree(degree);
        if (kernel == SVMB200_KERNEL_LINEAR) rc = launch_gram<SVMB200_KERNEL_LINEAR>(ctx, ma, mb, a);
        else if (kernel == SVMB200_KERNEL_POLY) rc = launch_gram<SVMB200_KERNEL_POLY>(ctx, ma, mb, a);
        else if (kernel == SVMB200_KERNEL_SIGMOID) rc = launch_gram<SVMB200_KERNEL_SIGMOID>(ctx, ma, mb, a);
        else rc = launch_gram<SVMB200_KERNEL_GAUSSIAN>(ctx, ma, mb, a);
    }
    return rc;
}

int svm_gram_int_degree(double degree) {
    if (getenv("SVMB200_POLY_LIBM_POW") != nullptr && atoi(getenv("SVMB200_POLY_LIBM_POW")) != 0) return 0;  // A/B
    return (degree >= 1.0 && degree <= 64.0 && degree == (double)(int)degree) ? (int)degree : 0;
}

int svm_row_sqnorms(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ld, int64_t d, double* out) {
    const int wpb = 8;
    row_sqnorm_kernel<<<(unsigned)((n + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(dX, n, ld, d, out);
    ctx->launches++;
    SVM_CUDA(cudaGetLastError());
    return SVMB200_OK;
}

extern "C" int svmb200_kernel_rows(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ldx, int64_t d, int kernel,
                                   double gamma, double coef0, double degree, const int64_t* rows_host, int64_t nrows,
                                   double* dout, int64_t ldo) {
    SVM_TRY(svm_use(ctx));
    SVM_CHECK_ARG(dX != nullptr && dout != nullptr, "null matrix");
    SVM_CHECK_ARG(n > 0 && d > 0 && nrows >= 0, "empty operand");
    SVM_CHECK_ARG(ldx >= d && ldx % 2 == 0 && (reinterpret_cast<uintptr_t>(dX) & 15) == 0,
                  "ldx must be even and >= d, X 16-byte aligned");
    SVM_CHECK_ARG(ldo >= n, "ldo must be >= n");
    SVM_CHECK_ARG(kernel >= SVMB200_KERNEL_LINEAR && kernel <= SVMB200_KERNEL_LAPLACIAN, "unknown kernel id");
    SVM_CHECK_ARG((kernel != SVMB200_KERNEL_GAUSSIAN && kernel != SVMB200_KERNEL_LAPLACIAN) || gamma >= 0.0,
                  "gamma must be >= 0 for the gaussian / laplacian kernels");
    SVM_CHECK_ARG(n < (1ll << 31) && d < (1ll << 31), "dimension too large");
    if (nrows == 0) return SVMB200_OK;
    SVM_CHECK_ARG(rows_host != nullptr, "null row list");
    for (int64_t r = 0; r < nrows; ++r) SVM_CHECK_ARG(rows_host[r] >= 0 && rows_host[r] < n, "row index out of range");
    const size_t idx_bytes = (size_t)nrows * sizeof(long long), sq_bytes = kernel == SVMB200_KERNEL_GAUSSIAN ? (size_t)n * sizeof(double) : 0;
    SVM_TRY(svm_scratch_reserve(ctx, &ctx->idx_buf, &ctx->idx_bytes, idx_bytes));
    cudaStream_t s = ctx->stream;
    SVM_CUDA(cudaMemcpyAsync(ctx->idx_buf, rows_host, idx_bytes, cudaMemcpyHostToDevice, s));
    KernelFn p;
    p.X = dX;
    p.ldx = ldx;
    p.d = d;
    p.sqn = nullptr;
    p.kernel = kernel;
    p.gamma = gamma;
    p.coef0 = coef0;
    p.degree = degree;
    p.int_degree = svm_gram_int_degree(degree);
    if (sq_bytes) {
        SVM_TRY(svm_scratch_reserve(ctx, &ctx->norm_buf, &ctx->norm_bytes, sq_bytes));
        p.sqn = static_cast<double*>(ctx->norm_buf);
        SVM_TRY(svm_row_sqnorms(ctx, dX, n, ldx, d, static_cast<double*>(ctx->norm_buf)));
    }
    const unsigned nt = 256;
    dim3 grid((unsigned)((ldo + nt - 1) / nt), (unsigned)(nrows < 65535 ? nrows : 65535));
    kernel_rows_kernel<<<grid, nt, 0, s>>>(p, n, static_cast<const long long*>(ctx->idx_buf), nrows, dout, ldo);
    ctx->launches++;
    SVM_CUDA(cudaGetLastError());
    SVM_CUDA(cudaStreamSynchronize(s));  // pageable row list: the caller may reuse it right away
    return SVMB200_OK;
}
