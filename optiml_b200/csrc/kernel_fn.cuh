// K12: one kernel value k(x_s, x_t) from X, for every kernel of K1 (gram.cu), with K1's arithmetic.
//
// SMO on problems whose Hessian does not fit in HBM computes the rows of Q it needs from X (k_smo.cuh, computed rows).
// kfn_value is the value K1 writes at out[s][t] for dA = dB = X, same = 1, bias 0 and no signs:
//   dot      per 16-feature chunk (K1's TMA box, features past d are its zero fill) four m8n8k4 steps; step s takes the
//            features 2s, 2s+1, 2s+8, 2s+9 (the k-slots 0..3 of K1's fragments, see gram.cu) -- one fma chain in that
//            order, which is how the host emulation evaluates K1's DMMA.  Whether the B200's DMMA rounds as that chain
//            does is measured, not assumed (tests/test_gpu_smo_rows.py).
//   gaussian exp(-gamma max(0, fma(-2, dot, |x_lo|^2) + |x_hi|^2)), lo = min(s, t), hi = max(s, t), distance 0 when
//            s == t; |x|^2 from K1's row_sqnorm_kernel
//   poly     (gamma dot + coef0)^degree: ipow_rn for integer degrees in [1, 64], pow otherwise
//   sigmoid  tanh(gamma dot + coef0)
//   laplacian exp(-gamma sum_k |x_sk - x_tk|), summed in feature order (laplacian_kernel)
// A value depends on (x_s, x_t, the kernel parameters) only -- never on the grid, the slice or the thread.
#pragma once
#include "common.cuh"
#include <math.h>

#ifdef SVMB200_HOST_EMULATION
#define KFN_NOINLINE EMU_NOINLINE
#else
#define KFN_NOINLINE __noinline__
#endif

namespace {

// pow() stays out of line (the poly epilogue is unrolled 64x per thread and pow is ~300 instructions).
__device__ KFN_NOINLINE double pow_outofline(double x, double y) { return pow(x, y); }
// x ** n for a small positive integer n (PolyKernel's default degree = 3, kernels.py:79, 95) by binary powering with
// separately rounded products: n = 2 is NumPy's own fast path (np.square, exact same bits); n = 3 is (x*x)*x, two
// roundings against libm pow's one (<= ~1.5 ulp apart, SURVEY.md A.12: far inside the 1e-12 Gram bar).  pow() was
// ~300 instructions per output and made the poly Gram 6x slower than the Gaussian one per element.
__device__ __forceinline__ double ipow_rn(double x, int n) {
    double r = 1.0, b = x;
    bool first = true;
    for (;;) {
        if (n & 1) {
            r = first ? b : __dmul_rn(r, b);
            first = false;
        }
        n >>= 1;
        if (n == 0) break;
        b = __dmul_rn(b, b);
    }
    return r;
}
__device__ KFN_NOINLINE double tanh_outofline(double x) { return tanh(x); }

// exp(x), x <= 0, for the Gaussian epilogue, evaluated for EIGHT independent arguments in lock-step so
// that the FP64 unit sees 8 independent dependency chains (a scalar exp() is one chain of dependent DFMAs,
// 9.4 cycles each).  Classic scheme: k = rint(x log2 e) through the 1.5*2^52 trick, r = x - k ln2 (hi/lo
// split), degree-13 Taylor polynomial on |r| <= ln2/2 (truncation 6e-18), then 2^k in two exact steps
// (2^(k+1000) on the exponent field, times 2^-1000) so that results in the denormal range are rounded once
// and everything below underflows to 0 -- no branch, no call.  <= 1.5 ulp; exp8(0) == 1 exactly.
__device__ __forceinline__ void exp8(const double (&x)[8], double (&out)[8]) {
    constexpr double L2E = 1.4426950408889634074, MAGIC = 6755399441055744.0;
    constexpr double LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10;
    constexpr double TWO_M1000 = 9.33263618503218878990e-302;  // 2^-1000
    double r[8], p[8];
    int k[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        // exp(-800) == 0 in FP64; keeps k in range.  A compare + select, not fmax(): fmax's NaN rule costs DSETP + 2 SEL +
        // LOP3 + moves (7 instructions), the select 3, and the results agree for every non-NaN argument
        const double xe = x[e] < -800.0 ? -800.0 : x[e];
        double t = fma(xe, L2E, MAGIC);
        k[e] = __double2loint(t);
        t -= MAGIC;
        r[e] = fma(t, -LN2_HI, xe);
        r[e] = fma(t, -LN2_LO, r[e]);
        p[e] = 1.0 / 6227020800.0;  // 1/13!
    }
    constexpr double C[13] = {1.0, 1.0, 1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320,
                              1.0 / 362880, 1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600};
#pragma unroll
    for (int j = 12; j >= 0; --j) {
#pragma unroll
        for (int e = 0; e < 8; ++e) p[e] = fma(p[e], r[e], C[j]);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e)
        out[e] = __hiloint2double(__double2hiint(p[e]) + ((k[e] + 1000) << 20), __double2loint(p[e])) * TWO_M1000;
}

// one lane of exp8: the same operations in the same order, so exp1(x) == exp8 of x bit for bit
__device__ __forceinline__ double exp1(double x) {
    constexpr double L2E = 1.4426950408889634074, MAGIC = 6755399441055744.0;
    constexpr double LN2_HI = 6.93147180369123816490e-01, LN2_LO = 1.90821492927058770002e-10;
    constexpr double TWO_M1000 = 9.33263618503218878990e-302;
    const double xe = x < -800.0 ? -800.0 : x;
    double t = fma(xe, L2E, MAGIC);
    const int k = __double2loint(t);
    t -= MAGIC;
    double r = fma(t, -LN2_HI, xe);
    r = fma(t, -LN2_LO, r);
    double p = 1.0 / 6227020800.0;
    constexpr double C[13] = {1.0, 1.0, 1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320,
                              1.0 / 362880, 1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600};
#pragma unroll
    for (int j = 12; j >= 0; --j) p = fma(p, r, C[j]);
    return __hiloint2double(__double2hiint(p) + ((k + 1000) << 20), __double2loint(p)) * TWO_M1000;
}

}  // namespace

// X (n x d, row stride ldx, 16-byte aligned rows) and the resolved kernel
struct KernelFn {
    const double* X;
    long long ldx, d;
    const double* sqn;  // |x_s|^2 per row (gaussian), else null
    int kernel;
    double gamma, coef0, degree;
    int int_degree;     // as K1: degree when it is an integer in [1, 64], else 0 (pow)
};

// 16 features of a row starting at k0: vector loads for a whole chunk, the zero fill past d otherwise
__device__ __forceinline__ void kfn_chunk(const double* x, long long k0, long long d, double (&v)[16]) {
    if (k0 + 16 <= d) {
#pragma unroll
        for (int e = 0; e < 16; e += 2) {
            const double2 w = __ldg(reinterpret_cast<const double2*>(x + k0 + e));
            v[e] = w.x;
            v[e + 1] = w.y;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] = k0 + e < d ? __ldg(x + k0 + e) : 0.0;
    }
}

__device__ __forceinline__ double kfn_dot(const double* a, const double* b, long long d) {
    double acc = 0.0;
    for (long long k0 = 0; k0 < d; k0 += 16) {
        double va[16], vb[16];
        kfn_chunk(a, k0, d, va);
        kfn_chunk(b, k0, d, vb);
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            acc = fma(va[2 * s], vb[2 * s], acc);
            acc = fma(va[2 * s + 1], vb[2 * s + 1], acc);
            acc = fma(va[2 * s + 8], vb[2 * s + 8], acc);
            acc = fma(va[2 * s + 9], vb[2 * s + 9], acc);
        }
    }
    return acc;
}

// k(x_s, x_t), unsigned, no bias: K1's out[s][t]
__device__ __forceinline__ double kfn_value(const KernelFn& p, long long s, long long t) {
    const double* xs = p.X + s * p.ldx;
    const double* xt = p.X + t * p.ldx;
    if (p.kernel == SVMB200_KERNEL_LAPLACIAN) {
        double acc = 0.0;
        for (long long k = 0; k < p.d; ++k) acc = __dadd_rn(acc, fabs(__dsub_rn(__ldg(xs + k), __ldg(xt + k))));
        return exp1(__dmul_rn(-p.gamma, acc));
    }
    const double dot = kfn_dot(xs, xt, p.d);
    if (p.kernel == SVMB200_KERNEL_GAUSSIAN) {
        const long long lo = s < t ? s : t, hi = s < t ? t : s;   // K1's self-Gram order: exactly symmetric
        double dist = __dadd_rn(fma(-2.0, dot, __ldg(p.sqn + lo)), __ldg(p.sqn + hi));
        dist = dist < 0.0 ? 0.0 : dist;
        if (s == t) dist = 0.0;
        return exp1(__dmul_rn(-p.gamma, dist));
    }
    if (p.kernel == SVMB200_KERNEL_POLY) {
        const double b = __dadd_rn(__dmul_rn(p.gamma, dot), p.coef0);
        return p.int_degree > 0 ? ipow_rn(b, p.int_degree) : pow_outofline(b, p.degree);
    }
    if (p.kernel == SVMB200_KERNEL_SIGMOID) return tanh_outofline(__dadd_rn(__dmul_rn(p.gamma, dot), p.coef0));
    return dot;
}

// host helpers (gram.cu): |x|^2 per row by K1's row_sqnorm_kernel, and K1's choice between ipow_rn and pow
int svm_row_sqnorms(svmb200_ctx* ctx, const double* dX, int64_t n, int64_t ld, int64_t d, double* out);
int svm_gram_int_degree(double degree);
