// common.cuh -- shared device helpers for the tlsq_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tlsq {

constexpr int kWarp = 32;

// ---------------------------------------------------------------------------------------------------
// FP64 tensor-core MMA (DMMA.8x8x4 in SASS).  Fragment layout (PTX ISA, mma.m8n8k4 .f64):
//   g = lane / 4, t = lane % 4
//   A (8x4, row):  a  = A[g][t]          B (4x8, col):  b = B[t][g]
//   C (8x8):       c0 = C[g][2t], c1 = C[g][2t+1]
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------------
// Element-wise ALM step, bit-faithful to the reference (no FMA contraction; Julia does not contract):
//   x = (d - a) + (1/mu)*y                          src/robustPCA.jl:188
//   e = max(x-eps,0) + min(x+eps,0)                 src/robustPCA.jl:1
//   e = max(e,0) if nonnegE                         src/robustPCA.jl:189-191
//   w = (d - e) + (1/mu)*y                          src/robustPCA.jl:192
// For eps >= 0 exactly one of max(x-eps,0), min(x+eps,0) is non-zero, so e == (|x| > eps ? x - sign(x)*eps : 0)
// bit for bit (up to the sign of zero).  The compare runs on the integer pipe: FP64 ops share the DMMA pipe
// (measured: profiles/r01_microbench_fp64_hbm.log), so every FP64 instruction saved here is tensor throughput.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double soft_th_dev(double x, double eps) {
    const long long xb = __double_as_longlong(x);
    const long long ab = xb & 0x7fffffffffffffffLL;                    // |x|
    const long long sb = xb & (long long)0x8000000000000000ULL;        // sign(x)
    const double seps = __longlong_as_double(__double_as_longlong(eps) | sb);   // copysign(eps, x)
    const double r = __dsub_rn(x, seps);
    return (ab > __double_as_longlong(eps)) ? r : 0.0;
}

__device__ __forceinline__ void alm_ew(double d, double a, double y, double im, double eps, int nonnegE,
                                       double& e, double& w) {
    const double t2 = __dmul_rn(im, y);
    const double x = __dadd_rn(__dsub_rn(d, a), t2);
    double ee = soft_th_dev(x, eps);
    if (nonnegE) ee = (__double_as_longlong(ee) > 0) ? ee : 0.0;       // max(e, 0)
    e = ee;
    w = __dadd_rn(__dsub_rn(d, ee), t2);
}

// warp / block reductions ---------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---------------------------------------------------------------------------------------------------
// Sort key of the robust Grassmann averages (the reference's sortperm over a row, Julia's isless): an order-preserving
// map double -> uint64 with -0.0 == +0.0 and every NaN (a zero column's 0 / 0) above +inf.  Shared by the per-row
// sorts (ga.cu) and the per-row selection (ga_select.cu), so both paths order a row identically.  No key maps above
// ~0 (NaN), so padding slots that hold ~0 with an index >= N sort after every real element.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t sel_order(double u) {
    uint64_t b = (uint64_t)__double_as_longlong(u);
    if ((b << 1) == 0) b = 0;                                              // -0.0 -> +0.0
    if ((b & 0x7fffffffffffffffull) > 0x7ff0000000000000ull) return ~0ull;   // NaN: last (Julia's isless)
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
// the double a sel_order key came from (-0.0 comes back as +0.0, a NaN key as a NaN)
__device__ __forceinline__ double sel_value(uint64_t k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// ---------------------------------------------------------------------------------------------------
// Plane rotation that (nearly) annihilates gamma = x_p . x_q given alpha = |x_p|^2, beta = |x_q|^2.
// The tangent only needs ~20 bits (a slightly inexact angle still converges; later sweeps finish the job), so it is
// built from the single-instruction MUFU reciprocal / rsqrt approximations instead of four IEEE FP64 div/sqrt
// sequences (measured: those dominated the latency of a Jacobi round).  c is Newton-refined to full precision so
// that c^2 + s^2 == 1 to rounding and the accumulated V stays orthogonal.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp_approx(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}
__device__ __forceinline__ double rsqrt_approx(double x) {
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}
// returns false when the pair is already orthogonal to the relative tolerance `tol` (or a column is null)
__device__ __forceinline__ bool jacobi_cs(double alpha, double beta, double gamma, double tol, double& c, double& s) {
    const double lim2 = tol * tol * alpha * beta;
    if (!(gamma * gamma > lim2) || lim2 == 0.0) return false;
    const double zeta = (beta - alpha) * (0.5 * rcp_approx(gamma));
    const double az = fabs(zeta);
    double tt;
    if (az > 1.0e7) {
        tt = 0.5 * rcp_approx(az);                                   // 1/(|z| + sqrt(1+z^2)) -> 1/(2|z|)
    } else {
        const double q = fma(zeta, zeta, 1.0);
        const double root = q * rsqrt_approx(q);                     // ~sqrt(1 + zeta^2)
        tt = rcp_approx(az + root);
    }
    tt = copysign(tt, zeta);
    const double q2 = fma(tt, tt, 1.0);                              // in [1, 2]
    double r = rsqrt_approx(q2);
    r = r * fma(-0.5 * q2 * r, r, 1.5);                              // two Newton steps: r -> 1/sqrt(q2) to FP64
    r = r * fma(-0.5 * q2 * r, r, 1.5);
    c = r;
    s = r * tt;
    return true;
}

// Matrix source: either a dense column-major matrix or an implicit Hankel embedding of a signal
// (H[k,l] = y[k*lag + l], src/robustPCA.jl:76-92, never materialised).
struct MatSrc {
    const double* p;   // dense: matrix base;  hankel: signal y
    int64_t ld;        // dense: leading dimension;  hankel: lag
};
template <bool HANKEL>
__device__ __forceinline__ double src_at(const MatSrc& s, int64_t row, int64_t col) {
    if (HANKEL) return __ldg(s.p + row * s.ld + col);
    return __ldg(s.p + col * s.ld + row);
}

}  // namespace tlsq
