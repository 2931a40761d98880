// eig_fast.cu -- fast path of the per-iteration n x n eigenproblem (n <= 256): the ALM step needs only the svp
// dominant eigenpairs of G = W'W plus the exact COUNT svp = #{sigma_i >= 1/mu} (src/robustPCA.jl:198, full-SVD
// semantics).  Diagonalising the ~n-svp "bulk" directions with a full Jacobi costs ~10 sweeps every iteration
// (measured: the bulk is not warm-startable, it changes completely between ALM iterations), so instead:
//
//  1. Warm-started block subspace iteration on a b = 32 column block:  X = G Q  (DMMA GEMM, atb_kernel), then a
//     one-sided Jacobi of the b columns of X inside ONE CTA (16 warps = 16 column pairs, warp-shuffle dot products,
//     rotations in registers, tournament exchange through shared memory) with Q rotated alongside.  This is a
//     Rayleigh-Ritz step on span(Q); theta_i = q_i'G q_i, residual r_i = ||G q_i - theta_i q_i||; the next basis is
//     the normalised X (one power step).  Stops when all wanted pairs (theta_i >= tau^2, plus the first unwanted
//     one) have r_i <= tol * theta_1.
//  2. Certificate of the count.  Ritz values are lower bounds (theta_i <= lambda_i), so at least svp eigenvalues are
//     >= tau^2.  For "at most": G_w = G - Q_w Theta_w Q_w' differs from G by a PSD rank-svp term, hence
//     lambda_{svp+1}(G) <= lambda_max(G_w) (Weyl), and lambda_max(G_w) <= ||G_w^(2^k)||_F^(1/2^k), evaluated by k
//     Frobenius-normalised squarings (DMMA, the same atb_kernel).  After k = 6 squarings the bound is within
//     n^(1/128) = 4.4 % of lambda_max.  If bound < tau^2 the count is proven; otherwise (or if step 1 does not
//     converge, e.g. when a wanted singular value sits at the edge of the bulk) a device flag routes the iteration
//     through the full Jacobi of eig.cu.  Every kernel looks at the flags itself -- there is no host round trip.
#include "kernels.h"

namespace tlsq {

namespace {

// ---------------------------------------------------------------------------------------------------
// C (na x nb) = (sa*A)' (sb*B),  A: K x na (lda), B: K x nb (ldb), column-major; 32 x 32 output tile per CTA,
// 8 warps = 2 (m) x 4 (n), warp tile 16 x 8 (2 DMMA accumulators); K staged in 64-row chunks, [col][68] padded.
// symmetric != 0: A == B, only tiles with ti <= tj are computed and mirrored; fro2 (optional) accumulates ||C||_F^2.
// run control: the kernel exits unless (flags[0] == want_conv) && (flags[1] == 0)   (flags may be null).
// ---------------------------------------------------------------------------------------------------
constexpr int AT = 32, AK = 64, AKS = AK + 4;

__global__ void __launch_bounds__(256)
atb_kernel(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb, int K, int na, int nb,
           const double* __restrict__ scale2, double* __restrict__ C, int ldc, int symmetric,
           double* __restrict__ fro2, const int* __restrict__ flags, int want_conv,
           const double* __restrict__ cert_f2 = nullptr, int cert_j = 0, double cert_thr = 0.0,
           const double* __restrict__ cert_theta = nullptr) {
    if (flags && !(flags[0] == want_conv && flags[1] == 0)) return;
    if (cert_f2) {
        // squaring j of the count certificate: stop as soon as the bound from the chain so far already proves it
        // (lambda_max <= f_0 u_0, u_j = 1, u_i = sqrt(f_{i+1} u_{i+1}); every CTA evaluates the same finished numbers)
        double u = 1.0;
        for (int j = cert_j - 1; j >= 0; --j) u = sqrt(sqrt(cert_f2[j + 1]) * u);
        const double bound = sqrt(cert_f2[0]) * u;
        const double thr = cert_theta ? cert_theta[0] : cert_thr;
        if (bound < thr * (1.0 - 1e-10)) return;
    }
    const int ti = blockIdx.x, tj = blockIdx.y;
    if (symmetric && ti > tj) return;
    __shared__ double As[AT * AKS];
    __shared__ double Bs[AT * AKS];
    __shared__ double red[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 1, wn = warp >> 1;
    double sc = 1.0;
    if (scale2) {                                   // operands are scaled by 1/sqrt(*scale2) each (Frobenius normalisation)
        const double s2 = *scale2;
        sc = s2 > 0.0 ? 1.0 / s2 : 0.0;             // product of the two operand scales
    }
    double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    const int lr = tid & 63, lc0 = tid >> 6;        // loader: 64 rows x 4 column groups
    for (int k0 = 0; k0 < K; k0 += AK) {
        const bool rok = k0 + lr < K;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int c = lc0 + 4 * q;
            const int ca = ti * AT + c, cb = tj * AT + c;
            As[c * AKS + lr] = (rok && ca < na) ? A[(int64_t)ca * lda + k0 + lr] : 0.0;
            Bs[c * AKS + lr] = (rok && cb < nb) ? B[(int64_t)cb * ldb + k0 + lr] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < AK; kk += 4) {
            const double a0 = As[(16 * wm + g) * AKS + kk + t];
            const double a1 = As[(16 * wm + 8 + g) * AKS + kk + t];
            const double b0 = Bs[(8 * wn + g) * AKS + kk + t];
            dmma884(acc[0][0], acc[0][1], a0, b0);
            dmma884(acc[1][0], acc[1][1], a1, b0);
        }
        __syncthreads();
    }
    double f2 = 0.0;
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = ti * AT + 16 * wm + 8 * mi + g;
            const int j = tj * AT + 8 * wn + 2 * t + e;
            if (i < na && j < nb) {
                const double v = acc[mi][e] * sc;
                C[(int64_t)j * ldc + i] = v;
                if (symmetric && ti != tj) C[(int64_t)i * ldc + j] = v;
                f2 = fma(v, v, f2);
            }
        }
    if (fro2) {
        if (symmetric && ti != tj) f2 *= 2.0;
        f2 = warp_sum(f2);
        if (lane == 0) red[warp] = f2;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) s += red[w];
            atomicAdd(fro2, s);
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// one Rayleigh-Ritz step of the block subspace iteration, single CTA, 16 warps <-> 16 column pairs (b = 32)
// ---------------------------------------------------------------------------------------------------
constexpr int SIB = 32;          // block width

template <int E>
__device__ __forceinline__ bool rotate_pair(double (&xp)[E], double (&xq)[E], double (&vp)[E], double (&vq)[E],
                                            double tol, double wanted2) {
    double alpha = 0.0, beta = 0.0, gamma = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        alpha = fma(xp[e], xp[e], alpha);
        beta = fma(xq[e], xq[e], beta);
        gamma = fma(xp[e], xq[e], gamma);
    }
    alpha = warp_sum(alpha);
    beta = warp_sum(beta);
    gamma = warp_sum(gamma);
    double c, s;
    const double tl = (alpha < wanted2 && beta < wanted2) ? 1.0e-6 : tol;
    if (!jacobi_cs(alpha, beta, gamma, tl, c, s)) return false;        // already orthogonal (or a null column)
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const double a = xp[e], b = xq[e];
        xp[e] = fma(c, a, -s * b);
        xq[e] = fma(s, a, c * b);
        const double va = vp[e], vb = vq[e];
        vp[e] = fma(c, va, -s * vb);
        vq[e] = fma(s, va, c * vb);
    }
    return true;
}

// flags: [0] conv, [1] need_full, [2] svp, [3] SI steps used, [4] certified, [5] jacobi sweeps of the last SI step
template <int E, int BW>
__global__ void __launch_bounds__(16 * BW, 1)
si_jacobi_kernel(const double* __restrict__ X, double* __restrict__ Q, int n, double tau2, int min_wanted,
                 double tol_jac, double tol_res, int last_step, double* __restrict__ theta_out,
                 double* __restrict__ Qout, int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    constexpr int LEN = 32 * E;
    extern __shared__ double sm[];                 // SIB slots x [X part | Q part]
    __shared__ double th[BW], rr[BW], nx[BW], ths[BW];
    __shared__ int order[BW];
    __shared__ int s_svp, s_conv;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;      // warp = seat 0..15
    constexpr int m = BW / 2;
    double xp[E], xq[E], vp[E], vq[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = lane + 32 * e;
        const bool ok = i < n;
        xp[e] = ok ? X[(int64_t)(2 * warp) * n + i] : 0.0;
        xq[e] = ok ? X[(int64_t)(2 * warp + 1) * n + i] : 0.0;
        vp[e] = ok ? Q[(int64_t)(2 * warp) * n + i] : 0.0;
        vq[e] = ok ? Q[(int64_t)(2 * warp + 1) * n + i] : 0.0;
    }
    // pairs of two UNWANTED columns (|x|^2 < tau^4, i.e. Ritz value below tau^2) only need to stay well conditioned
    const double wanted2 = tau2 < 1.0e150 ? 0.25 * tau2 * tau2 : 0.0;      // opnorm mode: tight everywhere
    int sweeps = 0;
    for (; sweeps < 30; ++sweeps) {
        int rotated = 0;
        for (int round = 0; round < 2 * m - 1; ++round) {
            rotated |= rotate_pair<E>(xp, xq, vp, vq, tol_jac, wanted2) ? 1 : 0;
            const int s = warp;
            int ts, tw, bs, bw;
            if (s == 0) { ts = 0; tw = 0; } else if (s == m - 1) { ts = m - 1; tw = 1; } else { ts = s + 1; tw = 0; }
            if (s == 0) { bs = 1; bw = 0; } else { bs = s - 1; bw = 1; }
            double* dt = sm + (size_t)(2 * ts + tw) * 2 * LEN;
            double* db = sm + (size_t)(2 * bs + bw) * 2 * LEN;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                dt[lane + 32 * e] = xp[e];
                dt[LEN + lane + 32 * e] = vp[e];
                db[lane + 32 * e] = xq[e];
                db[LEN + lane + 32 * e] = vq[e];
            }
            __syncthreads();
            const double* pt = sm + (size_t)(2 * s) * 2 * LEN;
            const double* pb = sm + (size_t)(2 * s + 1) * 2 * LEN;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                xp[e] = pt[lane + 32 * e];
                vp[e] = pt[LEN + lane + 32 * e];
                xq[e] = pb[lane + 32 * e];
                vq[e] = pb[LEN + lane + 32 * e];
            }
            __syncthreads();
        }
        if (!__syncthreads_or(rotated)) { ++sweeps; break; }
    }
    // Ritz values / residuals of the two columns of this warp (columns stay in their slots: index 2*warp + which)
#pragma unroll
    for (int which = 0; which < 2; ++which) {
        double dot = 0.0, xx = 0.0;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const double x = which ? xq[e] : xp[e];
            const double v = which ? vq[e] : vp[e];
            dot = fma(v, x, dot);
            xx = fma(x, x, xx);
        }
        dot = warp_sum(dot);
        xx = warp_sum(xx);
        double r2 = 0.0;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const double x = which ? xq[e] : xp[e];
            const double v = which ? vq[e] : vp[e];
            const double df = x - dot * v;
            r2 = fma(df, df, r2);
        }
        r2 = warp_sum(r2);
        if (lane == 0) {
            th[2 * warp + which] = dot;
            rr[2 * warp + which] = sqrt(r2);
            nx[2 * warp + which] = sqrt(xx);
        }
    }
    __syncthreads();
    if (tid < BW) {
        const double lj = th[tid];
        int rank = 0;
        for (int k = 0; k < BW; ++k) rank += (th[k] > lj) || (th[k] == lj && k < tid);
        order[rank] = tid;
        ths[rank] = lj;
    }
    __syncthreads();
    if (tid == 0) {
        int svp = 0;
        for (int i = 0; i < BW; ++i) svp += (ths[i] >= tau2) ? 1 : 0;
        // only the WANTED pairs must be converged: Ritz values are lower bounds, so the count is >= svp whatever the
        // state of the unwanted ones (they track the flat bulk and converge arbitrarily slowly); "<= svp" is proven
        // by the squaring certificate.
        if (svp < min_wanted) svp = min_wanted;       // top-k mode (opnorm: the dominant pair regardless of tau)
        int conv = (svp <= BW - 2) ? 1 : 0;
        const int need = svp;
        const double lim = tol_res * fabs(ths[0]);
        for (int i = 0; i < need; ++i) conv &= (rr[order[i]] <= lim) ? 1 : 0;
        s_svp = svp;
        s_conv = conv;
        flags[3] += 1;
        flags[5] = sweeps;
        if (conv) { flags[0] = 1; flags[2] = svp; }
        else if (svp > BW - 2 || last_step) flags[1] = 1;
    }
    __syncthreads();
    const int conv = s_conv;
    // outputs: sorted Ritz vectors (used when converged) / normalised power step (next basis)
#pragma unroll
    for (int which = 0; which < 2; ++which) {
        const int col = 2 * warp + which;
        int rank = 0;
        for (int k = 0; k < BW; ++k) rank = (order[k] == col) ? k : rank;
        const double nrm = nx[col];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = lane + 32 * e;
            if (i < n) {
                const double x = which ? xq[e] : xp[e];
                const double v = which ? vq[e] : vp[e];
                if (conv) Qout[(int64_t)rank * n + i] = v;
                else Q[(int64_t)col * n + i] = nrm > 0.0 ? x / nrm : v;
            }
        }
        if (conv && lane == 0) theta_out[rank] = th[col];
    }
}

// Gd = G - sum_{c < svp} theta_c q_c q_c'  (+ ||Gd||_F^2), runs only when the subspace iteration converged
__global__ void __launch_bounds__(256)
deflate_kernel(const double* __restrict__ G, int n, const double* __restrict__ Qs, const double* __restrict__ theta,
               const int* __restrict__ flags, double* __restrict__ Gd, double* __restrict__ fro2) {
    if (!(flags[0] == 1 && flags[1] == 0)) return;
    const int svp = flags[2];
    double f2 = 0.0;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < (int64_t)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        double v = G[idx];
        for (int c = 0; c < svp; ++c) v = fma(-theta[c] * Qs[(int64_t)c * n + i], Qs[(int64_t)c * n + j], v);
        Gd[idx] = v;
        f2 = v * v;
    }
    f2 = warp_sum(f2);
    if ((threadIdx.x & 31) == 0 && f2 != 0.0) atomicAdd(fro2, f2);
}

// certificate + outputs of the fast path (single CTA)
__global__ void __launch_bounds__(256)
fast_finish_kernel(int n, int nsq, const double* __restrict__ f2, double tau2, int top1, double tau, int nukeA,
                   const double* __restrict__ theta, const double* __restrict__ Qs, double* __restrict__ Qb,
                   double* __restrict__ Vs, double* __restrict__ lam, double* __restrict__ sigma,
                   double* __restrict__ fvec, int* __restrict__ svp_out, int* __restrict__ flags, int bw) {
    __shared__ int ok;
    if (threadIdx.x == 0) {
        int good = (flags[0] == 1 && flags[1] == 0) ? 1 : 0;
        if (good) {
            // lambda_max(Gd) <= f_0 * u_0,  u_k = 1, u_j = sqrt(f_{j+1} u_{j+1})
            // (the squaring chain stops early once it has proven the count: use the part that was computed)
            int ne = 0;
            while (ne < nsq && f2[ne + 1] > 0.0) ++ne;
            double u = 1.0;
            for (int j = ne - 1; j >= 0; --j) u = sqrt(sqrt(f2[j + 1]) * u);
            const double bound = sqrt(f2[0]) * u;
            // ALM step: nothing left above tau^2.  opnorm mode: nothing left above theta_1, i.e. theta_1 IS lambda_max.
            const double thr = top1 ? theta[0] : tau2;
            good = (bound < thr * (1.0 - 1e-10)) ? 1 : 0;
            if (!(bound == bound)) good = 0;
        }
        if (!good) flags[1] = 1;
        flags[4] = good;
        ok = good;
    }
    __syncthreads();
    if (!ok) return;
    const int svp = flags[2];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double l = i < bw ? theta[i] : 0.0;
        const double sg = l > 0.0 ? sqrt(l) : 0.0;
        lam[i] = l;
        sigma[i] = sg;
        const bool keep = i < svp;
        fvec[i] = keep ? (nukeA ? (sg - tau) / sg : 1.0) : 0.0;
    }
    for (int idx = threadIdx.x; idx < n * bw; idx += blockDim.x) {
        const double v = Qs[idx];
        Vs[idx] = v;
        Qb[idx] = v;
    }
    if (threadIdx.x == 0) *svp_out = svp;
}

// Qb = Vs[:, 0:32]  after a full Jacobi (only when the fallback ran)
__global__ void copy_block_kernel(const double* __restrict__ Vs, int n, double* __restrict__ Qb,
                                  const int* __restrict__ flags) {
    if (flags && flags[1] == 0) return;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n * SIB; idx += gridDim.x * blockDim.x)
        Qb[idx] = Vs[idx];
}

// ||G||_F^2 of an n x n matrix
__global__ void __launch_bounds__(256)
fro2_kernel(const double* __restrict__ G, int64_t nn, double* __restrict__ out) {
    double f2 = 0.0;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < nn; idx += (int64_t)gridDim.x * blockDim.x)
        f2 = fma(G[idx], G[idx], f2);
    f2 = warp_sum(f2);
    if ((threadIdx.x & 31) == 0 && f2 != 0.0) atomicAdd(out, f2);
}

// bounds[0] <= lambda_max(G) <= bounds[1] from the Frobenius norms of the squaring chain:
//   upper: u_k = 1,          u_j = sqrt(f_{j+1} u_{j+1});   lower: l_k = 1/sqrt(n), l_j = sqrt(f_{j+1} l_{j+1})
__global__ void lmax_bounds_kernel(const double* __restrict__ f2, int nsq, int n, double* __restrict__ bounds) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double u = 1.0, l = 1.0 / sqrt((double)n);
    for (int j = nsq - 1; j >= 0; --j) {
        const double f = sqrt(f2[j + 1]);
        u = sqrt(f * u);
        l = sqrt(f * l);
    }
    const double f0 = sqrt(f2[0]);
    bounds[0] = f0 * l;
    bounds[1] = f0 * u;
}

__global__ void init_block_kernel(double* __restrict__ Qb, int n) {      // Qb = [e_1 ... e_32]
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n * SIB; idx += gridDim.x * blockDim.x)
        Qb[idx] = (idx % n == idx / n) ? 1.0 : 0.0;
}

template <int E, int BW>
cudaError_t launch_si(const double* X, double* Q, int n, double tau2, int min_wanted, double tol_jac, double tol_res,
                      int last, double* theta, double* Qout, int* flags, cudaStream_t st) {
    const size_t smem = (size_t)BW * 2 * 32 * E * sizeof(double);
    auto kern = si_jacobi_kernel<E, BW>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<1, 16 * BW, smem, st>>>(X, Q, n, tau2, min_wanted, tol_jac, tol_res, last, theta, Qout, flags);
    return cudaGetLastError();
}


// =====================================================================================================================
// Large embeddings (512 < n <= 4096): the same algorithm with the block kept in global memory (L2 resident) and the
// Rayleigh-Ritz step done on the 32 x 32 projected matrix.  One step, given an orthonormal n x 32 basis Q:
//   X = G Q (DMMA)            H = Q'X (32 x 32)            H = R Theta R'  (one-sided Jacobi, one CTA, registers)
//   Q~ = Q R, X~ = X R        r_i = |x~_i - theta_i q~_i|  (Ritz pairs and residuals)
//   converged (all wanted pairs)  ->  Qout = Q~, theta;    else Q <- orth(X~) by CholeskyQR2 on the normalised columns
// followed by the same deflation + squaring certificate of the count as the small path.  All kernels look at the device
// flags themselves, so the host enqueues a fixed number of steps without a round trip.
// =====================================================================================================================
constexpr int LB = 32;

__global__ void __launch_bounds__(16 * LB, 1)
rr_small_eig_kernel(const double* __restrict__ H, double* __restrict__ theta, double* __restrict__ R,
                    const int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ double sm[LB * 2 * LB];              // slot c: [X part (32) | V part (32)]
    __shared__ double th[LB];
    __shared__ int order[LB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int m = LB / 2;
    double xp[1], xq[1], vp[1], vq[1];
    {
        const int cp = 2 * warp, cq = 2 * warp + 1;
        xp[0] = 0.5 * (H[cp * LB + lane] + H[lane * LB + cp]);      // symmetrised
        xq[0] = 0.5 * (H[cq * LB + lane] + H[lane * LB + cq]);
        vp[0] = lane == cp ? 1.0 : 0.0;
        vq[0] = lane == cq ? 1.0 : 0.0;
    }
    const double tol = 1.0e-15 * 6.0;
    for (int sweeps = 0; sweeps < 30; ++sweeps) {
        int rotated = 0;
        for (int round = 0; round < 2 * m - 1; ++round) {
            rotated |= rotate_pair<1>(xp, xq, vp, vq, tol, 0.0) ? 1 : 0;
            const int s = warp;
            int ts, tw, bs, bw;
            if (s == 0) { ts = 0; tw = 0; } else if (s == m - 1) { ts = m - 1; tw = 1; } else { ts = s + 1; tw = 0; }
            if (s == 0) { bs = 1; bw = 0; } else { bs = s - 1; bw = 1; }
            double* dt = sm + (size_t)(2 * ts + tw) * 2 * LB;
            double* db = sm + (size_t)(2 * bs + bw) * 2 * LB;
            dt[lane] = xp[0]; dt[LB + lane] = vp[0];
            db[lane] = xq[0]; db[LB + lane] = vq[0];
            __syncthreads();
            const double* pt = sm + (size_t)(2 * s) * 2 * LB;
            const double* pb = sm + (size_t)(2 * s + 1) * 2 * LB;
            xp[0] = pt[lane]; vp[0] = pt[LB + lane];
            xq[0] = pb[lane]; vq[0] = pb[LB + lane];
            __syncthreads();
        }
        if (!__syncthreads_or(rotated)) break;
    }
    // eigenvalue of column c: v_c . x_c  (X = H V, V orthogonal)
    {
        const double dp = warp_sum(vp[0] * xp[0]);
        const double dq = warp_sum(vq[0] * xq[0]);
        if (lane == 0) { th[2 * warp] = dp; th[2 * warp + 1] = dq; }
    }
    __syncthreads();
    if (tid < LB) {
        const double lj = th[tid];
        int rank = 0;
        for (int k = 0; k < LB; ++k) rank += (th[k] > lj) || (th[k] == lj && k < tid);
        order[tid] = rank;
        theta[rank] = lj;
    }
    __syncthreads();
    R[order[2 * warp] * LB + lane] = vp[0];
    R[order[2 * warp + 1] * LB + lane] = vq[0];
}

// Qr = Q R, Xr = X R   (n x 32 times 32 x 32; thread <-> row)
__global__ void __launch_bounds__(128)
rr_rotate_kernel(const double* __restrict__ Q, const double* __restrict__ X, const double* __restrict__ R, int n,
                 double* __restrict__ Qr, double* __restrict__ Xr, const int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ double Rs[LB * LB];
    for (int i = threadIdx.x; i < LB * LB; i += blockDim.x) Rs[i] = R[i];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double q[LB], x[LB];
#pragma unroll
    for (int c = 0; c < LB; ++c) { q[c] = Q[(int64_t)c * n + i]; x[c] = X[(int64_t)c * n + i]; }
#pragma unroll 4
    for (int j = 0; j < LB; ++j) {
        double aq = 0.0, ax = 0.0;
#pragma unroll
        for (int c = 0; c < LB; ++c) { aq = fma(q[c], Rs[j * LB + c], aq); ax = fma(x[c], Rs[j * LB + c], ax); }
        Qr[(int64_t)j * n + i] = aq;
        Xr[(int64_t)j * n + i] = ax;
    }
}

// res[j] = |Xr_j - theta_j Qr_j|, nx[j] = |Xr_j|     (one CTA per column)
__global__ void __launch_bounds__(256)
rr_resid_kernel(const double* __restrict__ Qr, const double* __restrict__ Xr, const double* __restrict__ theta, int n,
                double* __restrict__ res, double* __restrict__ nx, const int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ double r1[8], r2[8];
    const int j = blockIdx.x;
    const double th = theta[j];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double x = Xr[(int64_t)j * n + i];
        const double d = x - th * Qr[(int64_t)j * n + i];
        a = fma(d, d, a);
        b = fma(x, x, b);
    }
    a = warp_sum(a); b = warp_sum(b);
    if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = a; r2[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sa = 0.0, sb = 0.0;
        for (int w = 0; w < 8; ++w) { sa += r1[w]; sb += r2[w]; }
        res[j] = sqrt(sa);
        nx[j] = sqrt(sb);
    }
}

// convergence decision of one step (same rules as si_jacobi_kernel) + outputs: converged -> Qout = Qr, theta_out;
// otherwise the next (not yet orthonormal) basis Q = Xr with normalised columns.  Single CTA.
__global__ void __launch_bounds__(1024)
rr_decide_kernel(const double* __restrict__ Qr, const double* __restrict__ Xr, const double* __restrict__ theta,
                 const double* __restrict__ res, const double* __restrict__ nx, int n, double tau2, int min_wanted,
                 double tol_res, int last_step, double* __restrict__ Q, double* __restrict__ Qout,
                 double* __restrict__ theta_out, int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ int s_conv;
    if (threadIdx.x == 0) {
        int svp = 0;
        for (int i = 0; i < LB; ++i) svp += (theta[i] >= tau2) ? 1 : 0;
        if (svp < min_wanted) svp = min_wanted;
        int conv = (svp <= LB - 2) ? 1 : 0;
        const double lim = tol_res * fabs(theta[0]);
        for (int i = 0; i < svp && i < LB; ++i) conv &= (res[i] <= lim) ? 1 : 0;
        s_conv = conv;
        flags[3] += 1;
        if (conv) { flags[0] = 1; flags[2] = svp; }
        else if (svp > LB - 2 || last_step) flags[1] = 1;
    }
    __syncthreads();
    const int conv = s_conv;
    if (conv) {
        for (int idx = threadIdx.x; idx < n * LB; idx += blockDim.x) Qout[idx] = Qr[idx];
        if (threadIdx.x < LB) theta_out[threadIdx.x] = theta[threadIdx.x];
    } else {
        for (int idx = threadIdx.x; idx < n * LB; idx += blockDim.x) {
            const double nrm = nx[idx / n];
            Q[idx] = nrm > 0.0 ? Xr[idx] / nrm : Qr[idx];
        }
    }
}

// Q <- Q Rc^-1 for an upper-triangular 32 x 32 Rc (row-wise forward substitution y Rc = x; a zero pivot zeroes the column)
__global__ void __launch_bounds__(128)
rr_trsm_kernel(double* __restrict__ Q, const double* __restrict__ Rc, int n, const int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ double Rs[LB * LB];
    for (int i = threadIdx.x; i < LB * LB; i += blockDim.x) Rs[i] = Rc[i];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double y[LB];
#pragma unroll
    for (int j = 0; j < LB; ++j) {
        double v = Q[(int64_t)j * n + i];
#pragma unroll
        for (int c = 0; c < LB; ++c)
            if (c < j) v = fma(-y[c], Rs[j * LB + c], v);
        const double d = Rs[j * LB + j];
        y[j] = d > 0.0 ? v / d : 0.0;
    }
#pragma unroll
    for (int j = 0; j < LB; ++j) Q[(int64_t)j * n + i] = y[j];
}

// in-place upper Cholesky of the 32 x 32 Gram of the basis (single warp per column sweep; zero-pivot deflation)
__global__ void __launch_bounds__(LB)
rr_chol32_kernel(double* __restrict__ S, const int* __restrict__ flags) {
    if (flags[0] == 1 || flags[1] == 1) return;
    __shared__ double A[LB][LB + 1];               // A[i][k] = element (i, k), i <= k used
    const int t = threadIdx.x;
    for (int i = 0; i < LB; ++i) A[i][t] = S[t * LB + i];
    __syncwarp();
    const double d0 = A[t][t];
    for (int j = 0; j < LB; ++j) {
        const double ajj = A[j][j];
        const double dj = __shfl_sync(0xffffffffu, d0, j);
        const bool ok = ajj > 32.0 * 2.220446049250313e-16 * dj && dj > 0.0;
        const double piv = ok ? sqrt(ajj) : 0.0;
        const double ip = ok ? 1.0 / piv : 0.0;
        __syncwarp();
        double rjk = 0.0;
        if (t >= j) { rjk = (t == j) ? piv : A[j][t] * ip; A[j][t] = rjk; }
        __syncwarp();
        if (ok && t > j)
            for (int i = j + 1; i <= t; ++i) A[i][t] = fma(-A[j][i], rjk, A[i][t]);
        __syncwarp();
    }
    for (int i = 0; i < LB; ++i) S[t * LB + i] = (i <= t) ? A[i][t] : 0.0;
}

cudaError_t launch_eig_large(const double* G, int n, double tau, int nukeA, EigFastWork w, double* lam, double* Vs,
                             double* sigma, double* fvec, int* svp, cudaStream_t st, int64_t* launches, int top1,
                             int max_steps) {
    const int NSI = max_steps < 2 ? 2 : (max_steps > 16 ? 16 : max_steps);
    constexpr int NSQ = 6;
    cudaError_t e;
    const double tau2 = top1 ? 1.0e300 : tau * tau;
    const int min_wanted = top1 ? 1 : 0;
    const double tol_res = 4.0e-14;
    if ((e = cudaMemsetAsync(w.f2, 0, (16 + 8) * sizeof(double), st)) != cudaSuccess) return e;   // f2 + flags
    if ((e = cudaMemcpyAsync(w.Qwork, w.Qb, (size_t)n * LB * 8, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
    const dim3 gx((n + AT - 1) / AT, 1);
    const int rowblocks = (n + 127) / 128;
    int nl = 0;
    for (int it = 0; it < NSI; ++it) {
        atb_kernel<<<gx, 256, 0, st>>>(G, n, w.Qwork, n, n, n, LB, nullptr, w.X, n, 0, nullptr, w.flags, 0);        // X = G Q
        atb_kernel<<<dim3(1, 1), 256, 0, st>>>(w.Qwork, n, w.X, n, n, LB, LB, nullptr, w.Hs, LB, 0, nullptr, w.flags, 0);  // H = Q'X
        rr_small_eig_kernel<<<1, 16 * LB, 0, st>>>(w.Hs, w.theta, w.Rs, w.flags);
        rr_rotate_kernel<<<rowblocks, 128, 0, st>>>(w.Qwork, w.X, w.Rs, n, w.Qr, w.Xr, w.flags);
        rr_resid_kernel<<<LB, 256, 0, st>>>(w.Qr, w.Xr, w.theta, n, w.res, w.nx, w.flags);
        rr_decide_kernel<<<1, 1024, 0, st>>>(w.Qr, w.Xr, w.theta, w.res, w.nx, n, tau2, min_wanted, tol_res,
                                            it == NSI - 1 ? 1 : 0, w.Qwork, w.Qout, w.theta, w.flags);
        for (int rep = 0; rep < 2; ++rep) {                                                    // CholeskyQR2
            atb_kernel<<<dim3(1, 1), 256, 0, st>>>(w.Qwork, n, w.Qwork, n, n, LB, LB, nullptr, w.Ss, LB, 0, nullptr, w.flags, 0);
            rr_chol32_kernel<<<1, LB, 0, st>>>(w.Ss, w.flags);
            rr_trsm_kernel<<<rowblocks, 128, 0, st>>>(w.Qwork, w.Ss, n, w.flags);
        }
        nl += 12;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    deflate_kernel<<<(unsigned)(((int64_t)n * n + 255) / 256), 256, 0, st>>>(G, n, w.Qout, w.theta, w.flags, w.Ca, w.f2);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const dim3 gs((n + AT - 1) / AT, (n + AT - 1) / AT);
    double* cin = w.Ca;
    double* cout = w.Cb;
    for (int j = 0; j < NSQ; ++j) {
        atb_kernel<<<gs, 256, 0, st>>>(cin, n, cin, n, n, n, n, w.f2 + j, cout, n, 1, w.f2 + j + 1, w.flags, 1,
                                       w.f2, j, tau2, top1 ? w.theta : nullptr);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        double* tmp = cin; cin = cout; cout = tmp;
    }
    fast_finish_kernel<<<1, 256, 0, st>>>(n, NSQ, w.f2, tau2, top1, tau, nukeA, w.theta, w.Qout, w.Qb, Vs, lam, sigma, fvec,
                                          svp, w.flags, LB);
    if (launches) *launches += nl + 1 + NSQ + 1;
    return cudaGetLastError();
}

}  // namespace

size_t eig_fast_work_doubles(int n) {
    // Qb, Qwork, Qout, X (n x 32 each) + theta (32) + Ca, Cb (n x n) + f2 (16) + flags (8 ints -> 8 doubles)
    // large n: + Qr, Xr (n x 32), Hs, Rs, Ss (32 x 32), res, nx (32)
    return (size_t)6 * n * SIB + SIB + (size_t)2 * n * n + 16 + 8 + 16 + 3 * SIB * SIB + 2 * SIB;
}

bool eig_fast_supported(int n) { return n > 64 && n <= kEigMaxN; }
// small path: shared memory (block x 2 x n doubles) must fit; large path: always the 32-column block
int eig_fast_max_block(int n) { return (n <= 256 || n > kEigSmallN) ? 32 : 16; }

EigFastWork eig_fast_carve(double* base, int n) {
    EigFastWork w;
    w.Qb = base; base += (size_t)n * SIB;
    w.Qwork = base; base += (size_t)n * SIB;
    w.Qout = base; base += (size_t)n * SIB;
    w.X = base; base += (size_t)n * SIB;
    w.theta = base; base += SIB;
    w.Ca = base; base += (size_t)n * n;
    w.Cb = base; base += (size_t)n * n;
    w.f2 = base; base += 16;
    w.flags = reinterpret_cast<int*>(base); base += 8;
    w.Qr = base; base += (size_t)n * SIB;
    w.Xr = base; base += (size_t)n * SIB;
    w.Hs = base; base += SIB * SIB;
    w.Rs = base; base += SIB * SIB;
    w.Ss = base; base += SIB * SIB;
    w.res = base; base += SIB;
    w.nx = base; base += SIB;
    return w;
}

cudaError_t launch_lmax_bounds(const double* G, int n, double* Ca, double* Cb, double* f2, double* bounds,
                               cudaStream_t st, int64_t* launches) {
    constexpr int NSQ = 10;      // bracket ratio n^(1/2^(NSQ+1)): 0.27 % at n = 256
    cudaError_t e;
    if ((e = cudaMemsetAsync(f2, 0, 16 * sizeof(double), st)) != cudaSuccess) return e;
    fro2_kernel<<<32, 256, 0, st>>>(G, (int64_t)n * n, f2);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const dim3 gs((n + AT - 1) / AT, (n + AT - 1) / AT);
    const double* cin = G;
    double* cout = Ca;
    for (int j = 0; j < NSQ; ++j) {
        atb_kernel<<<gs, 256, 0, st>>>(cin, n, cin, n, n, n, n, f2 + j, cout, n, 1, f2 + j + 1, nullptr, 0);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        cin = cout;
        cout = (cout == Ca) ? Cb : Ca;
    }
    lmax_bounds_kernel<<<1, 32, 0, st>>>(f2, NSQ, n, bounds);
    if (launches) *launches += NSQ + 2;
    return cudaGetLastError();
}

cudaError_t launch_copy_block(const double* Vs, int n, double* Qb, const int* flags, cudaStream_t st,
                              int64_t* launches) {
    copy_block_kernel<<<8, 256, 0, st>>>(Vs, n, Qb, flags);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_init_block(double* Qb, int n, cudaStream_t st, int64_t* launches) {
    init_block_kernel<<<8, 256, 0, st>>>(Qb, n);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_eig_fast(const double* G, int n, double tau, int nukeA, EigFastWork w, double* lam, double* Vs,
                            double* sigma, double* fvec, int* svp, cudaStream_t st, int64_t* launches, int top1,
                            int bw, int max_steps) {
    if (n > kEigSmallN)
        return launch_eig_large(G, n, tau, nukeA, w, lam, Vs, sigma, fvec, svp, st, launches, top1, max_steps);
    if (bw != 16) bw = SIB;
    if (n > 256) bw = 16;
    // subspace-iteration steps attempted before falling back (launches after convergence exit at once, but each still
    // costs a launch slot: the caller passes last iteration's step count + a margin)
    const int NSI = max_steps < 2 ? 2 : (max_steps > 16 ? 16 : max_steps);
    constexpr int NSQ = 6;       // squarings of the certificate: bound within n^(1/128) of lambda_max
    cudaError_t e;
    const double tau2 = top1 ? 1.0e300 : tau * tau;
    const int min_wanted = top1 ? 1 : 0;
    const double tol_jac = 1.0e-15 * sqrt((double)n);
    const double tol_res = 4.0e-14;
    if ((e = cudaMemsetAsync(w.f2, 0, (16 + 8) * sizeof(double), st)) != cudaSuccess) return e;   // f2 + flags
    if ((e = cudaMemcpyAsync(w.Qwork, w.Qb, (size_t)n * bw * 8, cudaMemcpyDeviceToDevice, st)) != cudaSuccess)
        return e;
    const dim3 gx((n + AT - 1) / AT, 1);
    for (int it = 0; it < NSI; ++it) {
        // X = G' Q = G Q   (skipped once converged / failed)
        atb_kernel<<<gx, 256, 0, st>>>(G, n, w.Qwork, n, n, n, bw, nullptr, w.X, n, 0, nullptr, w.flags, 0);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        const int last = (it == NSI - 1) ? 1 : 0;
        if (bw == 16) {
            if (n <= 128) e = launch_si<4, 16>(w.X, w.Qwork, n, tau2, min_wanted, tol_jac, tol_res, last, w.theta, w.Qout, w.flags, st);
            else if (n <= 256) e = launch_si<8, 16>(w.X, w.Qwork, n, tau2, min_wanted, tol_jac, tol_res, last, w.theta, w.Qout, w.flags, st);
            else e = launch_si<16, 16>(w.X, w.Qwork, n, tau2, min_wanted, tol_jac, tol_res, last, w.theta, w.Qout, w.flags, st);
        } else {
            if (n <= 128) e = launch_si<4, 32>(w.X, w.Qwork, n, tau2, min_wanted, tol_jac, tol_res, last, w.theta, w.Qout, w.flags, st);
            else e = launch_si<8, 32>(w.X, w.Qwork, n, tau2, min_wanted, tol_jac, tol_res, last, w.theta, w.Qout, w.flags, st);
        }
        if (e != cudaSuccess) return e;
    }
    deflate_kernel<<<(unsigned)(((int64_t)n * n + 255) / 256), 256, 0, st>>>(G, n, w.Qout, w.theta, w.flags, w.Ca,
                                                                            w.f2);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const dim3 gs((n + AT - 1) / AT, (n + AT - 1) / AT);
    double* cin = w.Ca;
    double* cout = w.Cb;
    for (int j = 0; j < NSQ; ++j) {
        // C_{j+1} = (C_j / f_j)' (C_j / f_j),  f2[j+1] = ||C_{j+1}||_F^2
        atb_kernel<<<gs, 256, 0, st>>>(cin, n, cin, n, n, n, n, w.f2 + j, cout, n, 1, w.f2 + j + 1, w.flags, 1,
                                       w.f2, j, tau2, top1 ? w.theta : nullptr);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        double* tmp = cin; cin = cout; cout = tmp;
    }
    fast_finish_kernel<<<1, 256, 0, st>>>(n, NSQ, w.f2, tau2, top1, tau, nukeA, w.theta, w.Qout, w.Qb, Vs, lam, sigma, fvec,
                                          svp, w.flags, bw);
    if (launches) *launches += 2 * NSI + 1 + NSQ + 1;
    return cudaGetLastError();
}

}  // namespace tlsq
