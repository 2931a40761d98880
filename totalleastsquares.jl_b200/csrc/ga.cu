// ga.cu -- Grassmann averages (rpca_ga, src/robustPCA.jl:255-316) as ONE streaming sweep of X per iteration.
//
// Reference iteration (:291-295): w_n = sign(u_n'q) ||x_n||  (sweep 1 of U),  mu = sum_n w_n u_n / sum_n w_n
// (sweep 2 of U, mu! :308-316),  q = mu/||mu||.  Because w_n u_n = sign(u_n'q) x_n the normalised copy U is never
// needed, and because the tile's rows of mu are complete as soon as the tile has been summed over n, the dot
// products x_n'mu that decide the NEXT iteration's signs (sign(u_n'q_new) = sign(x_n'mu)) are accumulated in the
// same sweep while the tile is still in shared memory.  One HBM read of X per iteration (the reference does two).
//
// ga_sweep_kernel<MODE>: persistent CTAs, row tiles of 32 rows x 256 columns staged in shared memory [col][32].
//   phase A (fused with the load): thread (row, column group) accumulates sum_n s_n X[row,n]
//   phase B: thread n accumulates sum_i X[i,n] mu_i over the tile with a skewed (conflict-free) row order.
#include <cuda.h>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int GA_R = 32;      // rows per tile
constexpr int GA_NC = 256;    // columns per chunk
constexpr int GA_DEFL = 3;    // TMA kernel only: deflation + column norms^2 + first dot products of the next component
constexpr int GA_PSTRIDE = 2 * GA_NC + 2;   // per-CTA partials: [256 sums | mm | 256 second sums | pad]

template <int MODE>
__global__ void __launch_bounds__(256, 3)
ga_sweep_kernel(const double* __restrict__ X, int64_t d, int64_t N, int64_t ld, double* __restrict__ vec,
                const double* __restrict__ s, const double* __restrict__ sumw, double* __restrict__ t,
                int ntiles) {
    extern __shared__ double sm[];
    double* Xs = sm;                       // GA_NC * GA_R
    double* sv = Xs + GA_NC * GA_R;        // GA_NC   signs of the current chunk
    double* red = sv + GA_NC;              // 8 * 32  partial row sums
    double* mus = red + 8 * GA_R;          // 32      mu (or q) rows of the tile
    __shared__ double mmred[8];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunks = (int)((N + GA_NC - 1) / GA_NC);
    const double inv_sumw_den = (MODE == GA_PASS) ? *sumw : 1.0;
    double tacc = 0.0;                     // column accumulator (single-chunk fast path)
    double mm = 0.0;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row = (int64_t)tile * GA_R + lane;
        const bool rok = row < d;

        if (MODE == GA_PASS) {
            // ---- phase A over all chunks: v_row = sum_n s_n X[row, n] -------------------------------------------
            double vpart = 0.0;
            for (int ch = 0; ch < nchunks; ++ch) {
                const int64_t cbase = (int64_t)ch * GA_NC;
                __syncthreads();
                if (cbase + tid < N) sv[tid] = s[cbase + tid]; else sv[tid] = 0.0;
                __syncthreads();
#pragma unroll 8
                for (int k = 0; k < 32; ++k) {
                    const int c = warp + 8 * k;
                    double x = 0.0;
                    if (rok && cbase + c < N) x = __ldg(X + (cbase + c) * ld + row);
                    if (nchunks == 1) Xs[c * GA_R + lane] = x;
                    vpart = fma(sv[c], x, vpart);
                }
            }
            red[warp * GA_R + lane] = vpart;
            __syncthreads();
            if (warp == 0) {
                double v = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) v += red[w * GA_R + lane];
                const double m = v / inv_sumw_den;                  // s ./= ws   (:315)
                mus[lane] = rok ? m : 0.0;
                if (rok) { vec[row] = m; mm = fma(m, m, mm); }
            }
            __syncthreads();
        } else if (MODE == GA_DOTS) {
            __syncthreads();
            if (warp == 0) mus[lane] = rok ? vec[row] : 0.0;
            __syncthreads();
        }

        // ---- phase B: t[n] += sum_i X[i,n] * (mu_i | q_i | X[i,n]) -------------------------------------------------
        for (int ch = 0; ch < nchunks; ++ch) {
            const int64_t cbase = (int64_t)ch * GA_NC;
            if (!(MODE == GA_PASS && nchunks == 1)) {
                __syncthreads();
#pragma unroll 8
                for (int k = 0; k < 32; ++k) {
                    const int c = warp + 8 * k;
                    double x = 0.0;
                    if (rok && cbase + c < N) x = __ldg(X + (cbase + c) * ld + row);
                    Xs[c * GA_R + lane] = x;
                }
                __syncthreads();
            }
            double acc = 0.0;
            const int n = tid;
#pragma unroll 8
            for (int i = 0; i < GA_R; ++i) {
                const int ii = (i + n) & (GA_R - 1);
                const double x = Xs[n * GA_R + ii];
                if (MODE == GA_NORMS) acc = fma(x, x, acc);
                else acc = fma(x, mus[ii], acc);
            }
            if (nchunks == 1) tacc += acc;
            else if (cbase + n < N) atomicAdd(t + cbase + n, acc);
        }
        __syncthreads();
    }

    if (nchunks == 1 && tid < N) atomicAdd(t + tid, tacc);
    if (MODE == GA_PASS) {
        // only warp 0 holds mm
        if (warp == 0) {
            mm = warp_sum(mm);
            if (lane == 0) atomicAdd(t + N, mm);
        }
    }
    (void)mmred;
}


// ---------------------------------------------------------------------------------------------------------------------
// TMA-staged form of the same sweep for N <= 256 (one column chunk): the 32-row x 256-column tiles (64 KB) arrive through
// a 3-stage mbarrier ring filled by cp.async.bulk.tensor (box {32 rows, 256 columns} lands in exactly the [col][32]
// layout the two phases use), so 128 KB per SM are always in flight and the load no longer alternates with the
// compute phases.  Column sums leave as per-CTA partials (summed in fixed order by ga_reduce_kernel: deterministic).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ga_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int MODE>
__global__ void __launch_bounds__(256, 1)
ga_sweep_tma_kernel(const __grid_constant__ CUtensorMap mX, int64_t d, int N, double* __restrict__ vec,
                    const double* __restrict__ s, const double* __restrict__ sumw, double* __restrict__ part,
                    int ntiles, int nstage, double* __restrict__ Xg, int64_t ld, const double* __restrict__ q2) {
    extern __shared__ __align__(1024) uint8_t smraw[];
    __shared__ uint64_t full[4];
    __shared__ double sv[GA_NC];
    __shared__ double red[8 * GA_R];
    __shared__ double mus[GA_R];
    constexpr int STG = GA_NC * GA_R;                          // doubles per stage (64 KB)
    double* stage = reinterpret_cast<double*>(smraw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int i = 0; i < 4; ++i)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ga_smem_u32(&full[i])), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    sv[tid] = ((MODE == GA_PASS || MODE == GA_DEFL) && tid < N) ? s[tid] : 0.0;      // signs, or q'X of the deflation
    __syncthreads();
    const double den = (MODE == GA_PASS) ? *sumw : 1.0;
    const int my_tiles = ((int)blockIdx.x < ntiles) ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    auto issue = [&](int i, int sg) {
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        const uint32_t bar = ga_smem_u32(&full[sg]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(STG * 8) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
            ::"r"(ga_smem_u32(stage + sg * STG)), "l"(&mX), "r"(tile * GA_R), "r"(0), "r"(bar) : "memory");
    };
    if (tid == 0)
        for (int i = 0; i < nstage && i < my_tiles; ++i) issue(i, i);
    double tacc = 0.0, tacc2 = 0.0, mm = 0.0;
    int sg = 0;
    uint32_t phase = 0;
    for (int i = 0; i < my_tiles; ++i) {
        const int64_t row = (int64_t)((int)blockIdx.x + i * (int)gridDim.x) * GA_R + lane;
        const bool rok = row < d;
        if (MODE == GA_DOTS && warp == 0) mus[lane] = rok ? vec[row] : 0.0;
        if (MODE == GA_DEFL && warp == 0) mus[lane] = (rok && q2) ? q2[row] : 0.0;
        {
            const uint32_t bar = ga_smem_u32(&full[sg]);
            uint32_t done;
            do {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                             "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar), "r"(phase) : "memory");
            } while (!done);
        }
        double* Xs = stage + sg * STG;                         // [col][32 rows]; rows >= d and columns >= N are zero
        if (MODE == GA_DEFL) {
            // deflation X[i,n] -= q_i (q'X)_n (:272), written back in place (coalesced: lanes along rows) and kept in the
            // tile for the column sums of the NEXT component (norms^2 :265 and the first dot products :292)
            const double qi = rok ? vec[row] : 0.0;
#pragma unroll 8
            for (int k = 0; k < 32; ++k) {
                const int c = warp + 8 * k;
                const double x = fma(-qi, sv[c], Xs[c * GA_R + lane]);
                Xs[c * GA_R + lane] = x;
                if (rok && c < N) Xg[(int64_t)c * ld + row] = x;
            }
        }
        if (MODE == GA_PASS) {
            // phase A: v_row = sum_n s_n X[row, n]; warp w takes columns w, w + 8, ...
            double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
#pragma unroll
            for (int k = 0; k < 32; k += 4) {
                v0 = fma(sv[warp + 8 * k], Xs[(warp + 8 * k) * GA_R + lane], v0);
                v1 = fma(sv[warp + 8 * (k + 1)], Xs[(warp + 8 * (k + 1)) * GA_R + lane], v1);
                v2 = fma(sv[warp + 8 * (k + 2)], Xs[(warp + 8 * (k + 2)) * GA_R + lane], v2);
                v3 = fma(sv[warp + 8 * (k + 3)], Xs[(warp + 8 * (k + 3)) * GA_R + lane], v3);
            }
            red[warp * GA_R + lane] = (v0 + v1) + (v2 + v3);
            __syncthreads();
            if (warp == 0) {
                double v = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) v += red[w * GA_R + lane];
                const double m = v / den;                                       // s ./= ws   (:315)
                mus[lane] = rok ? m : 0.0;
                if (rok) { vec[row] = m; mm = fma(m, m, mm); }
            }
        }
        __syncthreads();
        // phase B: t[n] += sum_i X[i,n] * (mu_i | q_i | X[i,n]); thread <-> column, skewed (conflict-free) row order
        {
            double a0 = 0.0, a1 = 0.0;
            const double* col = Xs + tid * GA_R;
#pragma unroll
            for (int r = 0; r < GA_R; r += 2) {
                const int i0 = (r + tid) & (GA_R - 1), i1 = (r + 1 + tid) & (GA_R - 1);
                const double x0 = col[i0], x1 = col[i1];
                if (MODE == GA_NORMS || MODE == GA_DEFL) { a0 = fma(x0, x0, a0); a1 = fma(x1, x1, a1); }
                else { a0 = fma(x0, mus[i0], a0); a1 = fma(x1, mus[i1], a1); }
                if (MODE == GA_DEFL) tacc2 = fma(x0, mus[i0], fma(x1, mus[i1], tacc2));
            }
            tacc += a0 + a1;
        }
        if (MODE == GA_DEFL) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // tile was rewritten in place
        __syncthreads();                                       // everybody is done with the stage (and with mus / red)
        if (tid == 0 && i + nstage < my_tiles) issue(i + nstage, sg);
        if (++sg == nstage) { sg = 0; phase ^= 1u; }
    }
    double* P = part + (size_t)blockIdx.x * GA_PSTRIDE;
    P[tid] = tacc;
    P[GA_NC + 1 + tid] = tacc2;
    if (MODE == GA_PASS && warp == 0) {
        mm = warp_sum(mm);
        if (lane == 0) P[GA_NC] = mm;
    } else if (tid == 0) {
        P[GA_NC] = 0.0;
    }
}

// t[n] += sum over the CTAs (fixed order) of their partial column sums; slot N carries sum mu_i^2 (GA_PASS)
__global__ void __launch_bounds__(256)
ga_reduce_kernel(const double* __restrict__ part, int ncta, int N, int with_mm, double* __restrict__ t,
                 double* __restrict__ t2) {
    const int n = threadIdx.x;
    double acc = 0.0, acc2 = 0.0;
    for (int c = 0; c < ncta; ++c) {
        acc += part[(size_t)c * GA_PSTRIDE + n];
        if (t2) acc2 += part[(size_t)c * GA_PSTRIDE + GA_NC + 1 + n];
    }
    if (n < N) { t[n] += acc; if (t2) t2[n] += acc2; }
    if (with_mm && n == 0) {
        double m = 0.0;
        for (int c = 0; c < ncta; ++c) m += part[(size_t)c * GA_PSTRIDE + GA_NC];
        t[N] += m;
    }
}

typedef CUresult (*GaEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
GaEncodeFn ga_encode_fn() {
    static GaEncodeFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* q = nullptr;
        cudaDriverEntryPointQueryResult r;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &r) == cudaSuccess &&
            r == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<GaEncodeFn>(q);
        else
            cudaGetLastError();
    }
    return fn;
}

__global__ void __launch_bounds__(256)
ga_signs_kernel(const double* __restrict__ t, const double* __restrict__ norms2, int64_t N,
                double* __restrict__ s, double* __restrict__ sumw) {
    __shared__ double red[8];
    double local = 0.0;
    for (int64_t n = threadIdx.x; n < N; n += blockDim.x) {
        const double tn = t[n];
        const double nrm = sqrt(norms2[n]);                                   // Xnorms[n]   (:265)
        double sg = (tn > 0.0) ? 1.0 : ((tn < 0.0) ? -1.0 : 0.0);            // sign(U[:,n]'q)   (:292)
        if (!(nrm > 0.0)) sg = 0.0;
        s[n] = sg;
        local += sg * nrm;                                                    // ws += w[n]   (:312)
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[w];
        *sumw = v;
    }
}

__global__ void __launch_bounds__(256)
ga_update_kernel(const double* __restrict__ mu, const double* __restrict__ mm, int64_t d, const double* qold,
                 double* qnew, double* __restrict__ dq2) {
    const double nrm = sqrt(*mm);
    double local = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (int64_t)gridDim.x * blockDim.x) {
        const double qn = mu[i] / nrm;                                        // q .= mu ./ norm(mu)   (:295)
        const double df = qn - qold[i];
        local = fma(df, df, local);                                           // dq   (:296)
        qnew[i] = qn;                                                         // qold .= q   (:302)   (may alias qold)
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0 && local != 0.0) atomicAdd(dq2, local);
}

__global__ void __launch_bounds__(256)
vec_sumsq_kernel(const double* __restrict__ v, int64_t d, double* __restrict__ ss) {
    double local = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (int64_t)gridDim.x * blockDim.x)
        local = fma(v[i], v[i], local);
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0) atomicAdd(ss, local);
}

__global__ void __launch_bounds__(256)
vec_scale_rsqrt_kernel(const double* __restrict__ v, const double* __restrict__ ss, int64_t d,
                       double* __restrict__ out) {
    const double nrm = sqrt(*ss);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = v[i] / nrm;                                                  // q ./= norm(q)   (:287)
}

__global__ void __launch_bounds__(256)
ga_deflate_kernel(double* __restrict__ X, int64_t d, int64_t N, int64_t ld, const double* __restrict__ q,
                  const double* __restrict__ xs) {
    const int64_t total = d * N;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = idx % d, n = idx / d;
        const int64_t off = n * ld + i;
        X[off] = fma(-q[i], xs[n], X[off]);                                   // mul!(X, q, Xs1, -1, 1)   (:272)
    }
}

inline int vec_grid(int64_t total, int sm_count) {
    int64_t want = (total + 255) / 256;
    int64_t cap = (int64_t)sm_count * 8;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}


// ----------------------------------------------------------------------------------------------------------
// Robust entry-wise averages for rpca_ga (src/robustPCA.jl:323-333 entrywise_trimmed_mean, :349-357
// entrywise_median): per ROW j of the normalised data U[j,n] = X[j,n]/||x_n|| a sort over the N observations.
// A block stages 32 consecutive rows x N columns in shared memory with coalesced loads (lanes along rows); every
// warp then sorts its rows one after the other with a bitonic network on (key, index) pairs -- the index breaks ties
// like the reference's stable sortperm.
//   kind 1: keys = U[j,:]; s[j] = sum_{n in I} w_n U[j,n] / sum_{n in I} w_n, I = sorted[lo:hi)
//   kind 2: keys = w .* U[j,:]; m = sorted[N/2 - 1]; s[j] = sign(w_m) U[j,m]
// w_n = sgn_n * sqrt(n2_n) (sgn from the previous sweep's dot products, :291-293).
// ----------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ga_robust_kernel(const double* __restrict__ X, int64_t d, int N, int NP2, int RT, int64_t ld,
                 const double* __restrict__ sgn, const double* __restrict__ n2, int kind, int lo, int hi,
                 double* __restrict__ out) {
    extern __shared__ double smr[];
    const int TS = RT + 1;                                // RT rows per tile (32, or 8 for long observation axes)
    double* tile = smr;                                   // [N][RT + 1]  (padded: rows along the fast index)
    double* wv = tile + (size_t)N * TS;                   // [N] weights
    double* inv = wv + N;                                 // [N] 1 / ||x_n||
    double* keys = inv + N;                               // [8 warps][NP2]
    int* idxs = reinterpret_cast<int*>(keys + 8 * NP2);   // [8 warps][NP2]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int n = tid; n < N; n += 256) {
        const double nr = sqrt(n2[n]);
        wv[n] = sgn[n] * nr;
        inv[n] = nr;
    }
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    for (int64_t r0 = (int64_t)blockIdx.x * RT; r0 < d; r0 += (int64_t)gridDim.x * RT) {
        __syncthreads();
        for (int idx = tid; idx < N * RT; idx += 256) {
            const int n = idx / RT, r = idx % RT;
            const int64_t row = r0 + r;
            tile[n * TS + r] = row < d ? __ldg(X + (int64_t)n * ld + row) : 0.0;
        }
        __syncthreads();
        double* kk = keys + warp * NP2;
        int* ii = idxs + warp * NP2;
        for (int rr = warp; rr < RT; rr += 8) {
            const int64_t row = r0 + rr;
            if (row >= d) break;
            for (int n = lane; n < NP2; n += 32) {
                double u = INF;
                if (n < N) {
                    u = tile[n * TS + rr] / inv[n];                              // U[j,n] = X[j,n] / Xnorms[n]   :266
                    if (kind == 2) u = wv[n] * u;
                }
                kk[n] = u;
                ii[n] = n;
            }
            __syncwarp();
            for (int k = 2; k <= NP2; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int t = lane; t < NP2 / 2; t += 32) {
                        const int a = 2 * t - (t & (j - 1));                      // lower index of the pair (bit j clear)
                        const int b = a + j;
                        const bool up = (a & k) == 0;
                        const double ka = kk[a], kb = kk[b];
                        const int ia = ii[a], ib = ii[b];
                        const bool gt = (ka > kb) || (ka == kb && ia > ib);
                        if (gt == up) { kk[a] = kb; kk[b] = ka; ii[a] = ib; ii[b] = ia; }
                    }
                    __syncwarp();
                }
            if (kind == 1) {
                double num = 0.0, den = 0.0;
                for (int p = lo + lane; p < hi; p += 32) {
                    const double w = wv[ii[p]];
                    num = fma(w, kk[p], num);
                    den += w;
                }
                num = warp_sum(num);
                den = warp_sum(den);
                if (lane == 0) out[row] = num / den;
            } else if (lane == 0) {
                const int m = ii[N / 2 - 1];
                const double w = wv[m];
                const double u = tile[m * TS + rr] / inv[m];
                out[row] = (w > 0.0 ? 1.0 : (w < 0.0 ? -1.0 : 0.0)) * u;
            }
            __syncwarp();
        }
    }
}

// Long observation axes (1024 < N <= 16384): one CTA sorts one row at a time, keys and indices of the whole row in
// shared memory (block-wide bitonic network), weights and norms through the read-only path.  Same selection rules as
// ga_robust_kernel; a slow path for shapes the reference's tests never reach, but the result is defined for them.
__global__ void __launch_bounds__(512)
ga_robust_big_kernel(const double* __restrict__ X, int64_t d, int N, int NP2, int64_t ld, const double* __restrict__ sgn,
                     const double* __restrict__ n2, int kind, int lo, int hi, double* __restrict__ out) {
    extern __shared__ double smb[];
    double* kk = smb;                                     // [NP2]
    int* ii = reinterpret_cast<int*>(kk + NP2);           // [NP2]
    __shared__ double rn[16], rd[16];
    const int tid = threadIdx.x;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    for (int64_t row = blockIdx.x; row < d; row += gridDim.x) {
        __syncthreads();
        for (int n = tid; n < NP2; n += blockDim.x) {
            double u = INF;
            if (n < N) {
                const double nr = sqrt(__ldg(n2 + n));
                u = __ldg(X + (int64_t)n * ld + row) / nr;                       // U[j,n] = X[j,n] / Xnorms[n]   :266
                if (kind == 2) u = (__ldg(sgn + n) * nr) * u;
            }
            kk[n] = u;
            ii[n] = n;
        }
        __syncthreads();
        for (int k = 2; k <= NP2; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < NP2 / 2; t += blockDim.x) {
                    const int a = 2 * t - (t & (j - 1));
                    const int b = a + j;
                    const bool up = (a & k) == 0;
                    const double ka = kk[a], kb = kk[b];
                    const int ia = ii[a], ib = ii[b];
                    const bool gt = (ka > kb) || (ka == kb && ia > ib);
                    if (gt == up) { kk[a] = kb; kk[b] = ka; ii[a] = ib; ii[b] = ia; }
                }
                __syncthreads();
            }
        if (kind == 1) {
            double num = 0.0, den = 0.0;
            for (int p = lo + tid; p < hi; p += blockDim.x) {
                const int n = ii[p];
                const double w = __ldg(sgn + n) * sqrt(__ldg(n2 + n));
                num = fma(w, kk[p], num);
                den += w;
            }
            num = warp_sum(num);
            den = warp_sum(den);
            if ((tid & 31) == 0) { rn[tid >> 5] = num; rd[tid >> 5] = den; }
            __syncthreads();
            if (tid == 0) {
                double a = 0.0, b = 0.0;
                for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += rn[w]; b += rd[w]; }
                out[row] = a / b;
            }
        } else if (tid == 0) {
            const int m = ii[N / 2 - 1];
            const double nr = sqrt(__ldg(n2 + m));
            const double w = __ldg(sgn + m) * nr;
            const double u = __ldg(X + (int64_t)m * ld + row) / nr;
            out[row] = (w > 0.0 ? 1.0 : (w < 0.0 ? -1.0 : 0.0)) * u;
        }
    }
}

}  // namespace

size_t ga_partial_doubles(int sm_count) { return (size_t)sm_count * GA_PSTRIDE; }

namespace {
bool ga_tma_ok(const double* X, int64_t d, int64_t N, int64_t ld, const double* part) {
    return part && N <= GA_NC && N >= 8 && d >= 8192 && !(ld & 1) && !(reinterpret_cast<uintptr_t>(X) & 15) &&
           d < ((int64_t)1 << 31) && ga_encode_fn() != nullptr;
}
bool ga_encode(CUtensorMap* map, const double* X, int64_t d, int64_t N, int64_t ld) {
    const cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)N};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * 8};
    const cuuint32_t box[2] = {(cuuint32_t)GA_R, (cuuint32_t)GA_NC};
    const cuuint32_t estr[2] = {1, 1};
    return ga_encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(X), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace

// Fused tail of one component and head of the next (TMA kernel only): X -= q xs' in place (:272), n2[n] += |x_n|^2 of
// the deflated columns (:265) and, when q2 != null, t2[n] += x_n'q2 (the first dot products, :292).  Returns
// cudaErrorNotSupported when the shape does not qualify (the caller then runs the separate kernels).
cudaError_t launch_ga_deflate_fused(double* X, int64_t d, int64_t N, int64_t ld, const double* q, const double* xs,
                                    const double* q2, double* n2, double* t2, double* part, int sm_count,
                                    cudaStream_t st, int64_t* launches) {
    if (!ga_tma_ok(X, d, N, ld, part)) return cudaErrorNotSupported;
    CUtensorMap map;
    if (!ga_encode(&map, X, d, N, ld)) return cudaErrorNotSupported;
    const int ntiles = (int)((d + GA_R - 1) / GA_R);
    const int nstage = 3;
    const size_t smem = (size_t)nstage * GA_NC * GA_R * sizeof(double);
    const int grid = sm_count < ntiles ? sm_count : ntiles;
    auto kern = ga_sweep_tma_kernel<GA_DEFL>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, 256, smem, st>>>(map, d, (int)N, const_cast<double*>(q), xs, nullptr, part, ntiles, nstage, X, ld, q2);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    ga_reduce_kernel<<<1, 256, 0, st>>>(part, grid, (int)N, 0, n2, q2 ? t2 : nullptr);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

// xs[n] = t[n] / sqrt(t[N]):  q'x_n from the dot products x_n'mu of the converged iteration (q = mu / |mu|)
__global__ void ga_xs_kernel(const double* __restrict__ t, int64_t N, double* __restrict__ xs) {
    const double nrm = sqrt(t[N]);
    for (int64_t n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) xs[n] = t[n] / nrm;
}
cudaError_t launch_ga_xs(const double* t, int64_t N, double* xs, cudaStream_t st, int64_t* launches) {
    ga_xs_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(t, N, xs);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ga_sweep(GaMode mode, const double* X, int64_t d, int64_t N, int64_t ld, double* vec,
                            const double* s, const double* sumw, double* t, int sm_count, cudaStream_t st,
                            int64_t* launches, double* part) {
    const int ntiles = (int)((d + GA_R - 1) / GA_R);
    cudaError_t e;
    // TMA-staged kernel: one column chunk, 16-byte aligned base / stride, enough rows to fill the ring, workspace given
    if (ga_tma_ok(X, d, N, ld, part)) {
        CUtensorMap map;
        if (ga_encode(&map, X, d, N, ld)) {
            const int nstage = 3;
            const size_t smem = (size_t)nstage * GA_NC * GA_R * sizeof(double);
            int grid = sm_count < ntiles ? sm_count : ntiles;
#define TLSQ_GA_TMA_LAUNCH(MODE)                                                                                  \
            do {                                                                                                  \
                auto kern = ga_sweep_tma_kernel<MODE>;                                                            \
                e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);           \
                if (e != cudaSuccess) return e;                                                                   \
                kern<<<grid, 256, smem, st>>>(map, d, (int)N, vec, s, sumw, part, ntiles, nstage, nullptr, ld,    \
                                              nullptr);                                                           \
            } while (0)
            switch (mode) {
                case GA_NORMS: TLSQ_GA_TMA_LAUNCH(GA_NORMS); break;
                case GA_DOTS:  TLSQ_GA_TMA_LAUNCH(GA_DOTS); break;
                default:       TLSQ_GA_TMA_LAUNCH(GA_PASS); break;
            }
#undef TLSQ_GA_TMA_LAUNCH
            if ((e = cudaGetLastError()) != cudaSuccess) return e;
            ga_reduce_kernel<<<1, 256, 0, st>>>(part, grid, (int)N, mode == GA_PASS ? 1 : 0, t, nullptr);
            if (launches) *launches += 2;
            return cudaGetLastError();
        }
    }
    int grid = sm_count * 3;
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
    const size_t smem = (size_t)(GA_NC * GA_R + GA_NC + 8 * GA_R + GA_R) * sizeof(double);
#define TLSQ_GA_LAUNCH(MODE)                                                                          \
    do {                                                                                              \
        auto kern = ga_sweep_kernel<MODE>;                                                            \
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
        if (e != cudaSuccess) return e;                                                               \
        kern<<<grid, 256, smem, st>>>(X, d, N, ld, vec, s, sumw, t, ntiles);                          \
    } while (0)
    switch (mode) {
        case GA_NORMS: TLSQ_GA_LAUNCH(GA_NORMS); break;
        case GA_DOTS:  TLSQ_GA_LAUNCH(GA_DOTS); break;
        default:       TLSQ_GA_LAUNCH(GA_PASS); break;
    }
#undef TLSQ_GA_LAUNCH
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ga_signs(const double* t, const double* norms2, int64_t N, double* s, double* sumw,
                            cudaStream_t st, int64_t* launches) {
    ga_signs_kernel<<<1, 256, 0, st>>>(t, norms2, N, s, sumw);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ga_update(const double* mu, const double* mm, int64_t d, const double* qold, double* qnew, double* dq2,
                             int sm_count, cudaStream_t st, int64_t* launches) {
    ga_update_kernel<<<vec_grid(d, sm_count), 256, 0, st>>>(mu, mm, d, qold, qnew, dq2);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_vec_sumsq(const double* v, int64_t d, double* ss, int sm_count, cudaStream_t st,
                             int64_t* launches) {
    vec_sumsq_kernel<<<vec_grid(d, sm_count), 256, 0, st>>>(v, d, ss);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_vec_scale_rsqrt(const double* v, const double* ss, int64_t d, double* out, int sm_count,
                                   cudaStream_t st, int64_t* launches) {
    vec_scale_rsqrt_kernel<<<vec_grid(d, sm_count), 256, 0, st>>>(v, ss, d, out);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ga_deflate(double* X, int64_t d, int64_t N, int64_t ld, const double* q, const double* xs,
                              int sm_count, cudaStream_t st, int64_t* launches) {
    ga_deflate_kernel<<<vec_grid(d * N, sm_count), 256, 0, st>>>(X, d, N, ld, q, xs);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ga_robust(const double* X, int64_t d, int64_t N, int64_t ld, const double* sgn, const double* n2,
                             int kind, double P, double* out, int sm_count, cudaStream_t st, int64_t* launches) {
    int np2 = 2;
    while (np2 < N) np2 <<= 1;
    int rt = 32;
    auto need = [&](int rows) {
        return ((size_t)N * (rows + 1) + 2 * (size_t)N + 8 * (size_t)np2) * sizeof(double) + 8 * (size_t)np2 * sizeof(int);
    };
    if (need(rt) > (size_t)220 * 1024) rt = 8;
    const size_t smem = need(rt);
    const int lo_ = (int)floor(P * (double)N), hi_ = (int)floor((1.0 - P) * (double)N);    // :325
    if (smem > (size_t)220 * 1024) {
        // long observation axis: one row per CTA, the whole row sorted in shared memory (N <= kGaRobustMaxN)
        const size_t smb = (size_t)np2 * (sizeof(double) + sizeof(int));
        if (N > kGaRobustMaxN || smb > (size_t)220 * 1024) return cudaErrorInvalidValue;
        cudaError_t e = cudaFuncSetAttribute(ga_robust_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smb);
        if (e != cudaSuccess) return e;
        int64_t blocks = d < (int64_t)sm_count ? d : (int64_t)sm_count;
        ga_robust_big_kernel<<<(unsigned)blocks, 512, smb, st>>>(X, d, (int)N, np2, ld, sgn, n2, kind, lo_, hi_, out);
        if (launches) *launches += 1;
        return cudaGetLastError();
    }
    static size_t attr = 0;
    if (smem > attr) {
        cudaError_t e = cudaFuncSetAttribute(ga_robust_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr = smem;
    }
    const int lo = (int)floor(P * (double)N), hi = (int)floor((1.0 - P) * (double)N);      // :325
    int64_t blocks = (d + rt - 1) / rt;
    if (blocks > (int64_t)sm_count * 2) blocks = (int64_t)sm_count * 2;
    ga_robust_kernel<<<(unsigned)blocks, 256, smem, st>>>(X, d, (int)N, np2, rt, ld, sgn, n2, kind, lo, hi, out);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

}  // namespace tlsq
