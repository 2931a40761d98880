// elementwise.cu -- streaming helper kernels: max|D| (src/robustPCA.jl:178), Y = D/dual & A = 0 (:174-181),
// E recomputation for the returned value (:188-191,238), transpose (M < N inputs), hankel / unhankel
// (:76-92, :28-39, :53-68).
#include "kernels.h"

namespace tlsq {

namespace {

// max |x_i| over a contiguous array (dense D with ld == M, or the signal span of an implicit Hankel matrix: every
// sample y[0 .. (M-1) lag + N - 1] appears in H because lag <= N, src/robustPCA.jl:80)
__global__ void __launch_bounds__(256)
maxabs_linear_kernel(const double* __restrict__ x, int64_t total, double* __restrict__ out) {
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; idx + 3 * stride < total; idx += 4 * stride) {
        m0 = fmax(m0, fabs(__ldg(x + idx)));
        m1 = fmax(m1, fabs(__ldg(x + idx + stride)));
        m2 = fmax(m2, fabs(__ldg(x + idx + 2 * stride)));
        m3 = fmax(m3, fabs(__ldg(x + idx + 3 * stride)));
    }
    for (; idx < total; idx += stride) m0 = fmax(m0, fabs(__ldg(x + idx)));
    double m = warp_max(fmax(fmax(m0, m1), fmax(m2, m3)));
    // non-negative doubles order like their bit patterns
    if ((threadIdx.x & 31) == 0)
        atomicMax(reinterpret_cast<unsigned long long*>(out), (unsigned long long)__double_as_longlong(m));
}

// dense D with a leading dimension > M: thread <-> row, loop over the columns (no 64-bit divisions)
__global__ void __launch_bounds__(256)
maxabs_kernel(const MatSrc D, int64_t M, int64_t N, double* __restrict__ out) {
    double m = 0.0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < M; row += (int64_t)gridDim.x * blockDim.x)
        for (int64_t col = 0; col < N; ++col) m = fmax(m, fabs(__ldg(D.p + col * D.ld + row)));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0)
        atomicMax(reinterpret_cast<unsigned long long*>(out), (unsigned long long)__double_as_longlong(m));
}

// Y = D / dual (:181), A = 0, and (optionally) the first SVT input W_1; thread <-> row, coalesced column sweeps
template <bool HANKEL>
__global__ void __launch_bounds__(256)
init_ya_kernel(const MatSrc D, int64_t M, int64_t N, double dual, double* __restrict__ Y, double* __restrict__ A,
               double* __restrict__ W, double im, double eps, int nonnegE, int64_t ldy) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < M; row += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll 4
        for (int64_t col = 0; col < N; ++col) {
            const double d = src_at<HANKEL>(D, row, col);
            const double y = __ddiv_rn(d, dual);                         // Y ./= dual_norm   (:181)
            Y[col * ldy + row] = y;
            if (A) A[col * M + row] = 0.0;
            if (W) {
                double e, w;
                alm_ew(d, 0.0, y, im, eps, nonnegE, e, w);               // first SVT input   (:188-192)
                W[col * M + row] = w;
            }
        }
    }
}

template <bool HANKEL>
__global__ void __launch_bounds__(256)
compute_e_kernel(const MatSrc D, int64_t M, int64_t N, const double* __restrict__ A, const double* __restrict__ Y,
                 double im, double eps, int nonnegE, double* __restrict__ E, double* __restrict__ Wout) {
    const int64_t total = M * N;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = idx % M, col = idx / M;
        double e, w;
        alm_ew(src_at<HANKEL>(D, row, col), A[idx], Y[idx], im, eps, nonnegE, e, w);
        if (E) E[idx] = e;
        if (Wout) Wout[idx] = w;
    }
}

__global__ void __launch_bounds__(256)
transpose_kernel(const double* __restrict__ in, int64_t M, int64_t N, double* __restrict__ out) {
    __shared__ double tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t i0 = (int64_t)blockIdx.x * 32, j0 = (int64_t)blockIdx.y * 32;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t i = i0 + tx, j = j0 + ty + 8 * r;
        if (i < M && j < N) tile[ty + 8 * r][tx] = in[j * M + i];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t j = j0 + tx, i = i0 + ty + 8 * r;
        if (i < M && j < N) out[i * N + j] = tile[tx][ty + 8 * r];
    }
}

__global__ void __launch_bounds__(256)
hankel_kernel(const double* __restrict__ x, int64_t K, int64_t L, int64_t lag, double* __restrict__ H) {
    const int64_t total = K * L;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = idx % K, l = idx / K;
        H[idx] = x[k * lag + l];                                     // X[k, l] = x[(k-1)lag + l]   (:87-88)
    }
}

// y[t] = mean over {(k,l): k*lag + l == t} of A[k,l]; entries are visited for increasing l (column-major order of
// the reference's accumulation, :62-65); for lag == 1 this is the anti-diagonal mean (:28-39).
__global__ void __launch_bounds__(256)
unhankel_kernel(const double* __restrict__ A, int64_t K, int64_t L, int64_t lag, int64_t Ns,
                double* __restrict__ y) {
    for (int64_t tt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; tt < Ns;
         tt += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        int64_t cnt = 0;
        for (int64_t l = 0; l < L; ++l) {
            const int64_t rem = tt - l;
            if (rem < 0) break;
            if (rem % lag) continue;
            const int64_t k = rem / lag;
            if (k >= K) continue;
            s += A[l * K + k];
            ++cnt;
        }
        y[tt] = s / (double)(cnt > 0 ? cnt : 1);                     // y ./= max.(counts, 1)   (:66)
    }
}

// sharded unhankel: this rank owns Hankel rows [r0, r0 + Kl); sums/counts of the anti-diagonals it touches
__global__ void __launch_bounds__(256)
unhankel_partial_kernel(const double* __restrict__ A, int64_t r0, int64_t Kl, int64_t L, int64_t lag, int64_t Ns,
                        double* __restrict__ sum, double* __restrict__ cnt) {
    const int64_t t_lo = r0 * lag, t_hi = (r0 + Kl - 1) * lag + L;          // [t_lo, t_hi)
    for (int64_t tt = t_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; tt < t_hi && tt < Ns;
         tt += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        int64_t c = 0;
        for (int64_t l = 0; l < L; ++l) {
            const int64_t rem = tt - l;
            if (rem < 0) break;
            if (rem % lag) continue;
            const int64_t k = rem / lag - r0;
            if (k < 0 || k >= Kl) continue;
            s += A[l * Kl + k];
            ++c;
        }
        sum[tt] = s;
        cnt[tt] = (double)c;
    }
}

__global__ void __launch_bounds__(256)
unhankel_divide_kernel(const double* __restrict__ sum, const double* __restrict__ cnt, int64_t Ns, double* __restrict__ y) {
    for (int64_t tt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; tt < Ns; tt += (int64_t)gridDim.x * blockDim.x) {
        const double c = cnt[tt];
        y[tt] = sum[tt] / (c > 0.0 ? c : 1.0);                                 // y ./= max.(counts, 1)   (:66)
    }
}

// Sums of A = clamp(T V') over {(k, j): k lag + j = t} for the local Hankel rows k in [r0, r0 + Kl), WITHOUT
// materialising A (unhankel of src/robustPCA.jl:53-68 applied to the factored iterate; lag 1 is :28-39):
//   sum[t] = sum_{j = t mod lag, step lag} clamp(T[(t - j) / lag - r0, :] . V[j, :]),   0 <= (t - j) / lag - r0 < Kl
// Terms are added for increasing j (decreasing k), the order of unhankel_kernel, so the sums are those of the dense
// route bit for bit.  A block owns 256 consecutive samples t; the rows k with 0 <= t - k lag < n for some of them,
// k in [ceil((t0 - n + 1) / lag), floor((t0 + 255) / lag)], at most (254 + n) / lag + 1, are staged in shared memory.
__device__ __forceinline__ int64_t ceil_div_any(int64_t a, int64_t b) {        // b > 0, a of either sign
    return a >= 0 ? (a + b - 1) / b : -((-a) / b);
}

__global__ void __launch_bounds__(256)
unhankel_factors_kernel(const double* __restrict__ T, int64_t ldt, const double* __restrict__ V, int rp, int nonnegA,
                        int64_t r0, int64_t Kl, int n, int lag, int64_t Ns, double* __restrict__ sum) {
    extern __shared__ double sm[];
    const int span = (254 + n) / lag + 1;
    double* Vsm = sm;                        // [n][rp]
    double* Tsm = sm + (size_t)n * rp;       // [rp][span]
    for (int idx = threadIdx.x; idx < n * rp; idx += 256) {
        const int j = idx % n, c = idx / n;
        Vsm[j * rp + c] = __ldg(V + (int64_t)c * n + j);
    }
    const int64_t nblk = (Ns + 255) / 256;
    for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        const int64_t tb = b * 256;
        const int64_t klo = ceil_div_any(tb - (n - 1), lag);      // first staged Hankel row
        const int64_t ilo = klo - r0;
        __syncthreads();
        for (int idx = threadIdx.x; idx < rp * span; idx += 256) {
            const int q = idx % span, c = idx / span;
            const int64_t i = ilo + q;
            Tsm[c * span + q] = (i >= 0 && i < Kl) ? __ldg(T + (int64_t)c * ldt + i) : 0.0;
        }
        __syncthreads();
        const int64_t t = tb + threadIdx.x;
        if (t < Ns) {
            double s = 0.0;
            const int j0 = (int)((tb % lag + threadIdx.x) % lag);
            int q = (int)((t - j0) / lag - klo);                   // staged row of (t, j): one less per step of j
            for (int j = j0; j < n; j += lag, --q) {
                const int64_t i = ilo + q;
                if (i < 0 || i >= Kl) continue;
                double av = 0.0;
                for (int c = 0; c < rp; ++c) av = fma(Tsm[c * span + q], Vsm[j * rp + c], av);
                if (nonnegA) av = (__double_as_longlong(av) > 0) ? av : 0.0;
                s += av;
            }
            sum[t] = s;
        }
    }
}

// Same result without shared-memory staging (V and T through the read-only path): taken when [n][rp] + [rp][span] does
// not fit in shared memory (n > 256 with a large rank estimate).  Once per solve, latency is irrelevant.
__global__ void __launch_bounds__(256)
unhankel_factors_direct_kernel(const double* __restrict__ T, int64_t ldt, const double* __restrict__ V, int rp,
                               int nonnegA, int64_t r0, int64_t Kl, int n, int lag, int64_t Ns,
                               double* __restrict__ sum) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < Ns; t += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        const int j0 = (int)(t % lag);
        int64_t i = (t - j0) / lag - r0;                          // local row of (t, j): one less per step of j
        for (int j = j0; j < n; j += lag, --i) {
            if (i < 0 || i >= Kl) continue;
            double av = 0.0;
            for (int c = 0; c < rp; ++c) av = fma(__ldg(T + (int64_t)c * ldt + i), __ldg(V + (int64_t)c * n + j), av);
            if (nonnegA) av = (__double_as_longlong(av) > 0) ? av : 0.0;
            s += av;
        }
        sum[t] = s;
    }
}

// y[t] = sum[t] / max(#{k in [0, K): 0 <= t - k lag < n}, 1)   (:66; the count is known in closed form: k runs from
// max(0, ceil((t - n + 1) / lag)) to min(K - 1, floor(t / lag)).  Samples no row covers -- the last (Ns - n) % lag --
// have sum 0 and get 0.)
__global__ void __launch_bounds__(256)
unhankel_divide_count_kernel(const double* __restrict__ sum, int64_t K, int64_t n, int64_t lag, int64_t Ns,
                             double* __restrict__ y) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < Ns; t += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = lag == 1 ? t - n + 1 : ceil_div_any(t - n + 1, lag), hi = lag == 1 ? t : t / lag;
        if (lo < 0) lo = 0;
        if (hi > K - 1) hi = K - 1;
        const int64_t c = hi >= lo ? hi - lo + 1 : 1;
        y[t] = sum[t] / (double)c;
    }
}

// multi-channel trajectory matrix (:83-90): x is Ns x D (column-major), H is K x (L*D), H[k, l*D + d] = x[k*lag + l, d]
__global__ void __launch_bounds__(256)
hankel_mc_kernel(const double* __restrict__ x, int64_t Ns, int64_t D, int64_t K, int64_t L, int64_t lag,
                 double* __restrict__ H) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < K; k += (int64_t)gridDim.x * blockDim.x)
        for (int64_t col = 0; col < L * D; ++col) {
            const int64_t l = col / D, d = col % D;
            H[col * K + k] = x[d * Ns + k * lag + l];
        }
}

// general unhankel (:53-68): y[t, d] = sum of A[k, l*D + d] over k*lag + l == t, divided by max(count, 1)
__global__ void __launch_bounds__(256)
unhankel_mc_kernel(const double* __restrict__ A, int64_t K, int64_t L, int64_t lag, int64_t Ns, int64_t D,
                   double* __restrict__ y) {
    const int64_t total = Ns * D;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t tt = idx % Ns, d = idx / Ns;
        double s = 0.0;
        int64_t cnt = 0;
        for (int64_t l = 0; l < L; ++l) {
            const int64_t rem = tt - l;
            if (rem < 0) break;
            if (rem % lag) continue;
            const int64_t k = rem / lag;
            if (k >= K) continue;
            s += A[(l * D + d) * K + k];
            ++cnt;
        }
        y[idx] = s / (double)(cnt > 0 ? cnt : 1);
    }
}

// rank-sv projection A = (H V_sv) V_sv' (the sv > 0 plain-SSA branch of lowrankfilter, :123-125); thread <-> row,
// V (n x n eigenvectors of H'H, ld n) is read through L1/L2, 16 components per sweep
template <bool HANKEL>
__global__ void __launch_bounds__(128)
ssa_project_kernel(const MatSrc H, int64_t M, int64_t N, const double* __restrict__ V, int sv, double* __restrict__ A) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < M; row += (int64_t)gridDim.x * blockDim.x) {
        for (int c0 = 0; c0 < sv; c0 += 16) {
            double t[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) t[c] = 0.0;
            for (int64_t j = 0; j < N; ++j) {
                const double hv = src_at<HANKEL>(H, row, j);
#pragma unroll
                for (int c = 0; c < 16; ++c)
                    if (c0 + c < sv) t[c] = fma(hv, __ldg(V + (int64_t)(c0 + c) * N + j), t[c]);
            }
            for (int64_t j = 0; j < N; ++j) {
                double acc = c0 ? A[j * M + row] : 0.0;
#pragma unroll
                for (int c = 0; c < 16; ++c)
                    if (c0 + c < sv) acc = fma(t[c], __ldg(V + (int64_t)(c0 + c) * N + j), acc);
                A[j * M + row] = acc;
            }
        }
    }
}

// soft_th(x, eps, l) = max(x - eps, l) + min(x + eps, l) - l            src/robustPCA.jl:2 (no FMA contraction)
__device__ __forceinline__ double soft_th_level(double x, double eps, double l) {
    return __dsub_rn(__dadd_rn(fmax(__dsub_rn(x, eps), l), fmin(__dadd_rn(x, eps), l)), l);
}

// hankel=true, second half of the iteration (thread <-> row):  A = soft_hankel(A_raw); clamp; E; Z; Y; ||Z||_F^2
template <bool HANKEL>
__global__ void __launch_bounds__(256)
hankel_finish_kernel(const EpiArgs a, const double* __restrict__ mean) {
    double zz = 0.0;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < a.M; row += (int64_t)gridDim.x * blockDim.x) {
        for (int64_t col = 0; col < a.N; ++col) {
            const int64_t off = col * a.ldw + row;
            const double d = src_at<HANKEL>(a.D, row, col);
            const double yp = __ldg(a.Yp + off);
            double e, w;
            alm_ew(d, __ldg(a.Ap + off), yp, a.im, a.eps, a.nonnegE, e, w);
            double an = soft_th_level(a.An[off], a.eps, __ldg(mean + row + col));        // soft_hankel!(A, lambda/mu) :215
            if (a.nonnegA) an = (__double_as_longlong(an) > 0) ? an : 0.0;               // :218
            const double z = __dsub_rn(__dsub_rn(d, an), e);                              // :221
            const double yn = __dadd_rn(yp, __dmul_rn(a.mu, z));                          // :222
            zz = fma(z, z, zz);
            a.An[off] = an;
            a.Yn[off] = yn;
            if (a.Zout) a.Zout[off] = z;
        }
    }
    zz = warp_sum(zz);
    if ((threadIdx.x & 31) == 0) atomicAdd(a.zz, zz);
}

// dense iterate, plain element-wise tail of an ALM iteration (callback path, solver.cu):
//   A = max(A, 0) [nonnegA] ; Z = (D - A) - E ; Y += mu Z ; zz += ||Z||_F^2              src/robustPCA.jl:217-222
__global__ void __launch_bounds__(256)
dense_update_kernel(const double* __restrict__ D, double* __restrict__ A, const double* __restrict__ E,
                    double* __restrict__ Y, double* __restrict__ Z, int64_t total, double mu, int nonnegA,
                    double* __restrict__ zz_out) {
    double zz = 0.0;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        double an = A[idx];
        if (nonnegA) { an = (__double_as_longlong(an) > 0) ? an : 0.0; A[idx] = an; }
        const double z = __dsub_rn(__dsub_rn(D[idx], an), E[idx]);
        Y[idx] = __dadd_rn(Y[idx], __dmul_rn(mu, z));
        Z[idx] = z;
        zz = fma(z, z, zz);
    }
    zz = warp_sum(zz);
    if ((threadIdx.x & 31) == 0) atomicAdd(zz_out, zz);
}

__global__ void __launch_bounds__(256)
soft_hankel_apply_kernel(double* __restrict__ X, int64_t M, int64_t N, const double* __restrict__ mean, double eps) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < M; row += (int64_t)gridDim.x * blockDim.x)
        for (int64_t col = 0; col < N; ++col)
            X[col * M + row] = soft_th_level(X[col * M + row], eps, __ldg(mean + row + col));
}

inline int stream_grid(int64_t total, int sm_count) {
    int64_t want = (total + 255) / 256;
    int64_t cap = (int64_t)sm_count * 8;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}

}  // namespace

cudaError_t launch_maxabs(const MatSrc& D, bool hankel, int64_t M, int64_t N, double* out, int sm_count,
                          cudaStream_t st, int64_t* launches) {
    if (hankel || D.ld == M) {
        const int64_t total = hankel ? (M - 1) * D.ld + N : M * N;
        maxabs_linear_kernel<<<stream_grid(total / 4 + 1, sm_count), 256, 0, st>>>(D.p, total, out);
    } else {
        maxabs_kernel<<<stream_grid(M, sm_count), 256, 0, st>>>(D, M, N, out);
    }
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_init_ya(const MatSrc& D, bool hankel, int64_t M, int64_t N, double dual, double* Y, double* A,
                           double* W, double im, double eps, int nonnegE, int sm_count, cudaStream_t st,
                           int64_t* launches, int64_t ldy) {
    const int grid = stream_grid(M, sm_count);
    if (ldy <= 0) ldy = M;
    if (hankel) init_ya_kernel<true><<<grid, 256, 0, st>>>(D, M, N, dual, Y, A, W, im, eps, nonnegE, ldy);
    else init_ya_kernel<false><<<grid, 256, 0, st>>>(D, M, N, dual, Y, A, W, im, eps, nonnegE, ldy);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_compute_e(const MatSrc& D, bool hankel, int64_t M, int64_t N, const double* A, const double* Y,
                             double im, double eps, int nonnegE, double* E, int sm_count, cudaStream_t st,
                             int64_t* launches, double* Wout) {
    const int grid = stream_grid(M * N, sm_count);
    if (hankel) compute_e_kernel<true><<<grid, 256, 0, st>>>(D, M, N, A, Y, im, eps, nonnegE, E, Wout);
    else compute_e_kernel<false><<<grid, 256, 0, st>>>(D, M, N, A, Y, im, eps, nonnegE, E, Wout);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_transpose(const double* in, int64_t M, int64_t N, double* out, cudaStream_t st,
                             int64_t* launches) {
    dim3 grid((unsigned)((M + 31) / 32), (unsigned)((N + 31) / 32));
    transpose_kernel<<<grid, 256, 0, st>>>(in, M, N, out);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_hankel(const double* x, int64_t K, int64_t L, int64_t lag, double* H, cudaStream_t st,
                          int64_t* launches) {
    const int grid = stream_grid(K * L, 148);
    hankel_kernel<<<grid, 256, 0, st>>>(x, K, L, lag, H);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel(const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, double* y,
                            cudaStream_t st, int64_t* launches) {
    const int grid = stream_grid(Ns, 148);
    unhankel_kernel<<<grid, 256, 0, st>>>(A, K, L, lag, Ns, y);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel_partial(const double* A, int64_t r0, int64_t Kl, int64_t L, int64_t lag, int64_t Ns,
                                    double* sum, double* cnt, cudaStream_t st, int64_t* launches) {
    const int64_t span = (Kl - 1) * lag + L;
    unhankel_partial_kernel<<<stream_grid(span, 148), 256, 0, st>>>(A, r0, Kl, L, lag, Ns, sum, cnt);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel_divide(const double* sum, const double* cnt, int64_t Ns, double* y, cudaStream_t st,
                                   int64_t* launches) {
    unhankel_divide_kernel<<<stream_grid(Ns, 148), 256, 0, st>>>(sum, cnt, Ns, y);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel_factors(const double* T, int64_t ldt, const double* V, int svp, int nonnegA, int64_t r0,
                                    int64_t Kl, int64_t n, int64_t lag, int64_t Ns, double* sum, int sm_count,
                                    cudaStream_t st, int64_t* launches) {
    if (svp < 1) return cudaMemsetAsync(sum, 0, (size_t)Ns * sizeof(double), st);     // A = 0
    const int rp = svp;
    const size_t smem = ((size_t)n * rp + (size_t)rp * ((254 + n) / lag + 1)) * sizeof(double);
    if (smem > (size_t)220 * 1024) {
        int64_t blocks = (Ns + 255) / 256;
        if (blocks > (int64_t)sm_count * 8) blocks = (int64_t)sm_count * 8;
        unhankel_factors_direct_kernel<<<(unsigned)blocks, 256, 0, st>>>(T, ldt, V, rp, nonnegA, r0, Kl, (int)n, (int)lag,
                                                                          Ns, sum);
        if (launches) *launches += 1;
        return cudaGetLastError();
    }
    // function attributes are per device: set on every launch (a process may run on several GPUs)
    cudaError_t e = cudaFuncSetAttribute(unhankel_factors_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t blocks = (Ns + 255) / 256;
    if (blocks > (int64_t)sm_count * 4) blocks = (int64_t)sm_count * 4;
    unhankel_factors_kernel<<<(unsigned)blocks, 256, smem, st>>>(T, ldt, V, rp, nonnegA, r0, Kl, (int)n, (int)lag, Ns,
                                                                 sum);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel_divide_count(const double* sum, int64_t K, int64_t n, int64_t lag, int64_t Ns, double* y,
                                         cudaStream_t st, int64_t* launches) {
    unhankel_divide_count_kernel<<<stream_grid(Ns, 148), 256, 0, st>>>(sum, K, n, lag, Ns, y);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_hankel_finish(const EpiArgs& a, bool hankel_src, const double* mean, int sm_count, cudaStream_t st,
                                 int64_t* launches) {
    const int grid = stream_grid(a.M, sm_count);
    if (hankel_src) hankel_finish_kernel<true><<<grid, 256, 0, st>>>(a, mean);
    else hankel_finish_kernel<false><<<grid, 256, 0, st>>>(a, mean);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_dense_update(const double* D, double* A, const double* E, double* Y, double* Z, int64_t M, int64_t N,
                                double mu, int nonnegA, double* zz, int sm_count, cudaStream_t st, int64_t* launches) {
    dense_update_kernel<<<stream_grid(M * N, sm_count), 256, 0, st>>>(D, A, E, Y, Z, M * N, mu, nonnegA, zz);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_soft_hankel_apply(double* X, int64_t M, int64_t N, const double* mean, double eps, int sm_count,
                                     cudaStream_t st, int64_t* launches) {
    soft_hankel_apply_kernel<<<stream_grid(M, sm_count), 256, 0, st>>>(X, M, N, mean, eps);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_hankel_mc(const double* x, int64_t Ns, int64_t D, int64_t K, int64_t L, int64_t lag, double* H,
                             cudaStream_t st, int64_t* launches) {
    hankel_mc_kernel<<<stream_grid(K, 148), 256, 0, st>>>(x, Ns, D, K, L, lag, H);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_unhankel_mc(const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, int64_t D, double* y,
                               cudaStream_t st, int64_t* launches) {
    unhankel_mc_kernel<<<stream_grid(Ns * D, 148), 256, 0, st>>>(A, K, L, lag, Ns, D, y);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_ssa_project(const MatSrc& H, bool hankel, int64_t M, int64_t N, const double* V, int sv, double* A,
                               int sm_count, cudaStream_t st, int64_t* launches) {
    int64_t blocks = (M + 127) / 128;
    if (blocks > (int64_t)sm_count * 16) blocks = (int64_t)sm_count * 16;
    if (hankel) ssa_project_kernel<true><<<(unsigned)blocks, 128, 0, st>>>(H, M, N, V, sv, A);
    else ssa_project_kernel<false><<<(unsigned)blocks, 128, 0, st>>>(H, M, N, V, sv, A);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

}  // namespace tlsq
