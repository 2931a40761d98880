// ga_select.cu -- the robust entry-wise averages of rpca_ga (src/robustPCA.jl:323-333, :349-357) for any number of
// observations, as per-row radix selection over streaming sweeps of X (no per-row sort, nothing of size d x N).
//
// Ordering is the reference's sortperm (stable argsort): ascending key, ties by ascending column index; keys compare
// as IEEE doubles with -0.0 == +0.0, and NaN keys (zero columns) sort last.  Each key is mapped to an order-preserving
// uint64 and the element of rank t of row j is found in two steps:
//   1. its key value kv: eight passes over X, each a per-row histogram of one byte of the keys that still match the
//      bytes found so far (integer counts only, so the result does not depend on the schedule);
//   2. its column: kv leaves t - #{key < kv} elements of the row equal to kv to skip; one pass counts those ties (and
//      notes the first one) per column split, and one warp per row picks the split that holds the wanted tie -- its
//      first tie, or a walk over its columns when earlier ties of the split are to be skipped (tied data only).
// Trimmed mean: the keys U[j,n] = X[j,n] / ||x_n|| do not depend on the weights, so the two boundaries of rows' kept
// range [lo, hi) are selected once per component and every iteration is one sweep that tests (key, n) against them.
// Median: the keys w_n U[j,n] change with the signs, so the selection runs every iteration.
//
// Work split of the sweeps: CTA (x, y) covers rows [x rt, x rt + rt) and column split y of S; thread t takes row
// t % rt and every (256 / rt)-th column of the split, so a warp reads whole 32-row (or d-row) column segments.
#include <cmath>
#include <cstdint>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int SEL_BINS = 256;
constexpr int SEL_THREADS = 256;
constexpr int SEL_UNROLL = 8;

// Where the keys come from.  n2 == nullptr: X already holds U and wt the weights w_n.  Otherwise (rpca_ga) X is the
// deflated data, u = X[j,n] / sqrt(n2[n]) and w_n = wt[n] sqrt(n2[n]) with wt the signs -- the same expressions as
// ga_robust_kernel, and the same key map sel_order, so the orders agree on both sides of kGaRobustMaxN
// (tests/test_gpu_ga_paths.py checks N = 16 384 and 16 385 on the same data kinds).
struct SelSrc {
    const double* X;
    int64_t ld;
    const double* wt;
    const double* n2;
    int kind;           // 1: key u (trimmed mean), 2: key w u (median)
};

struct SelPlan {
    int rt;             // rows per CTA (power of two, <= 32)
    int64_t tiles;      // row tiles
    int S;              // column splits
};

SelPlan sel_plan(int64_t d, int64_t N, int sm_count) {
    SelPlan p;
    p.rt = 1;
    while (p.rt < 32 && p.rt < d) p.rt <<= 1;
    p.tiles = (d + p.rt - 1) / p.rt;
    // about three resident CTAs per SM in total, and at least a few loads per thread in every split
    const int64_t want = 3 * (int64_t)sm_count;
    int64_t S = p.tiles >= want ? 1 : (want + p.tiles - 1) / p.tiles;
    const int64_t min_cols = (int64_t)(SEL_THREADS / p.rt) * SEL_UNROLL;
    const int64_t cap = (N + min_cols - 1) / min_cols;
    if (S > cap) S = cap;
    if (S > 65535) S = 65535;
    if (S < 1) S = 1;
    p.S = (int)S;
    return p;
}

// workspace layout (every array per row, or per row and split)
struct SelWs {
    uint64_t* pre;      // [2][d]  key prefix found so far (the whole key after the last pass)
    int64_t* rank;      // [2][d]  rank still to skip among the candidates
    int64_t* idx;       // [2][d]  column of the selected element
    unsigned* hist;     // [2][d][256]
    unsigned* cnt;      // [2][S][d]  ties per column split
    int64_t* first;     // [2][S][d]  column of the first tie in the split
    double* num;        // [S][d]  trimmed-mean partial sums
    double* den;        // [S][d]
};

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t sel_layout(int64_t d, const SelPlan& p, void* base, SelWs* w) {
    const size_t sizes[8] = {2 * (size_t)d * 8, 2 * (size_t)d * 8, 2 * (size_t)d * 8, 2 * (size_t)d * SEL_BINS * 4,
                             2 * (size_t)p.S * d * 4, 2 * (size_t)p.S * d * 8, (size_t)p.S * d * 8, (size_t)p.S * d * 8};
    size_t off[8], total = 0;
    for (int i = 0; i < 8; ++i) { off[i] = total; total += align256(sizes[i]); }
    if (w) {
        char* b = static_cast<char*>(base);
        w->pre = reinterpret_cast<uint64_t*>(b + off[0]);
        w->rank = reinterpret_cast<int64_t*>(b + off[1]);
        w->idx = reinterpret_cast<int64_t*>(b + off[2]);
        w->hist = reinterpret_cast<unsigned*>(b + off[3]);
        w->cnt = reinterpret_cast<unsigned*>(b + off[4]);
        w->first = reinterpret_cast<int64_t*>(b + off[5]);
        w->num = reinterpret_cast<double*>(b + off[6]);
        w->den = reinterpret_cast<double*>(b + off[7]);
    }
    return total;
}

// keys: sel_order (common.cuh), shared with the per-row sorts in ga.cu
__device__ __forceinline__ void sel_uw(const SelSrc& s, int64_t n, double x, double& u, double& w) {
    const double nr = s.n2 ? sqrt(__ldg(s.n2 + n)) : 1.0;
    u = x / nr;                                                            // U[j,n] = X[j,n] / Xnorms[n]   :266
    w = __ldg(s.wt + n) * nr;
}

__device__ __forceinline__ uint64_t sel_key(const SelSrc& s, int64_t n, double x) {
    if (s.kind == 1) {
        const double nr = s.n2 ? sqrt(__ldg(s.n2 + n)) : 1.0;
        return sel_order(x / nr);
    }
    double u, w;
    sel_uw(s, n, x, u, w);
    return sel_order(w * u);
}

__device__ __forceinline__ void sel_split(int64_t N, int S, int y, int64_t& c0, int64_t& c1) {
    c0 = N * y / S;
    c1 = N * (y + 1) / S;
}

// rank[k][j] = t[k], pre[k][j] = 0
__global__ void ga_sel_init_kernel(int64_t d, int T, int64_t t0, int64_t t1, uint64_t* pre, int64_t* rank) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < T * d; i += (int64_t)gridDim.x * blockDim.x) {
        pre[i] = 0;
        rank[i] = i < d ? t0 : t1;
    }
}

// One radix pass: hist[k][j][byte `shift` of the key] += 1 for every key of row j whose higher bytes equal pre[k][j]'s.
template <int T>
__global__ void __launch_bounds__(SEL_THREADS)
ga_sel_hist_kernel(SelSrc src, int64_t d, int64_t N, int rt, int S, int shift, const uint64_t* __restrict__ pre,
                   unsigned* __restrict__ hist) {
    extern __shared__ unsigned sh[];                                       // [T][rt][256]
    const int tid = threadIdx.x;
    for (int i = tid; i < T * rt * SEL_BINS; i += SEL_THREADS) sh[i] = 0;
    const int r = tid % rt, cstep = SEL_THREADS / rt;
    const int64_t row = (int64_t)blockIdx.x * rt + r;
    const bool rok = row < d;
    uint64_t p[T];
#pragma unroll
    for (int k = 0; k < T; ++k) p[k] = rok ? pre[k * d + row] : 0;
    __syncthreads();
    if (rok) {
        int64_t c0, c1;
        sel_split(N, S, blockIdx.y, c0, c1);
        const double* Xr = src.X + row;
        for (int64_t n = c0 + tid / rt; n < c1; n += (int64_t)cstep * SEL_UNROLL) {
            double x[SEL_UNROLL];
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                x[u] = nn < c1 ? __ldg(Xr + nn * src.ld) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                if (nn < c1) {
                    const uint64_t key = sel_key(src, nn, x[u]);
                    const unsigned bin = (unsigned)(key >> shift) & (SEL_BINS - 1);
#pragma unroll
                    for (int k = 0; k < T; ++k)
                        if (shift == 56 || ((key ^ p[k]) >> (shift + 8)) == 0)
                            atomicAdd(&sh[(k * rt + r) * SEL_BINS + bin], 1u);
                }
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < T * rt * SEL_BINS; i += SEL_THREADS) {
        const unsigned c = sh[i];
        const int k = i / (rt * SEL_BINS), rr = (i / SEL_BINS) % rt, bin = i % SEL_BINS;
        const int64_t rw = (int64_t)blockIdx.x * rt + rr;
        if (c && rw < d) atomicAdd(&hist[((int64_t)k * d + rw) * SEL_BINS + bin], c);
    }
}

// One warp per (target, row): the bin that holds the remaining rank fixes the next byte of the key; the rank drops by
// the candidates in lower bins.  The histogram row is cleared for the next pass.
__global__ void ga_sel_scan_kernel(int64_t d, int T, int shift, uint64_t* __restrict__ pre, int64_t* __restrict__ rank,
                                   unsigned* __restrict__ hist) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;       // k * d + row
    if (i >= T * d) return;
    unsigned* h = hist + i * SEL_BINS + lane * 8;
    unsigned c[8];
    unsigned long long own = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) { c[b] = h[b]; own += c[b]; h[b] = 0; }
    unsigned long long incl = own;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const long long r = rank[i];
    const long long excl = (long long)(incl - own);
    const unsigned hit = __ballot_sync(0xffffffffu, r >= excl && r < (long long)incl);
    if (hit && lane == __ffs(hit) - 1) {
        long long cum = excl;
        int b = 0;
        for (; b < 7; ++b) {
            if (r < cum + (long long)c[b]) break;
            cum += c[b];
        }
        pre[i] |= (uint64_t)(lane * 8 + b) << shift;
        rank[i] = r - cum;
    }
}

// ties: cnt[k][y][j] = #{n in split y : key(j, n) == pre[k][j]}, first[k][y][j] = the smallest such n
template <int T>
__global__ void __launch_bounds__(SEL_THREADS)
ga_sel_ties_kernel(SelSrc src, int64_t d, int64_t N, int rt, int S, const uint64_t* __restrict__ pre,
                   unsigned* __restrict__ cnt, int64_t* __restrict__ first) {
    __shared__ unsigned red[T][SEL_THREADS];
    __shared__ int64_t redf[T][SEL_THREADS];
    const int tid = threadIdx.x;
    const int r = tid % rt, cstep = SEL_THREADS / rt;
    const int64_t row = (int64_t)blockIdx.x * rt + r;
    const bool rok = row < d;
    unsigned c[T];
    int64_t f[T];
    uint64_t p[T];
#pragma unroll
    for (int k = 0; k < T; ++k) { c[k] = 0; f[k] = INT64_MAX; p[k] = rok ? pre[k * d + row] : 0; }
    if (rok) {
        int64_t c0, c1;
        sel_split(N, S, blockIdx.y, c0, c1);
        const double* Xr = src.X + row;
        for (int64_t n = c0 + tid / rt; n < c1; n += (int64_t)cstep * SEL_UNROLL) {
            double x[SEL_UNROLL];
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                x[u] = nn < c1 ? __ldg(Xr + nn * src.ld) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                if (nn < c1) {
                    const uint64_t key = sel_key(src, nn, x[u]);
#pragma unroll
                    for (int k = 0; k < T; ++k)
                        if (key == p[k]) {
                            c[k] += 1;
                            if (nn < f[k]) f[k] = nn;
                        }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < T; ++k) { red[k][tid] = c[k]; redf[k][tid] = f[k]; }
    __syncthreads();
    if (tid < rt && rok) {
#pragma unroll
        for (int k = 0; k < T; ++k) {
            unsigned s = 0;
            int64_t m = INT64_MAX;
            for (int q = tid; q < SEL_THREADS; q += rt) { s += red[k][q]; m = redf[k][q] < m ? redf[k][q] : m; }
            cnt[((int64_t)k * S + blockIdx.y) * d + row] = s;
            first[((int64_t)k * S + blockIdx.y) * d + row] = m;
        }
    }
}

// One warp per (target, row): the split that holds the remaining rank among the ties, then its first tie or, when
// earlier ties of the split are to be skipped, its columns in order.
// out != nullptr (median): out[row] = sign(w_m) U[row, m]   (:353-355)
__global__ void ga_sel_index_kernel(SelSrc src, int64_t d, int64_t N, int S, int T, const uint64_t* __restrict__ pre,
                                    const int64_t* __restrict__ rank, const unsigned* __restrict__ cnt,
                                    const int64_t* __restrict__ first, int64_t* __restrict__ idx,
                                    double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;       // k * d + row
    if (i >= T * d) return;
    const int k = (int)(i / d);
    const int64_t row = i - (int64_t)k * d;
    const uint64_t kv = pre[i];
    long long r = rank[i];
    int ys = -1;
    long long cum = 0;
    for (int y0 = 0; y0 < S && ys < 0; y0 += 32) {
        const long long c = y0 + lane < S ? (long long)cnt[((int64_t)k * S + y0 + lane) * d + row] : 0;
        long long incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const unsigned hit = __ballot_sync(0xffffffffu, r >= cum + incl - c && r < cum + incl);
        if (hit) {
            const int L = __ffs(hit) - 1;
            ys = y0 + L;
            r -= cum + __shfl_sync(0xffffffffu, incl - c, L);
        } else {
            cum += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    int64_t m = -1;
    if (ys >= 0 && r == 0) {
        m = first[((int64_t)k * S + ys) * d + row];
    } else if (ys >= 0) {
        int64_t c0, c1;
        sel_split(N, S, ys, c0, c1);
        for (int64_t n0 = c0; n0 < c1; n0 += 32) {
            const int64_t n = n0 + lane;
            const bool tie = n < c1 && sel_key(src, n, __ldg(src.X + n * src.ld + row)) == kv;
            const unsigned b = __ballot_sync(0xffffffffu, tie);
            const int pc = __popc(b);
            if (r < pc) {
                const unsigned at = __ballot_sync(0xffffffffu, tie && __popc(b & ((1u << lane) - 1u)) == r);
                m = n0 + __ffs(at) - 1;
                break;
            }
            r -= pc;
        }
    }
    if (lane == 0) {
        idx[i] = m;
        if (out) {
            double s = __longlong_as_double(0x7ff8000000000000LL);
            if (m >= 0) {
                double u, w;
                sel_uw(src, m, __ldg(src.X + m * src.ld + row), u, w);
                s = (w > 0.0 ? 1.0 : (w < 0.0 ? -1.0 : 0.0)) * u;
            }
            out[row] = s;
        }
    }
}

// Trimmed mean sweep: per row, sum_n w_n u_n and sum_n w_n over the (key, n) between the two selected boundaries;
// per-CTA partials in fixed order (no floating-point atomics).
__global__ void __launch_bounds__(SEL_THREADS)
ga_sel_trim_kernel(SelSrc src, int64_t d, int64_t N, int rt, int S, int empty, const uint64_t* __restrict__ pre,
                   const int64_t* __restrict__ idx, double* __restrict__ pnum, double* __restrict__ pden) {
    __shared__ double rn[SEL_THREADS], rd[SEL_THREADS];
    const int tid = threadIdx.x;
    const int r = tid % rt, cstep = SEL_THREADS / rt;
    const int64_t row = (int64_t)blockIdx.x * rt + r;
    const bool rok = row < d && !empty;
    double num = 0.0, den = 0.0;
    if (rok) {
        const uint64_t klo = pre[row], khi = pre[d + row];
        const int64_t nlo = idx[row], nhi = idx[d + row];
        int64_t c0, c1;
        sel_split(N, S, blockIdx.y, c0, c1);
        const double* Xr = src.X + row;
        for (int64_t n = c0 + tid / rt; n < c1; n += (int64_t)cstep * SEL_UNROLL) {
            double x[SEL_UNROLL];
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                x[u] = nn < c1 ? __ldg(Xr + nn * src.ld) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < SEL_UNROLL; ++u) {
                const int64_t nn = n + (int64_t)u * cstep;
                if (nn < c1) {
                    double uu, w;
                    sel_uw(src, nn, x[u], uu, w);
                    const uint64_t key = sel_order(uu);
                    const bool in = (key > klo || (key == klo && nn >= nlo)) && (key < khi || (key == khi && nn <= nhi));
                    if (in) {
                        num = fma(w, uu, num);
                        den += w;
                    }
                }
            }
        }
    }
    rn[tid] = num;
    rd[tid] = den;
    __syncthreads();
    if (tid < rt && row < d) {
        double a = 0.0, b = 0.0;
        for (int q = tid; q < SEL_THREADS; q += rt) { a += rn[q]; b += rd[q]; }
        pnum[(int64_t)blockIdx.y * d + row] = a;
        pden[(int64_t)blockIdx.y * d + row] = b;
    }
}

__global__ void ga_sel_trim_finish_kernel(int64_t d, int S, const double* __restrict__ pnum,
                                          const double* __restrict__ pden, double* __restrict__ out) {
    for (int64_t row = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; row < d; row += (int64_t)gridDim.x * blockDim.x) {
        double a = 0.0, b = 0.0;
        for (int y = 0; y < S; ++y) { a += pnum[(int64_t)y * d + row]; b += pden[(int64_t)y * d + row]; }
        out[row] = a / b;                                                  // s[j] = (w[I] U[j,I]) / sum(w[I])   :329
    }
}

// kept positions [lo, hi) of the stable order of each row (0-based, :325)
void trim_range(double P, int64_t N, int64_t* lo, int64_t* hi) {
    *lo = (int64_t)floor(P * (double)N);
    *hi = (int64_t)floor((1.0 - P) * (double)N);
}

unsigned grid_for(int64_t warps_or_threads, int per_block) {
    return (unsigned)((warps_or_threads + per_block - 1) / per_block);
}

// selection of the elements of ranks t0 (and t1 when T == 2) of every row: keys into w.pre, columns into w.idx
cudaError_t sel_run(const SelSrc& src, int64_t d, int64_t N, int T, int64_t t0, int64_t t1, const SelPlan& p,
                    const SelWs& w, double* out, cudaStream_t st, int64_t* launches) {
    cudaError_t e;
    if ((e = cudaMemsetAsync(w.hist, 0, (size_t)T * d * SEL_BINS * 4, st)) != cudaSuccess) return e;
    ga_sel_init_kernel<<<grid_for(T * d, 256) < 1024 ? grid_for(T * d, 256) : 1024, 256, 0, st>>>(d, T, t0, t1, w.pre,
                                                                                                  w.rank);
    const size_t smem = (size_t)T * p.rt * SEL_BINS * 4;
    auto hk = T == 2 ? ga_sel_hist_kernel<2> : ga_sel_hist_kernel<1>;
    if ((e = cudaFuncSetAttribute(hk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    const dim3 grid((unsigned)p.tiles, (unsigned)p.S);
    const unsigned wgrid = grid_for(T * d * 32, 256);
    for (int shift = 56; shift >= 0; shift -= 8) {
        hk<<<grid, SEL_THREADS, smem, st>>>(src, d, N, p.rt, p.S, shift, w.pre, w.hist);
        ga_sel_scan_kernel<<<wgrid, 256, 0, st>>>(d, T, shift, w.pre, w.rank, w.hist);
    }
    if (T == 2) ga_sel_ties_kernel<2><<<grid, SEL_THREADS, 0, st>>>(src, d, N, p.rt, p.S, w.pre, w.cnt, w.first);
    else ga_sel_ties_kernel<1><<<grid, SEL_THREADS, 0, st>>>(src, d, N, p.rt, p.S, w.pre, w.cnt, w.first);
    ga_sel_index_kernel<<<wgrid, 256, 0, st>>>(src, d, N, p.S, T, w.pre, w.rank, w.cnt, w.first, w.idx, out);
    if (launches) *launches += 1 + 2 * 8 + 2;
    return cudaGetLastError();
}

}  // namespace

size_t ga_select_bytes(int64_t d, int64_t N, int sm_count) {
    return sel_layout(d, sel_plan(d, N, sm_count), nullptr, nullptr);
}

cudaError_t launch_ga_select(const double* X, int64_t d, int64_t N, int64_t ld, const double* wt, const double* n2,
                             int kind, double P, void* ws, double* out, int sm_count, cudaStream_t st,
                             int64_t* launches) {
    if (d < 1 || N < 1 || N > (int64_t)0xffffffffLL || (kind != 1 && kind != 2)) return cudaErrorInvalidValue;
    const SelPlan p = sel_plan(d, N, sm_count);
    SelWs w;
    sel_layout(d, p, ws, &w);
    const SelSrc src{X, ld, wt, n2, kind};
    if (kind == 2) {
        const int64_t t = N >= 2 ? N / 2 - 1 : 0;                          // I[end ÷ 2] (1-based)   :353
        return sel_run(src, d, N, 1, t, t, p, w, out, st, launches);
    }
    int64_t lo, hi;
    trim_range(P, N, &lo, &hi);
    if (lo >= hi) return cudaSuccess;                                      // nothing kept: the sweep gives 0 / 0
    return sel_run(src, d, N, 2, lo, hi - 1, p, w, nullptr, st, launches);
}

cudaError_t launch_ga_trimmed_sweep(const double* X, int64_t d, int64_t N, int64_t ld, const double* wt,
                                    const double* n2, double P, const void* ws, double* out, int sm_count,
                                    cudaStream_t st, int64_t* launches) {
    if (d < 1 || N < 1 || N > (int64_t)0xffffffffLL) return cudaErrorInvalidValue;
    const SelPlan p = sel_plan(d, N, sm_count);
    SelWs w;
    sel_layout(d, p, const_cast<void*>(ws), &w);
    const SelSrc src{X, ld, wt, n2, 1};
    int64_t lo, hi;
    trim_range(P, N, &lo, &hi);
    ga_sel_trim_kernel<<<dim3((unsigned)p.tiles, (unsigned)p.S), SEL_THREADS, 0, st>>>(src, d, N, p.rt, p.S, lo >= hi,
                                                                                      w.pre, w.idx, w.num, w.den);
    ga_sel_trim_finish_kernel<<<grid_for(d, 256) < 1024 ? grid_for(d, 256) : 1024, 256, 0, st>>>(d, p.S, w.num, w.den,
                                                                                                  out);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

}  // namespace tlsq
