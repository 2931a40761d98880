// gemm.cu -- C (M x N) = X (M x K) * B (K x N) for a tall X and small K, N (<= 512): the left singular vectors
// U = W V diag(1/s) of the SVD that rpca returns (src/robustPCA.jl:194,238).  FP64 tensor cores (DMMA.8x8x4),
// 128 x 128 output tile per CTA (8 warps, warp tile 32 x 64), K streamed in 16-wide chunks through a double-buffered
// cp.async pipeline into padded shared memory:
//   Xs[k][132]  (row stride 132: the A fragment (m = g, k = t) of a half-warp hits 16 distinct 8-byte banks)
//   Bs[n][20]   (k contiguous, stride 20: same property for the B fragment (k = t, n = g))
#include "kernels.h"

namespace tlsq {

namespace {

constexpr int GT = 128;          // output tile edge
constexpr int GK = 16;           // K chunk
constexpr int XRS = GT + 4;      // 132
constexpr int BKS = GK + 4;      // 20

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool pred) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    const int sz = pred ? 16 : 0;                       // src-size 0 -> zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(256, 1)
gemm_xb_kernel(const double* __restrict__ X, int64_t M, int K, int64_t ldx, const double* __restrict__ B, int N,
               double* __restrict__ C) {
    extern __shared__ double smg[];
    double* Xs = smg;                                   // 2 x [GK][XRS]
    double* Bs = smg + 2 * GK * XRS;                    // 2 x [GT][BKS]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wi = warp & 3, wj = warp >> 2;            // warp tile rows [32wi,+32), cols [64wj,+64)
    const int64_t row0 = (int64_t)blockIdx.x * GT;
    const int col0 = blockIdx.y * GT;

    auto load_chunk = [&](int kc, int buf) {
        // X chunk: GK columns (k) x 128 rows -> 16 x 64 sixteen-byte pieces; 4 per thread
        double* xs = Xs + buf * GK * XRS;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int piece = tid + 256 * q;            // 0..1023
            const int k = piece >> 6, r2 = (piece & 63) * 2;
            const int kk = kc * GK + k;
            const bool ok = (kk < K) && (row0 + r2 + 1 < M + 1) && (row0 + r2 < M);
            const double* src = X + (int64_t)(kk < K ? kk : 0) * ldx + (row0 + r2 < M ? row0 + r2 : 0);
            cp_async16(xs + k * XRS + r2, src, ok);
        }
        // B chunk: 128 columns (n) x GK k -> 128 x 8 pieces; 4 per thread
        double* bs = Bs + buf * GT * BKS;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int piece = tid + 256 * q;
            const int nn = piece >> 3, k2 = (piece & 7) * 2;
            const int ncol = col0 + nn, kk = kc * GK + k2;
            const bool ok = (ncol < N) && (kk < K);
            const double* src = B + (int64_t)(ncol < N ? ncol : 0) * K + (kk < K ? kk : 0);
            cp_async16(bs + nn * BKS + k2, src, ok);
        }
        cp_async_commit();
    };

    double acc[4][8][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

    const int nchunks = (K + GK - 1) / GK;
    load_chunk(0, 0);
    for (int kc = 0; kc < nchunks; ++kc) {
        const int buf = kc & 1;
        if (kc + 1 < nchunks) { load_chunk(kc + 1, buf ^ 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
        const double* xs = Xs + buf * GK * XRS;
        const double* bs = Bs + buf * GT * BKS;
#pragma unroll
        for (int k0 = 0; k0 < GK; k0 += 4) {
            double a[4], b[8];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) a[mi] = xs[(k0 + t) * XRS + 32 * wi + 8 * mi + g];
#pragma unroll
            for (int ni = 0; ni < 8; ++ni) b[ni] = bs[(64 * wj + 8 * ni + g) * BKS + k0 + t];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 8; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) {
            const int64_t r = row0 + 32 * wi + 8 * mi + g;
            const int c = col0 + 64 * wj + 8 * ni + 2 * t;
            if (r < M) {
                if (c < N) C[(int64_t)c * M + r] = acc[mi][ni][0];
                if (c + 1 < N) C[(int64_t)(c + 1) * M + r] = acc[mi][ni][1];
            }
        }
}

// any shape / alignment: 32 x 32 output tile, K in 32-wide chunks through shared memory, plain FP64 FMA
__global__ void __launch_bounds__(256)
gemm_plain_kernel(const double* __restrict__ X, int64_t M, int K, int64_t ldx, const double* __restrict__ B, int N,
                  double* __restrict__ C) {
    __shared__ double Xs[32][33];      // [k][row]
    __shared__ double Bs[32][33];      // [col][k]
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * 32;
    const int c0 = blockIdx.y * 32;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int kk = ty + 8 * q;
            Xs[kk][tx] = (r0 + tx < M && k0 + kk < K) ? X[(int64_t)(k0 + kk) * ldx + r0 + tx] : 0.0;
            Bs[kk][tx] = (c0 + kk < N && k0 + tx < K) ? B[(int64_t)(c0 + kk) * K + k0 + tx] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int cc = ty + 8 * q;
            double a = acc[q];
#pragma unroll
            for (int kk = 0; kk < 32; ++kk) a = fma(Xs[kk][tx], Bs[cc][kk], a);
            acc[q] = a;
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int cc = c0 + ty + 8 * q;
        if (r0 + tx < M && cc < N) C[(int64_t)cc * M + r0 + tx] = acc[q];
    }
}

__global__ void scale_cols_inv_kernel(const double* __restrict__ V, const double* __restrict__ sigma, int n,
                                      double* __restrict__ B) {
    const int c = blockIdx.x;
    const double s = sigma[c];
    const double f = s > 0.0 ? 1.0 / s : 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) B[(int64_t)c * n + i] = V[(int64_t)c * n + i] * f;
}

}  // namespace

bool gemm_xb_eligible(const double* X, int64_t M, int K, int64_t ldx, int N) {
    // 16-byte cp.async pieces: even leading dimension / row count, aligned bases, even K
    return M >= 1024 && !(ldx & 1) && !(M & 1) && !(K & 1) && !(reinterpret_cast<uintptr_t>(X) & 15) && N >= 1;
}

cudaError_t launch_gemm_xb(const double* X, int64_t M, int K, int64_t ldx, const double* B, int N, double* C,
                           cudaStream_t st, int64_t* launches) {
    const size_t smem = (size_t)(2 * GK * XRS + 2 * GT * BKS) * sizeof(double);     // 33792 + 40960 = 74752 B
    // function attributes are per device: set on every launch (a process may run on several GPUs)
    cudaError_t e = cudaFuncSetAttribute(gemm_xb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid((unsigned)((M + GT - 1) / GT), (unsigned)((N + GT - 1) / GT));
    gemm_xb_kernel<<<grid, 256, smem, st>>>(X, M, K, ldx, B, N, C);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_gemm_any(const double* X, int64_t M, int K, int64_t ldx, const double* B, int N, double* C,
                            cudaStream_t st, int64_t* launches) {
    if (gemm_xb_eligible(X, M, K, ldx, N) && !(reinterpret_cast<uintptr_t>(B) & 15))
        return launch_gemm_xb(X, M, K, ldx, B, N, C, st, launches);
    dim3 grid((unsigned)((M + 31) / 32), (unsigned)((N + 31) / 32));
    gemm_plain_kernel<<<grid, 256, 0, st>>>(X, M, K, ldx, B, N, C);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_scale_cols_inv(const double* V, const double* sigma, int n, double* B, cudaStream_t st,
                                  int64_t* launches) {
    scale_cols_inv_kernel<<<n, 128, 0, st>>>(V, sigma, n, B);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

}  // namespace tlsq
