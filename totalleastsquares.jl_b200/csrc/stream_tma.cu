// stream_tma.cu -- TMA-staged form of the two streaming kernels of the ALM epilogue (factored iterate, svp <= 32):
//
//   tproj_tma_kernel   T_k = (W_k V_r) .* f                      one read of the materialised SVT input W_k
//   alm_ew_tma_kernel  E_k, A_k = clamp(T_k V_k'), Z, Y_k, ||Z||_F^2, W_{k+1}       src/robustPCA.jl:188-192, 205-222
//                      one read of D and Y_{k-1}, one write of Y_k and W_{k+1}
//
// Same per-element arithmetic and operation order as alm_stream_kernel (stream.cu); what changes is the data path.  The
// register-prefetch version is bound by load latency (ncu: 38 % of the stall samples sit on the first DFMA that
// consumes a global load, 24 % warps active at 122 registers) and reaches 4.2 - 4.8 TB/s.  Here every CTA streams
// 32 KB stages of 256-row x 4-column boxes through a ring of up to 6 shared-memory buffers filled by TMA
// (cp.async.bulk.tensor.2d, completion on mbarriers) without a single register or warp spent on it, the threads only
// ever wait on shared memory.  Each thread owns two rows, so every shared-memory load of a V row feeds two elements;
// the inner loops are branch-free (out-of-range rows arrive zero-filled, only the stores are predicated).
#include <cuda.h>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int TRB = 256;     // rows per TMA box
constexpr int TT = 512;      // rows per tile of the element-wise pass; threads per CTA of the projection
constexpr int TS = 6;        // ring stages (the launcher uses as many as fit beside the V blocks)
constexpr int TC2 = 4;       // columns per stage, element-wise pass (stage = D + Y = 32 KB)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}

template <int RP>
__device__ __forceinline__ double dot_rp(const double (&t)[RP], const double* __restrict__ v) {
    double a0 = 0.0, a1 = 0.0;                     // two chains: half the dependent-FMA latency per element
#pragma unroll
    for (int c = 0; c < RP; c += 2) {
        const double2 vv = *reinterpret_cast<const double2*>(v + c);
        a0 = fma(t[c], vv.x, a0);
        a1 = fma(t[c + 1], vv.y, a1);
    }
    return a0 + a1;
}

// one stage = TC columns x TT rows of one matrix: two boxes of TRB rows
template <int TC>
__device__ __forceinline__ void load_stage(double* dst, const CUtensorMap* map, int row0, int col0, uint64_t* bar) {
    tma_load_2d(dst, map, row0, col0, bar);
    tma_load_2d(dst + TC * TRB, map, row0 + TRB, col0, bar);
}
// element (row r of the tile, column u of the stage)
template <int TC>
__device__ __forceinline__ double stage_at(const double* st, int r, int u) {
    return st[(r >> 8) * (TC * TRB) + u * TRB + (r & (TRB - 1))];
}

// ---------------------------------------------------------------------------------------------------------------------
// T[row, :] = f .* (W[row, :] V_r)          (tiles are dealt round-robin: a tile's sum stays in one CTA).
// Every thread owns TWO rows (tid and tid + 512 of a 1024-row tile): the row of V it reads from shared memory (a
// broadcast LDS.128 per two ranks) is used twice -- the one-row version was bound by the LDS issue rate (ncu: 46 % mio).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int PR = 2;                     // rows per thread
constexpr int TT1 = PR * TT;              // rows per tile of the projection kernel
constexpr int TC1 = 4;                    // columns per stage: 4 x 1024 x 8 B = 32 KB

template <int RP>
__global__ void __launch_bounds__(TT, 1)
tproj_tma_kernel(const __grid_constant__ CUtensorMap mW, const EpiArgs a, int svp_host, const int* __restrict__ svp_dev,
                 int ntiles, int nstage) {
    const int svp = svp_dev ? __ldg(svp_dev) : svp_host;
    if (svp > RP) return;                           // rank guess too small: nothing is touched (solver.cu relaunches)
    extern __shared__ __align__(1024) uint8_t smraw[];
    __shared__ uint64_t full[TS];
    __shared__ double fsm[RP];
    constexpr int STG = TC1 * TT1;                             // doubles per stage: [PR * 2 boxes][TC1][TRB]
    double* stage = reinterpret_cast<double*>(smraw);          // [nstage][STG]
    double* Vsm = stage + nstage * STG;                        // [N][RP]
    const int N = (int)a.N;
    const int tid = threadIdx.x;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < TS; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < RP) fsm[tid] = tid < svp ? __ldg(a.fvec + tid) : 0.0;
    for (int idx = tid; idx < N * RP; idx += TT) {
        const int j = idx % N, c = idx / N;
        Vsm[j * RP + c] = c < svp ? __ldg(a.Vs + (int64_t)c * N + j) : 0.0;
    }
    __syncthreads();
    const int nch = N / TC1;                                   // N % 8 == 0 (eligibility)
    const int my_tiles = ((int)blockIdx.x < ntiles) ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int total = my_tiles * nch;
    auto issue = [&](int q, int s) {
        const int tile = (int)blockIdx.x + (q / nch) * (int)gridDim.x;
        double* st = stage + s * STG;
        mbar_expect_tx(&full[s], STG * 8);
#pragma unroll
        for (int bx = 0; bx < TT1 / TRB; ++bx)
            tma_load_2d(st + bx * (TC1 * TRB), &mW, tile * TT1 + bx * TRB, (q % nch) * TC1, &full[s]);
    };
    if (tid == 0)
        for (int q = 0; q < nstage && q < total; ++q) issue(q, q);
    double tr[PR][RP];
    int s = 0;
    uint32_t phase = 0;
    for (int q = 0; q < total; ++q) {
        const int ch = q % nch;
        if (ch == 0) {
#pragma unroll
            for (int p = 0; p < PR; ++p)
#pragma unroll
                for (int c = 0; c < RP; ++c) tr[p][c] = 0.0;
        }
        mbar_wait(&full[s], phase);
        double w[PR][TC1];
#pragma unroll
        for (int p = 0; p < PR; ++p)
#pragma unroll
            for (int u = 0; u < TC1; ++u) w[p][u] = stage_at<TC1>(stage + s * STG, tid + p * TT, u);
#pragma unroll
        for (int u = 0; u < TC1; ++u) {
            const double* v = Vsm + (ch * TC1 + u) * RP;
#pragma unroll
            for (int c = 0; c < RP; c += 2) {
                const double2 vv = *reinterpret_cast<const double2*>(v + c);
#pragma unroll
                for (int p = 0; p < PR; ++p) {
                    tr[p][c] = fma(w[p][u], vv.x, tr[p][c]);
                    tr[p][c + 1] = fma(w[p][u], vv.y, tr[p][c + 1]);
                }
            }
        }
        if (ch == nch - 1) {
            const int64_t row0 = (int64_t)((int)blockIdx.x + (q / nch) * (int)gridDim.x) * TT1 + tid;
#pragma unroll
            for (int p = 0; p < PR; ++p) {
                const int64_t row = row0 + p * TT;
                if (row < a.M) {
#pragma unroll
                    for (int c = 0; c < RP; ++c) a.Tn[(int64_t)c * a.M + row] = tr[p][c] * fsm[c];
                }
            }
        }
        // Refill the stage only AFTER every value read from it has been consumed by an FMA: a shared-memory load that is
        // still in flight when its thread reaches the barrier is not ordered against the TMA (async-proxy) write that
        // thread 0 issues behind the barrier -- refilling right after the register copy produced sporadic stale / early
        // data (non-deterministic results, caught by the repeat test in tests/test_gpu_scale.py).
        __syncthreads();
        if (tid == 0 && q + nstage < total) issue(q + nstage, s);
        if (++s == nstage) { s = 0; phase ^= 1u; }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// element-wise pass with both iterates factored (A_{k-1} = clamp(T_{k-1} V_{k-1}'), A_k = clamp(T_k V_k')).
// Work unit = (tile, 4-column stage); the units are split evenly over the CTAs (a CTA may start in the middle of a tile).
// Every thread owns TWO rows (tid and tid + EWT of a 2 EWT-row tile), so each broadcast LDS.128 of a V row feeds two
// elements: the one-row form spent 14 of its ~75 instructions per element on those loads.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int EWT = 256;                  // threads per CTA of the element-wise pass
static_assert(PR * EWT == TT, "the element-wise tile is TT rows");

// dot_rp for the two rows of a thread: the same two FMA chains and final add per row, one load of each V pair
template <int RP>
__device__ __forceinline__ void dot_rp2(const double (&t)[PR][RP], const double* __restrict__ v, double (&r)[PR]) {
    double a0[PR], a1[PR];
#pragma unroll
    for (int p = 0; p < PR; ++p) a0[p] = a1[p] = 0.0;
#pragma unroll
    for (int c = 0; c < RP; c += 2) {
        const double2 vv = *reinterpret_cast<const double2*>(v + c);
#pragma unroll
        for (int p = 0; p < PR; ++p) {
            a0[p] = fma(t[p][c], vv.x, a0[p]);
            a1[p] = fma(t[p][c + 1], vv.y, a1[p]);
        }
    }
#pragma unroll
    for (int p = 0; p < PR; ++p) r[p] = a0[p] + a1[p];
}

template <int RP, bool HANKEL>
__global__ void __launch_bounds__(EWT, 1)
alm_ew_tma_kernel(const __grid_constant__ CUtensorMap mD, const __grid_constant__ CUtensorMap mY, const EpiArgs a,
                  int svp_host, const int* __restrict__ svp_dev, int ntiles, int nstage) {
    const int svp = svp_dev ? __ldg(svp_dev) : svp_host;
    if (svp > RP) return;
    extern __shared__ __align__(1024) uint8_t smraw[];
    __shared__ uint64_t full[TS];
    __shared__ double red[TT / 32];
    constexpr int HALF = TC2 * TT;                             // doubles of one matrix per stage
    constexpr int STG = 2 * HALF;                              // D boxes, then Y boxes
    double* stage = reinterpret_cast<double*>(smraw);          // [nstage][STG]
    const int N = (int)a.N;
    double* Vsm = stage + nstage * STG;                        // [N][RP]  V_k
    double* Vpm = Vsm + (size_t)N * RP;                        // [N][RP]  V_{k-1}
    const int tid = threadIdx.x;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < TS; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int idx = tid; idx < N * RP; idx += EWT) {
        const int j = idx % N, c = idx / N;
        Vsm[j * RP + c] = c < svp ? __ldg(a.Vs + (int64_t)c * N + j) : 0.0;
        Vpm[j * RP + c] = c < a.svp_prev ? __ldg(a.Vp + (int64_t)c * N + j) : 0.0;
    }
    __syncthreads();
    const int nch = N / TC2;                                   // N % TC2 == 0 (eligibility)
    const int64_t units = (int64_t)ntiles * nch;
    const int64_t g0 = units * (int64_t)blockIdx.x / (int64_t)gridDim.x;
    const int64_t g1 = units * ((int64_t)blockIdx.x + 1) / (int64_t)gridDim.x;
    const int total = (int)(g1 - g0);
    constexpr uint32_t tx = (HANKEL ? 1u : 2u) * HALF * 8u;
    auto issue = [&](int q, int s) {
        const int64_t g = g0 + q;
        const int tile = (int)(g / nch), ch = (int)(g % nch);
        double* st = stage + s * STG;
        mbar_expect_tx(&full[s], tx);
        if (!HANKEL) load_stage<TC2>(st, &mD, tile * TT, ch * TC2, &full[s]);
        load_stage<TC2>(st + HALF, &mY, tile * TT, ch * TC2, &full[s]);
    };
    if (tid == 0)
        for (int q = 0; q < nstage && q < total; ++q) issue(q, q);
    double tr[PR][RP], tp[PR][RP];
    double zz[PR] = {};                                        // per row: the grouping of the one-row-per-thread form
    int64_t row[PR];
    bool rowok[PR];
    int s = 0;
    uint32_t phase = 0;
    int tile = (int)(g0 / nch), ch = (int)(g0 % nch);
    for (int q = 0; q < total; ++q) {
        if (q == 0 || ch == 0) {
#pragma unroll
            for (int p = 0; p < PR; ++p) {
                row[p] = (int64_t)tile * TT + tid + p * EWT;
                rowok[p] = row[p] < a.M;
#pragma unroll
                for (int c = 0; c < RP; ++c) {
                    tr[p][c] = (rowok[p] && c < svp) ? __ldg(a.Tn + (int64_t)c * a.M + row[p]) : 0.0;
                    tp[p][c] = (rowok[p] && c < a.svp_prev) ? __ldg(a.Tp + (int64_t)c * a.M + row[p]) : 0.0;
                }
            }
        }
        const int j0 = ch * TC2;
        double dv[PR][TC2], yv[PR][TC2];
        if (HANKEL) {
#pragma unroll
            for (int p = 0; p < PR; ++p)
#pragma unroll
                for (int u = 0; u < TC2; ++u) dv[p][u] = rowok[p] ? src_at<true>(a.D, row[p], j0 + u) : 0.0;
        }
        mbar_wait(&full[s], phase);
        const double* st = stage + s * STG;
#pragma unroll
        for (int p = 0; p < PR; ++p)
#pragma unroll
            for (int u = 0; u < TC2; ++u) {
                if (!HANKEL) dv[p][u] = stage_at<TC2>(st, tid + p * EWT, u);
                yv[p][u] = stage_at<TC2>(st + HALF, tid + p * EWT, u);
            }
        double yn[PR][TC2], w2[PR][TC2], zv[PR][TC2], ev[PR][TC2];
#pragma unroll
        for (int u = 0; u < TC2; ++u) {
            const int j = j0 + u;
            double an[PR], ap[PR];
            dot_rp2<RP>(tr, Vsm + j * RP, an);
            dot_rp2<RP>(tp, Vpm + j * RP, ap);                                       // A_{k-1} from its factors
#pragma unroll
            for (int p = 0; p < PR; ++p) {
                if (a.nonnegA) {                                                      // A .= max.(A, 0)   :218
                    an[p] = (__double_as_longlong(an[p]) > 0) ? an[p] : 0.0;
                    ap[p] = (__double_as_longlong(ap[p]) > 0) ? ap[p] : 0.0;
                }
                const double d = dv[p][u], yp = yv[p][u];
                double e, w;
                alm_ew(d, ap[p], yp, a.im, a.eps, a.nonnegE, e, w);
                const double z = __dsub_rn(__dsub_rn(d, an[p]), e);                   // @. Z = D - A - E  :221
                yn[p][u] = __dadd_rn(yp, __dmul_rn(a.mu, z));                         // @. Y = Y + mu*Z   :222
                zz[p] = fma(z, z, zz[p]);                                             // (rows beyond M are all-zero)
                zv[p][u] = z;
                ev[p][u] = e;
                double e2;
                alm_ew(d, an[p], yn[p][u], a.im_next, a.eps_next, a.nonnegE, e2, w2[p][u]);   // SVT input of k+1
            }
        }
#pragma unroll
        for (int p = 0; p < PR; ++p) {
            if (rowok[p]) {
#pragma unroll
                for (int u = 0; u < TC2; ++u) {
                    const int64_t off = (int64_t)(j0 + u) * a.ldw + row[p];
                    a.Yn[off] = yn[p][u];
                    a.Wn[off] = w2[p][u];
                    if (a.Eout) a.Eout[off] = ev[p][u];
                    if (a.Zout) a.Zout[off] = zv[p][u];
                }
            }
        }
        // refill only after the values read from the stage have been consumed (see tproj_tma_kernel)
        __syncthreads();
        if (tid == 0 && q + nstage < total) issue(q + nstage, s);
        if (++s == nstage) { s = 0; phase ^= 1u; }
        if (++ch == nch) { ch = 0; ++tile; }
    }
    // rows tid + p * EWT: warp w's sums of p = 0 and 1 are those of rows [32 w, +32) and [EWT + 32 w, +32)
#pragma unroll
    for (int p = 0; p < PR; ++p) {
        const double v = warp_sum(zz[p]);
        if ((tid & 31) == 0) red[p * (EWT / 32) + (tid >> 5)] = v;
    }
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < TT / 32; ++w8) t += red[w8];
        atomicAdd(a.zz, t);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* q = nullptr;
        cudaDriverEntryPointQueryResult r;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &r) == cudaSuccess &&
            r == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(q);
        else
            cudaGetLastError();
    }
    return fn;
}
bool encode_box(CUtensorMap* map, const double* base, int64_t rows, int64_t cols, int64_t ld, int box_cols) {
    const cuuint64_t gdim[2] = {(cuuint64_t)rows, (cuuint64_t)cols};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * 8};
    const cuuint32_t box[2] = {(cuuint32_t)TRB, (cuuint32_t)box_cols};
    const cuuint32_t estr[2] = {1, 1};
    return encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <int RP>
cudaError_t launch_rp(const EpiArgs& a, const double* W, int svp, const int* svp_dev, bool hankel, int sm_count,
                      cudaStream_t st) {
    CUtensorMap mW, mD, mY;
    if (!encode_box(&mW, W, a.M, a.N, a.ldw, TC1) || !encode_box(&mY, a.Yp, a.M, a.N, a.ldw, TC2))
        return cudaErrorInvalidValue;
    if (hankel) mD = mY;
    else if (!encode_box(&mD, a.D.p, a.M, a.N, a.D.ld, TC2)) return cudaErrorInvalidValue;
    const int ntiles = (int)((a.M + TT - 1) / TT);
    const int ntiles1 = (int)((a.M + TT1 - 1) / TT1);
    const size_t stage_bytes = (size_t)TC1 * TT1 * 8;                      // == 2 * TC2 * TT * 8 == 32 KB
    const size_t v1 = (size_t)a.N * RP * 8, v2 = 2 * v1;
    int ns1 = TS, ns2 = TS;
    while (ns1 > 2 && ns1 * stage_bytes + v1 > (size_t)220 * 1024) --ns1;
    while (ns2 > 2 && ns2 * stage_bytes + v2 > (size_t)220 * 1024) --ns2;
    const size_t sm1 = ns1 * stage_bytes + v1, sm2 = ns2 * stage_bytes + v2;
    int grid = sm_count < ntiles1 ? sm_count : ntiles1;
    cudaError_t e;
    {
        auto kern = tproj_tma_kernel<RP>;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1)) != cudaSuccess) return e;
        kern<<<grid, TT, sm1, st>>>(mW, a, svp, svp_dev, ntiles1, ns1);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (hankel) {
        auto kern = alm_ew_tma_kernel<RP, true>;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2)) != cudaSuccess) return e;
        kern<<<sm_count, EWT, sm2, st>>>(mD, mY, a, svp, svp_dev, ntiles, ns2);
    } else {
        auto kern = alm_ew_tma_kernel<RP, false>;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2)) != cudaSuccess) return e;
        kern<<<sm_count, EWT, sm2, st>>>(mD, mY, a, svp, svp_dev, ntiles, ns2);
    }
    return cudaGetLastError();
}

}  // namespace

// Can the TMA-staged pair replace the register-prefetch kernels for this launch?  (factored iterate, all columns in one
// launch, 16-byte aligned bases and strides, both V blocks + the ring within shared memory)
bool stream_tma_eligible(const EpiArgs& a, const double* W, int rp, bool hankel) {
    if (rp < 4 || rp > 12 || !a.Tn || !a.Tp || !a.Wn || a.c1 > 0) return false;   // rp > 12: > 128 registers at 512 threads
    if (a.M < 16384 || a.N < 8 || (a.N & 7) || (a.ldw & 1) || !aligned16(W) || !aligned16(a.Yp)) return false;
    if (!hankel && ((a.D.ld & 1) || !aligned16(a.D.p))) return false;
    if (a.M >= (int64_t)1 << 31) return false;
    if ((size_t)2 * 32768 + (size_t)2 * a.N * rp * 8 > (size_t)216 * 1024) return false;      // >= 2 stages + V blocks
    return encode_fn() != nullptr;
}

cudaError_t launch_stream_tma(const EpiArgs& a, const double* W, int rp, int svp, const int* svp_dev, bool hankel,
                              int sm_count, cudaStream_t st) {
    switch (rp) {
        case 4:  return launch_rp<4>(a, W, svp, svp_dev, hankel, sm_count, st);
        case 8:  return launch_rp<8>(a, W, svp, svp_dev, hankel, sm_count, st);
        default: return launch_rp<12>(a, W, svp, svp_dev, hankel, sm_count, st);
    }
}

}  // namespace tlsq
