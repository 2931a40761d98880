// syrk_tma.cu -- G = X'X for a dense, materialised tall matrix X (M x N, column-major) at FP64 tensor-core rate.
//
// This is the hot Gram pass of the ALM loop once the SVT input W_k is materialised by the previous epilogue
// (replaces LAPACK dgesdd of src/robustPCA.jl:194; also used for opnorm(D), :177).  Blackwell-native data path:
//   * TMA (cp.async.bulk.tensor.2d, SASS UTMALDG) streams 16-row x 128-column boxes of X into a 4-stage shared
//     memory ring, completion signalled on mbarriers (no register staging, 128 KB in flight per SM);
//   * the boxes land with the hardware 128-byte swizzle; together with a permuted k order inside each 16-row
//     tile (lane t takes k = 2s + (t&1) + 8(t>>1)) every 8-byte DMMA fragment load of a half-warp hits 16
//     distinct banks -- no padding, no conflicts;
//   * 8 warps in a 4 x 2 layout own a 128 x 128 output block, warp tile 32 x 64 = 32 DMMA.8x8x4 accumulators
//     (64 FP64 registers pairs) per k-step, FP64 tensor pipe (mma.sync.m8n8k4.f64; tcgen05 has no FP64 kind).
// grid.x enumerates the upper-triangular 128-blocks (bi <= bj), grid.y splits the rows; CTAs of one split stream
// the same rows at the same time so the panels shared between blocks are served by L2.  Partial blocks are
// summed in fixed order by gram_reduce (deterministic).
#include <cuda.h>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int SB = kSyrkBlk;      // 128 output block edge
constexpr int SR = 16;            // rows per TMA box (128-byte inner extent = the swizzle span)
constexpr int SRS = 32;           // rows per pipeline stage (two boxes per panel)
constexpr int SST = 3;            // pipeline stages
constexpr int BOX_BYTES = SB * SR * 8;         // 16 KB
constexpr int PANEL_BYTES = 2 * BOX_BYTES;     // 32 KB: 32 rows x 128 columns
constexpr int STAGE_BYTES = 2 * PANEL_BYTES;   // 64 KB: panel i + panel j

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

// Warp -> output tiles.  Off-diagonal block: 4 x 2 warps, warp tile 32 x 64 (32 DMMA accumulators).  Diagonal block:
// only the 10 upper 32 x 32 tiles are computed; they are cut into 40 strips of 32 x 8 columns, enumerated tile row by
// tile row, and warp w takes strips [5w, 5w + 5) -- 20 DMMAs per k-step on every warp (perfectly balanced, a diagonal
// block costs 5/8 of an off-diagonal one and gets proportionally fewer CTAs, see syrk_plan).  A warp's strips span at
// most two tile rows: the first n1 take their A fragments from tile row rowA, the others from rowB.
struct DiagStrips { int rowA, rowB, n1; int cs[5]; };
__device__ __forceinline__ DiagStrips diag_strips(int warp) {
    DiagStrips d;
    int n = 0, k = 0;
    d.rowA = d.rowB = 0; d.n1 = 0;
#pragma unroll
    for (int arow = 0; arow < 4; ++arow)
#pragma unroll
        for (int c = 4 * arow; c < 16; ++c, ++n) {
            if (n >= 5 * warp && n < 5 * warp + 5) {
                if (k == 0) d.rowA = arow;
                d.rowB = arow;
                if (arow == d.rowA) d.n1 = k + 1;
                d.cs[k++] = c;
            }
        }
    return d;
}

// the first N1 strips use a1, the others a2 (N1 is per-warp constant: the switch keeps accumulator indexing static)
template <int N1>
__device__ __forceinline__ void diag_stage(double (&acc)[4][8][2], const uint8_t* pa, uint32_t aA, uint32_t aB,
                                           const uint32_t (&bo)[5], const uint32_t (&koff)[4]) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const uint8_t* ph = pa + half * BOX_BYTES;
#pragma unroll
        for (int s4 = 0; s4 < 4; ++s4) {
            double a1[4], a2[4];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                a1[mi] = *reinterpret_cast<const double*>(ph + aA + (uint32_t)mi * 1024u + koff[s4]);
                if (N1 < 5) a2[mi] = *reinterpret_cast<const double*>(ph + aB + (uint32_t)mi * 1024u + koff[s4]);
            }
#pragma unroll
            for (int s = 0; s < 5; ++s) {
                const double b = *reinterpret_cast<const double*>(ph + bo[s] + koff[s4]);
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) dmma884(acc[mi][s][0], acc[mi][s][1], s < N1 ? a1[mi] : a2[mi], b);
            }
        }
    }
}

__global__ void __launch_bounds__(256, 1)
syrk_tma_kernel(const __grid_constant__ CUtensorMap tmap, double* __restrict__ partial,
                const __grid_constant__ SyrkPlan plan) {
    // 1024-byte alignment is required by the 128B swizzle pattern.  The pointer is NOT re-aligned with integer
    // arithmetic: that would turn every fragment load into a generic LD instead of LDS.
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    __shared__ uint64_t full_bar[SST];
    uint8_t* base = smem_dyn;
    if ((smem_u32(base) & 1023u) != 0u) __trap();

    int blk = 0;
    while (blk + 1 < plan.nblk && (int)blockIdx.x >= plan.cta_begin[blk + 1]) ++blk;
    const int split = blockIdx.x - plan.cta_begin[blk];
    const int nsplit = plan.nsplit_blk[blk];
    int bi = 0, bj = 0;
    {
        int rem = blk;
        for (bi = 0; bi < plan.nb; ++bi) {
            const int cnt = plan.nb - bi;
            if (rem < cnt) { bj = bi + rem; break; }
            rem -= cnt;
        }
    }
    const bool diag = (bi == bj);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int a0 = 32 * (warp & 3), b0 = 64 * (warp >> 2);       // off-diagonal warp tile
    const DiagStrips ds = diag_strips(warp);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < SST; ++s) mbar_init(&full_bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int nmy = (plan.ntiles - split + nsplit - 1) / nsplit;       // 32-row tiles of this CTA
    const uint32_t stage_tx = diag ? PANEL_BYTES : STAGE_BYTES;

    auto issue = [&](int i) {
        const int s = i % SST;
        const int kt = split + i * nsplit;
        uint8_t* st = base + (size_t)s * STAGE_BYTES;
        mbar_expect_tx(&full_bar[s], stage_tx);
        tma_load_2d(st, &tmap, kt * SRS, bi * SB, &full_bar[s]);
        tma_load_2d(st + BOX_BYTES, &tmap, kt * SRS + SR, bi * SB, &full_bar[s]);
        if (!diag) {
            tma_load_2d(st + PANEL_BYTES, &tmap, kt * SRS, bj * SB, &full_bar[s]);
            tma_load_2d(st + PANEL_BYTES + BOX_BYTES, &tmap, kt * SRS + SR, bj * SB, &full_bar[s]);
        }
    };
    if (tid == 0) {
        for (int i = 0; i < SST && i < nmy; ++i) issue(i);
    }

    // per-lane swizzled byte offsets of the 4 k-steps:  k = 2s + (t&1) + 8(t>>1);  chunk16 = (k>>1) ^ (col&7), col&7 == g
    uint32_t koff[4];
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
        const int k = 2 * s4 + (t & 1) + 8 * (t >> 1);
        koff[s4] = (uint32_t)((((k >> 1) ^ g) << 4) | ((k & 1) << 3));
    }
    const uint32_t a_col = (uint32_t)(a0 + g) * 128u;
    const uint32_t b_col = (uint32_t)(b0 + g) * 128u;
    const uint32_t dA = (uint32_t)(32 * ds.rowA + g) * 128u, dB = (uint32_t)(32 * ds.rowB + g) * 128u;
    uint32_t dbo[5];
#pragma unroll
    for (int s5 = 0; s5 < 5; ++s5) dbo[s5] = (uint32_t)(8 * ds.cs[s5] + g) * 128u;

    double acc[4][8][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

    for (int i = 0; i < nmy; ++i) {
        const int s = i % SST;
        const uint32_t parity = (uint32_t)((i / SST) & 1);
        mbar_wait(&full_bar[s], parity);
        const uint8_t* pa = base + (size_t)s * STAGE_BYTES;
        const uint8_t* pb = diag ? pa : pa + PANEL_BYTES;
        if (!diag) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
#pragma unroll
                for (int s4 = 0; s4 < 4; ++s4) {
                    double a[4], b[8];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
                        a[mi] = *reinterpret_cast<const double*>(pa + half * BOX_BYTES + a_col + (uint32_t)mi * 1024u + koff[s4]);
#pragma unroll
                    for (int ni = 0; ni < 8; ++ni)
                        b[ni] = *reinterpret_cast<const double*>(pb + half * BOX_BYTES + b_col + (uint32_t)ni * 1024u + koff[s4]);
#pragma unroll
                    for (int ni = 0; ni < 8; ++ni)
#pragma unroll
                        for (int mi = 0; mi < 4; ++mi) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                }
            }
        } else {
            switch (ds.n1) {
                case 1: diag_stage<1>(acc, pa, dA, dB, dbo, koff); break;
                case 2: diag_stage<2>(acc, pa, dA, dB, dbo, koff); break;
                case 3: diag_stage<3>(acc, pa, dA, dB, dbo, koff); break;
                case 4: diag_stage<4>(acc, pa, dA, dB, dbo, koff); break;
                default: diag_stage<5>(acc, pa, dA, dB, dbo, koff); break;
            }
        }
        __syncthreads();                               // every warp is done with stage s -> refill it
        if (tid == 0 && i + SST < nmy) issue(i + SST);
    }

    double* P = partial + ((size_t)plan.part_off[blk] + split) * (SB * SB);
    if (!diag) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 8; ++ni) {
                const int il = a0 + 8 * mi + g;
                const int jl = b0 + 8 * ni + 2 * t;
                P[jl * SB + il] = acc[mi][ni][0];
                P[(jl + 1) * SB + il] = acc[mi][ni][1];
            }
    } else {
#pragma unroll
        for (int s5 = 0; s5 < 5; ++s5) {
            const int ra = 32 * (s5 < ds.n1 ? ds.rowA : ds.rowB);
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int il = ra + 8 * mi + g;
                const int jl = 8 * ds.cs[s5] + 2 * t;
                P[jl * SB + il] = acc[mi][s5][0];
                P[(jl + 1) * SB + il] = acc[mi][s5][1];
            }
        }
    }
}

// G[i,j] = G[j,i] = sum over the splits of block(i,j), fixed order; diagonal blocks only hold their upper 32-tiles
__global__ void syrk_reduce_kernel(const double* __restrict__ partial, const __grid_constant__ SyrkPlan plan, int N,
                                   double* __restrict__ G) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)N * N) return;
    int i = (int)(idx % N), j = (int)(idx / N);
    if (i > j) return;
    const int bi = i / SB, bj = j / SB;
    int il = i % SB, jl = j % SB;
    if (bi == bj && (il >> 5) > (jl >> 5)) return;      // cannot happen for i <= j; kept for clarity
    const int blk = bi * plan.nb - (bi * (bi - 1)) / 2 + (bj - bi);
    const double* p = partial + (size_t)plan.part_off[blk] * (SB * SB) + jl * SB + il;
    double sum = 0.0;
    const int ns = plan.nsplit_blk[blk];
    for (int sp = 0; sp < ns; ++sp) sum += p[(size_t)sp * (SB * SB)];
    G[(int64_t)j * N + i] = sum;
    G[(int64_t)i * N + j] = sum;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}

}  // namespace

bool syrk_tma_eligible(const double* X, int64_t M, int64_t N, int64_t ld) {
    if (N < 65 || N > kEigMaxN) return false;             // small n: the generic 64-block kernel is the better fit
    if (M < 4096) return false;
    if ((ld & 1) || (reinterpret_cast<uintptr_t>(X) & 15)) return false;   // TMA: 16-byte aligned base and stride
    if (M >= (int64_t)1 << 31) return false;              // int32 TMA coordinates
    return get_encode_fn() != nullptr;
}

SyrkPlan syrk_plan(int64_t M, int64_t N, int sm_count) {
    SyrkPlan p = {};
    p.nb = (int)((N + SB - 1) / SB);
    p.nblk = p.nb * (p.nb + 1) / 2;
    p.ntiles = (int)((M + SRS - 1) / SRS);
    // CTAs per block proportional to the block's cost (off-diagonal: 32 DMMAs per warp and k-step, diagonal: 20)
    int ndiag = p.nb, noff = p.nblk - p.nb;
    double unit = (double)sm_count / (4.0 * noff + 2.5 * ndiag);
    int total = 0, blk = 0;
    for (int bi = 0; bi < p.nb; ++bi)
        for (int bj = bi; bj < p.nb; ++bj, ++blk) {
            int ns = (int)((bi == bj ? 2.5 : 4.0) * unit);
            if (ns < 1) ns = 1;
            if (ns > p.ntiles) ns = p.ntiles;
            p.nsplit_blk[blk] = ns;
            total += ns;
        }
    // hand left-over SMs to the off-diagonal blocks first (they are the longest)
    for (int pass = 0; pass < 4 && total < sm_count; ++pass) {
        blk = 0;
        for (int bi = 0; bi < p.nb && total < sm_count; ++bi)
            for (int bj = bi; bj < p.nb && total < sm_count; ++bj, ++blk)
                if (((bi != bj) == (pass % 2 == 0)) && p.nsplit_blk[blk] < p.ntiles) { ++p.nsplit_blk[blk]; ++total; }
    }
    int off = 0;
    for (blk = 0; blk < p.nblk; ++blk) {
        p.cta_begin[blk] = off;
        p.part_off[blk] = off;
        off += p.nsplit_blk[blk];
    }
    p.cta_begin[p.nblk] = off;
    p.ncta = off;
    p.nsplit = p.nsplit_blk[0];
    p.partial_bytes = (size_t)off * SB * SB * sizeof(double);
    return p;
}

cudaError_t launch_syrk_tma(const double* X, int64_t M, int64_t N, int64_t ld, const SyrkPlan& plan, double* partial,
                            double* G, cudaStream_t st, int64_t* launches) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    CUtensorMap map;
    const cuuint64_t gdim[2] = {(cuuint64_t)M, (cuuint64_t)N};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * 8};
    const cuuint32_t box[2] = {(cuuint32_t)SR, (cuuint32_t)SB};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(X), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    const size_t smem = (size_t)SST * STAGE_BYTES;
    // function attributes are per device: set on every launch (a process may run on several GPUs)
    cudaError_t e = cudaFuncSetAttribute(syrk_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    syrk_tma_kernel<<<plan.ncta, 256, smem, st>>>(map, partial, plan);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int64_t nn = N * N;
    syrk_reduce_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, st>>>(partial, plan, (int)N, G);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

}  // namespace tlsq
