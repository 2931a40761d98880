// syrk_tma.cu -- G = X'X for a dense, materialised tall matrix X (M x N, column-major) at FP64 tensor-core rate.
//
// This is the hot Gram pass of the ALM loop once the SVT input W_k is materialised by the previous epilogue
// (replaces LAPACK dgesdd of src/robustPCA.jl:194; also used for opnorm(D), :177).  Blackwell-native data path:
//   * TMA (cp.async.bulk.tensor.2d, SASS UTMALDG) streams 16-row x 128-column boxes of X into a 6-stage shared
//     memory ring, completion signalled on mbarriers (no register staging, 192 KB of ring per SM); each warp releases
//     a stage on a second mbarrier when it is done with it, and no CTA-wide barrier paces the warps;
//   * the boxes land with the hardware 128-byte swizzle; together with a permuted k order inside each 16-row
//     tile (lane t takes k = 2s + (t&1) + 8(t>>1)) every 8-byte DMMA fragment load of a half-warp hits 16
//     distinct banks -- no padding, no conflicts;
//   * 8 compute warps in a 4 x 2 layout own a 128 x 128 output block, warp tile 32 x 64 = 32 DMMA.8x8x4 accumulators
//     (64 FP64 registers pairs) per k-step, FP64 tensor pipe (mma.sync.m8n8k4.f64; tcgen05 has no FP64 kind).
// grid.x enumerates the upper-triangular 128-blocks (bi <= bj), grid.y splits the rows; CTAs of one split stream
// the same rows at the same time so the panels shared between blocks are served by L2.  Partial blocks are
// summed in fixed order by gram_reduce (deterministic).
#include <cuda.h>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int SB = kSyrkBlk;      // 128 output block edge
constexpr int SR = 16;            // rows per TMA box (128-byte inner extent = the swizzle span) and per ring stage
constexpr int SRS = 32;           // rows per tile: the unit the row splits are dealt in
constexpr int SST = 6;            // ring stages (three tiles)
constexpr int BOX_BYTES = SB * SR * 8;         // 16 KB
constexpr int STAGE_BYTES = 2 * BOX_BYTES;     // 32 KB: box of panel i + box of panel j (diagonal blocks: panel i only)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// only the 8 x 8 tiles on or above the diagonal are computed -- the 6 upper off-diagonal 32 x 32 tiles in full and the
// upper triangles (1 + 2 + 3 + 4 tiles) of the 4 diagonal ones, 136 tiles.  They are enumerated by 32-row tile row,
// then 8-column strip, then row inside the strip, and warp w takes tiles [17w, 17w + 17): 17 DMMAs per k-step on every
// warp.  Both operands of a diagonal block come from the same panel, so a tile (r8, c8) reads fragments r8 and c8 of it.
constexpr int DT = 17;                                    // 8 x 8 tiles per warp in a diagonal block
struct DiagMap { int r8[DT], c8[DT]; uint32_t frags; };   // frags: bit f = fragment f is read by this warp
__host__ __device__ constexpr DiagMap diag_map(int warp) {
    DiagMap m{};
    int n = 0;
    for (int arow = 0; arow < 4; ++arow)
        for (int c = 4 * arow; c < 16; ++c) {
            const int h = (c >> 2) == arow ? (c & 3) + 1 : 4;     // rows of the strip on or above the diagonal
            for (int mi = 0; mi < h; ++mi, ++n)
                if (n >= DT * warp && n < DT * warp + DT) {
                    m.r8[n - DT * warp] = 4 * arow + mi;
                    m.c8[n - DT * warp] = c;
                    m.frags |= (1u << (4 * arow + mi)) | (1u << c);
                }
        }
    return m;
}
static_assert(diag_map(7).c8[DT - 1] == 15 && diag_map(7).r8[DT - 1] == 15, "136 tiles over 8 warps");

template <int W>
__device__ __forceinline__ void diag_stage(double (&acc)[4][8][2], const uint8_t* pa, uint32_t fcol,
                                           const uint32_t (&koff)[4]) {
    constexpr DiagMap m = diag_map(W);
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
        double f[16];
#pragma unroll
        for (int q = 0; q < 16; ++q)
            if ((m.frags >> q) & 1u) f[q] = *reinterpret_cast<const double*>(pa + fcol + (uint32_t)q * 1024u + koff[s4]);
#pragma unroll
        for (int k = 0; k < DT; ++k) dmma884(acc[k >> 3][k & 7][0], acc[k >> 3][k & 7][1], f[m.r8[k]], f[m.c8[k]]);
    }
}

template <int W>
__device__ __forceinline__ void diag_store(const double (&acc)[4][8][2], double* P, int g, int t) {
    constexpr DiagMap m = diag_map(W);
#pragma unroll
    for (int k = 0; k < DT; ++k) {
        const int il = 8 * m.r8[k] + g, jl = 8 * m.c8[k] + 2 * t;
        P[jl * SB + il] = acc[k >> 3][k & 7][0];
        P[(jl + 1) * SB + il] = acc[k >> 3][k & 7][1];
    }
}

// A stage is refilled once all 8 warps have arrived on its "empty" mbarrier, and a warp arrives only after its last
// fragment read from the stage has gone into a DMMA (the fragments are register operands of the asm DMMAs, which stay
// ahead of the asm arrive): an LDS still in flight is not ordered against the TMA engine's write of the refill (see
// DESIGN §4).  Thread 0 refills one stage late -- after consuming stage i it waits for stage i - 1 to be released,
// which the other warps have normally done by then -- and the other warps never wait for each other.  A dedicated
// producer warp would cap the registers at 168 (three warps on one SM sub-partition) and spill the accumulators.
constexpr int SWARPS = 8;

__global__ void __launch_bounds__(32 * SWARPS, 1)
syrk_tma_kernel(const __grid_constant__ CUtensorMap tmap, double* __restrict__ partial,
                const __grid_constant__ SyrkPlan plan) {
    // 1024-byte alignment is required by the 128B swizzle pattern.  The pointer is NOT re-aligned with integer
    // arithmetic: that would turn every fragment load into a generic LD instead of LDS.
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    __shared__ uint64_t full_bar[SST], empty_bar[SST];
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

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < SST; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], SWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // stage i = rows [16 (i & 1), +16) of this CTA's (i >> 1)-th 32-row tile
    const int nst = 2 * ((plan.ntiles - split + nsplit - 1) / nsplit);
    const uint32_t stage_tx = diag ? BOX_BYTES : STAGE_BYTES;
    auto issue = [&](int i) {
        const int s = i % SST;
        const int row = (split + (i >> 1) * nsplit) * SRS + (i & 1) * SR;
        uint8_t* st = base + (size_t)s * STAGE_BYTES;
        mbar_expect_tx(&full_bar[s], stage_tx);
        tma_load_2d(st, &tmap, row, bi * SB, &full_bar[s]);
        if (!diag) tma_load_2d(st + BOX_BYTES, &tmap, row, bj * SB, &full_bar[s]);
    };
    if (tid == 0)
        for (int i = 0; i < SST && i < nst; ++i) issue(i);

    const int a0 = 32 * (warp & 3), b0 = 64 * (warp >> 2);       // off-diagonal warp tile
    // per-lane swizzled byte offsets of the 4 k-steps:  k = 2s + (t&1) + 8(t>>1);  chunk16 = (k>>1) ^ (col&7), col&7 == g
    uint32_t koff[4];
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
        const int k = 2 * s4 + (t & 1) + 8 * (t >> 1);
        koff[s4] = (uint32_t)((((k >> 1) ^ g) << 4) | ((k & 1) << 3));
    }
    const uint32_t a_col = (uint32_t)(a0 + g) * 128u;
    const uint32_t b_col = (uint32_t)(b0 + g) * 128u;
    const uint32_t f_col = (uint32_t)g * 128u;

    double acc[4][8][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 8; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

    for (int i = 0; i < nst; ++i) {
        const int s = i % SST;
        mbar_wait(&full_bar[s], (uint32_t)((i / SST) & 1));
        const uint8_t* pa = base + (size_t)s * STAGE_BYTES;
        if (!diag) {
            const uint8_t* pb = pa + BOX_BYTES;
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) {
                double a[4], b[8];
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
                    a[mi] = *reinterpret_cast<const double*>(pa + a_col + (uint32_t)mi * 1024u + koff[s4]);
#pragma unroll
                for (int ni = 0; ni < 8; ++ni)
                    b[ni] = *reinterpret_cast<const double*>(pb + b_col + (uint32_t)ni * 1024u + koff[s4]);
#pragma unroll
                for (int ni = 0; ni < 8; ++ni)
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
            }
        } else {
            switch (warp) {
                case 0: diag_stage<0>(acc, pa, f_col, koff); break;
                case 1: diag_stage<1>(acc, pa, f_col, koff); break;
                case 2: diag_stage<2>(acc, pa, f_col, koff); break;
                case 3: diag_stage<3>(acc, pa, f_col, koff); break;
                case 4: diag_stage<4>(acc, pa, f_col, koff); break;
                case 5: diag_stage<5>(acc, pa, f_col, koff); break;
                case 6: diag_stage<6>(acc, pa, f_col, koff); break;
                default: diag_stage<7>(acc, pa, f_col, koff); break;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
        if (tid == 0 && i >= 1 && i - 1 + SST < nst) {
            const int r = i - 1;
            mbar_wait(&empty_bar[r % SST], (uint32_t)((r / SST) & 1));
            issue(r + SST);
        }
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
        switch (warp) {
            case 0: diag_store<0>(acc, P, g, t); break;
            case 1: diag_store<1>(acc, P, g, t); break;
            case 2: diag_store<2>(acc, P, g, t); break;
            case 3: diag_store<3>(acc, P, g, t); break;
            case 4: diag_store<4>(acc, P, g, t); break;
            case 5: diag_store<5>(acc, P, g, t); break;
            case 6: diag_store<6>(acc, P, g, t); break;
            default: diag_store<7>(acc, P, g, t); break;
        }
    }
}

// G[i,j] = G[j,i] = sum over the splits of block(i,j), fixed order; diagonal blocks only hold their 8 x 8 tiles on or
// above the diagonal, which cover every (il, jl) with il <= jl
__global__ void syrk_reduce_kernel(const double* __restrict__ partial, const __grid_constant__ SyrkPlan plan, int N,
                                   double* __restrict__ G) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)N * N) return;
    int i = (int)(idx % N), j = (int)(idx / N);
    if (i > j) return;
    const int bi = i / SB, bj = j / SB;
    const int il = i % SB, jl = j % SB;
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
    // CTAs per block roughly proportional to the block's cost (off-diagonal: 32 DMMAs per warp and k-step, diagonal: 17).
    // The diagonal weight stays at the 20 / 32 of the kernel that computed whole 32 x 32 diagonal tiles: a split's rows
    // fix the partial sum, and weighting by 17 / 32 would move rows between partial sums.  G would then change in its
    // last bits, and so would the nearly degenerate trailing singular vectors of the returned SVD.  The diagonal CTAs
    // finish early instead; the off-diagonal ones set the pace.
    constexpr double kOff = 4.0, kDiag = 2.5;
    int ndiag = p.nb, noff = p.nblk - p.nb;
    double unit = (double)sm_count / (kOff * noff + kDiag * ndiag);
    int total = 0, blk = 0;
    for (int bi = 0; bi < p.nb; ++bi)
        for (int bj = bi; bj < p.nb; ++bj, ++blk) {
            int ns = (int)((bi == bj ? kDiag : kOff) * unit);
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
    syrk_tma_kernel<<<plan.ncta, 32 * SWARPS, smem, st>>>(map, partial, plan);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int64_t nn = N * N;
    syrk_reduce_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, st>>>(partial, plan, (int)N, G);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

}  // namespace tlsq
