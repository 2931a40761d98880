// fused.cu -- ONE HBM pass per ALM iteration (n = 256): the epilogue of iteration k and the Gram of the SVT input of
// iteration k+1 in a single persistent kernel.  Replaces, inside the loop, the pair (alm_stream_kernel, syrk_tma_kernel)
// and with it the materialised SVT input W: per iteration the kernel reads D and Y_{k-1} and writes Y_k (3 S of HBM
// traffic instead of 7 S); the low-rank iterate stays factored (A_k = clamp(T_k V_k'), T: M x 32).
//
//   reference lines (src/robustPCA.jl):  E-step :188-191, SVT input :192, A = U_r (S_r - 1/mu) V_r' :205-208 (as
//   A = (W V_r) diag(f) V_r'), clamp :217-219, Z / Y / ||Z|| :221-225, and W'W of the next iteration for svd! :194.
//
// Work decomposition.  The upper triangle of a 256 x 256 FP64 Gram is 36 tiles of 32 x 32 = 288 KB of accumulators --
// more than one SM's register file.  A thread-block CLUSTER of two CTAs therefore shares every 32-row tile:
//   * CTA r owns columns [128 r, 128 r + 128) for the element-wise work (no redundant flops or HBM reads);
//   * the row reduction T = W V_r needs all 256 columns: the two 32 x RP partial sums are exchanged through
//     distributed shared memory (4 KB per tile);
//   * every CTA pushes the W_{k+1} values its peer needs into the peer's shared memory (st.shared::cluster) so that
//     both hold the operand tile; CTA 0 accumulates Gram tiles (a, b <= 5), a <= 3, CTA 1 the other 18 tiles;
//   * each warp owns 9 strips of 32 x 8 (36 DMMA.8x8x4 per k-step, 72 FP64 accumulators per thread).
// Per tile: TMA (cp.async.bulk.tensor) brings the D / Y / T tiles into single-buffered staging while the previous
// tile's DMMA phase runs; phases are separated by one __syncthreads and two cluster barriers.
// Partial Grams are written per cluster and summed in fixed order (deterministic), as is ||Z||_F^2.
#include <cuda.h>

#include "kernels.h"

namespace tlsq {

namespace {

constexpr int FR = 32;                 // rows per tile
constexpr int FN = kFusedN;            // 256 columns
constexpr int FH = FN / 2;             // columns owned by one CTA of the pair
constexpr int FWS = 36;                // column stride (doubles) of the DMMA operand tile: 36 = 4 mod 16 -> the
                                       // fragment loads (lane (g,t) -> column c0+g, row 4ks+t) hit 16 distinct banks
constexpr int W2_BYTES = FN * FWS * 8;
constexpr int TILE_DOUBLES = FH * FR;
constexpr int TILE_BYTES = TILE_DOUBLES * 8;

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
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t map_peer(uint32_t local_addr, uint32_t peer) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(peer));
    return r;
}
__device__ __forceinline__ void st_cluster(uint32_t addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

// sum_c t[c] v[c] with four independent FMA chains (RP is a multiple of 4; v is 16-byte aligned shared memory)
template <int RP>
__device__ __forceinline__ double dot_rp(const double (&t)[RP], const double* __restrict__ v) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
    for (int c = 0; c < RP; c += 4) {
        const double2 v0 = *reinterpret_cast<const double2*>(v + c);
        const double2 v1 = *reinterpret_cast<const double2*>(v + c + 2);
        a0 = fma(t[c], v0.x, a0);
        a1 = fma(t[c + 1], v0.y, a1);
        a2 = fma(t[c + 2], v1.x, a2);
        a3 = fma(t[c + 3], v1.y, a3);
    }
    return (a0 + a1) + (a2 + a3);
}

// TMA store of a shared-memory tile (bulk async group); the generic-proxy writes must be fenced by their writers
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int x, int y, const void* src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(map), "r"(x), "r"(y), "r"(smem_u32(src)) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// One 32-row tile of the Gram: the first N1 strips of the warp take their A fragments from tile row A, the others
// from tile row B (N1 is a per-warp constant; the switch at the call site keeps the accumulator indexing static).
template <int N1>
__device__ __forceinline__ void gram_phase(double (&acc)[9][4][2], const double* __restrict__ W2s, int aoffA, int aoffB,
                                           const int (&boff)[9], int ks0, int ks1) {
#pragma unroll 1
    for (int ks = ks0; ks < ks1; ++ks) {
        const double* wk = W2s + 4 * ks;
        double a1[4], a2[4];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
            a1[mi] = wk[aoffA + 8 * mi * FWS];
            if (N1 < 9) a2[mi] = wk[aoffB + 8 * mi * FWS];
        }
#pragma unroll
        for (int s = 0; s < 9; ++s) {
            const double b = wk[boff[s]];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) dmma884(acc[s][mi][0], acc[s][mi][1], s < N1 ? a1[mi] : a2[mi], b);
        }
    }
}

struct FusedDev {
    FusedArgs a;
    FusedStripTab tab;
    int ntiles, ncluster;
    int has_tp, has_tn, has_y, has_d;      // which TMA loads are issued per tile
};

template <int RP, bool HANKEL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(256, 1)
alm_fused_kernel(const __grid_constant__ CUtensorMap mD, const __grid_constant__ CUtensorMap mY,
                 const __grid_constant__ CUtensorMap mTp, const __grid_constant__ CUtensorMap mTn,
                 const __grid_constant__ CUtensorMap mYo, const __grid_constant__ CUtensorMap mTo, const FusedDev p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    double* W2s = reinterpret_cast<double*>(smem);              // [256][36] DMMA operand tile (both halves)
    double* Ds = reinterpret_cast<double*>(smem + W2_BYTES);    // [128][32] own-half D tile          (TMA)
    double* Ys = Ds + TILE_DOUBLES;                             // [128][32] own-half Y_{k-1} tile    (TMA)
    double* Es = Ys + TILE_DOUBLES;                             // [128][32] E_k (or the Gram operand in W / D mode)
    double* Vps = Es + TILE_DOUBLES;                            // [128][RP] own-half rows of V_{k-1}
    double* Vks = Vps + FH * RP;                                // [128][RP] own-half rows of V_k
    double* Tps = Vks + FH * RP;                                // [RP][32]  T_{k-1} tile             (TMA)
    double* Tns = Tps + RP * FR;                                // [RP][32]  T_k tile: TMA load when given, else TMA-store staging
    double* Tsum = Tns + RP * FR;                               // [2][RP][32] partial row sums of the two CTAs
    double* fs = Tsum + 2 * RP * FR;                            // [RP] shrink factors
    double* red = fs + RP;                                      // [8]
    uint64_t* bar = reinterpret_cast<uint64_t*>(red + 8);
    double* Tpart = W2s;                                        // [8][RP][32] aliases the operand tile (see S3)

    const FusedArgs& a = p.a;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const uint32_t rank = cluster_ctarank(), peer = rank ^ 1u;
    const int cl = blockIdx.x >> 1;
    const int c0 = (int)rank * FH;
    const int go = a.gram_of;
    const bool simple = (go == FUSED_GRAM_W) || (go == FUSED_GRAM_D);
    const bool nnA = a.nonnegA != 0;
    constexpr int UB = 8;

    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int idx = tid; idx < FH * RP; idx += 256) {
        const int jl = idx % FH, c = idx / FH;
        Vps[jl * RP + c] = (c < a.svp_prev && a.Vp) ? __ldg(a.Vp + (int64_t)c * FN + c0 + jl) : 0.0;
        Vks[jl * RP + c] = (c < a.svp && a.Vs) ? __ldg(a.Vs + (int64_t)c * FN + c0 + jl) : 0.0;
    }
    if (tid < RP) fs[tid] = (tid < a.svp && a.fvec) ? __ldg(a.fvec + tid) : 0.0;
    __syncthreads();
    cluster_arrive();            // the peer's shared memory must be live before the first remote store
    cluster_wait();

    const uint32_t tx_bytes = (uint32_t)((p.has_d ? TILE_BYTES : 0) + (p.has_y ? TILE_BYTES : 0) +
                                         (p.has_tp ? RP * FR * 8 : 0) + (p.has_tn ? RP * FR * 8 : 0));
    auto issue = [&](int tile) {
        mbar_expect_tx(bar, tx_bytes);
        if (p.has_d) tma_load_2d(Ds, &mD, tile * FR, c0, bar);
        if (p.has_y) tma_load_2d(Ys, &mY, tile * FR, c0, bar);
        if (p.has_tp) tma_load_2d(Tps, &mTp, tile * FR, 0, bar);
        if (p.has_tn) tma_load_2d(Tns, &mTn, tile * FR, 0, bar);
    };
    if (tid == 0 && cl < p.ntiles) issue(cl);

    // ---- this warp's 9 strips (32 x 8) of the Gram: at most two distinct tile rows --------------------------------
    int boff[9];
    int rowA, rowB, n1 = 0;
    {
        const uint8_t* rt = p.tab.row[rank][warp];
        const uint8_t* ct = p.tab.cs[rank][warp];
        rowA = rt[0];
        rowB = rt[8];
#pragma unroll
        for (int s = 0; s < 9; ++s) {
            boff[s] = (8 * (int)ct[s] + g) * FWS + t;
            n1 += ((int)rt[s] == rowA) ? 1 : 0;
        }
    }
    const int aoffA = (32 * rowA + g) * FWS + t;
    const int aoffB = (32 * rowB + g) * FWS + t;

    double acc[9][4][2];
#pragma unroll
    for (int s = 0; s < 9; ++s)
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) acc[s][mi][0] = acc[s][mi][1] = 0.0;
    double zz = 0.0;

    const uint32_t w2_peer = map_peer(smem_u32(W2s), peer);
    const uint32_t tsum_peer = map_peer(smem_u32(Tsum), peer);
    const bool push = (rank == 0) || (warp < 4);      // CTA 0 needs columns 128..191 of CTA 1; CTA 1 all of CTA 0's

    int it = 0;
    for (int tile = cl; tile < p.ntiles; tile += p.ncluster, ++it) {
        const int64_t row = (int64_t)tile * FR + lane;
        const bool rowok = row < a.M;
        mbar_wait(bar, (uint32_t)(it & 1));

        // ---- phase 2: E_k, W_k and the partial row sums of T = W_k V_k over this warp's 16 columns --------------
        if (go == FUSED_GRAM_D) {
#pragma unroll 1
            for (int u = 0; u < 16; ++u) {
                const int jl = 16 * warp + u;
                const double d = HANKEL ? (rowok ? __ldg(a.D.p + row + c0 + jl) : 0.0) : Ds[jl * FR + lane];
                Es[jl * FR + lane] = d;
            }
        } else {
            // staged in batches of UB elements so that every stage exposes UB independent dependency chains (the
            // FP64 pipe is shared by only two warps per scheduler: instruction-level parallelism must hide its latency)
            double tp[RP], tr[RP];
#pragma unroll
            for (int c = 0; c < RP; ++c) {
                tp[c] = (p.has_tp && c < a.svp_prev) ? Tps[c * FR + lane] : 0.0;
                tr[c] = 0.0;
            }
#pragma unroll 1
            for (int u0 = 0; u0 < 16; u0 += UB) {
                double av[UB], wv[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) av[u] = dot_rp<RP>(tp, Vps + (16 * warp + u0 + u) * RP);
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int jl = 16 * warp + u0 + u;
                    const double d = HANKEL ? (rowok ? __ldg(a.D.p + row + c0 + jl) : 0.0) : Ds[jl * FR + lane];
                    const double yp = Ys[jl * FR + lane];
                    const double ap = (nnA && !(__double_as_longlong(av[u]) > 0)) ? 0.0 : av[u];
                    double e, w;
                    alm_ew(d, ap, yp, a.im, a.eps, a.nonnegE, e, w);
                    Es[jl * FR + lane] = (go == FUSED_GRAM_W) ? w : e;
                    wv[u] = w;
                }
                if (a.compute_T) {
#pragma unroll
                    for (int u = 0; u < UB; ++u) {
                        const double* v = Vks + (16 * warp + u0 + u) * RP;
#pragma unroll
                        for (int c = 0; c < RP; c += 2) {
                            const double2 vv = *reinterpret_cast<const double2*>(v + c);
                            tr[c] = fma(wv[u], vv.x, tr[c]);
                            tr[c + 1] = fma(wv[u], vv.y, tr[c + 1]);
                        }
                    }
                }
            }
            if (a.compute_T) {
#pragma unroll
                for (int c = 0; c < RP; ++c) Tpart[(warp * RP + c) * FR + lane] = tr[c];
                __syncthreads();                                                       // S1
                for (int idx = tid; idx < RP * FR; idx += 256) {
                    double s = 0.0;
#pragma unroll
                    for (int w8 = 0; w8 < 8; ++w8) s += Tpart[w8 * RP * FR + idx];
                    Tsum[rank * RP * FR + idx] = s;
                    st_cluster(tsum_peer + (uint32_t)((rank * RP * FR + idx) * 8), s);
                }
            }
        }
        cluster_arrive();                                                              // C1
        cluster_wait();

        // ---- phase 4: A_k, Z, Y_k, ||Z||^2, W_{k+1}; operand tile to both CTAs -----------------------------------
        if (simple) {
#pragma unroll 1
            for (int u = 0; u < 16; ++u) {
                const int jl = 16 * warp + u;
                const double val = Es[jl * FR + lane];
                const int off = (c0 + jl) * FWS + lane;
                W2s[off] = val;
                if (push) st_cluster(w2_peer + (uint32_t)off * 8u, val);
            }
        } else {
            double tk[RP];
            if (a.compute_T) {
#pragma unroll
                for (int c = 0; c < RP; ++c) {
                    tk[c] = fs[c] * (Tsum[c * FR + lane] + Tsum[(RP + c) * FR + lane]);
                    if (rank == 0 && (c & 7) == warp) Tns[c * FR + lane] = tk[c];          // staged for the TMA store
                }
            } else {
#pragma unroll
                for (int c = 0; c < RP; ++c) tk[c] = c < a.svp ? Tns[c * FR + lane] : 0.0;
            }
#pragma unroll 1
            for (int u0 = 0; u0 < 16; u0 += UB) {
                double av[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) av[u] = dot_rp<RP>(tk, Vks + (16 * warp + u0 + u) * RP);
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    const int jl = 16 * warp + u0 + u;
                    const double d = HANKEL ? (rowok ? __ldg(a.D.p + row + c0 + jl) : 0.0) : Ds[jl * FR + lane];
                    const double yp = Ys[jl * FR + lane];
                    const double e = Es[jl * FR + lane];
                    const double an = (nnA && !(__double_as_longlong(av[u]) > 0)) ? 0.0 : av[u];   // max.(A, 0) :218
                    const double z = __dsub_rn(__dsub_rn(d, an), e);                    // @. Z = D - A - E  :221
                    const double yn = __dadd_rn(yp, __dmul_rn(a.mu, z));                // @. Y = Y + mu*Z   :222
                    zz = fma(z, z, zz);
                    Es[jl * FR + lane] = yn;                                            // staged for the TMA store
                    double e2, w2;
                    alm_ew(d, an, yn, a.im_next, a.eps_next, a.nonnegE, e2, w2);        // SVT input of iteration k+1
                    const double val = (go == FUSED_GRAM_WNEXT) ? w2 : z;
                    const int off = (c0 + jl) * FWS + lane;
                    W2s[off] = val;
                    if (push) st_cluster(w2_peer + (uint32_t)off * 8u, val);
                }
            }
        }
        if (!simple) fence_async_smem();        // Y_k / T_k tiles were written through the generic proxy
        cluster_arrive();                                                              // C2
        cluster_wait();
        if (tid == 0 && !simple) {
            if (a.write_Y) tma_store_2d(&mYo, tile * FR, c0, Es);
            if (a.compute_T && rank == 0 && a.Tn) tma_store_2d(&mTo, tile * FR, 0, Tns);
            tma_commit();
        }
        if (tid == 0 && tile + p.ncluster < p.ntiles) issue(tile + p.ncluster);        // D / Y / T staging is free again

        // ---- DMMA phase: G += W2' W2 over this warp's 9 strips; the next tile's loads are issued half-way, when the
        //      TMA stores above have long finished reading their staging buffers -------------------------------------
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            const int ks0 = half * (FR / 8), ks1 = ks0 + FR / 8;
            switch (n1) {
                case 1: gram_phase<1>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 2: gram_phase<2>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 3: gram_phase<3>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 4: gram_phase<4>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 5: gram_phase<5>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 6: gram_phase<6>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 7: gram_phase<7>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                case 8: gram_phase<8>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
                default: gram_phase<9>(acc, W2s, aoffA, aoffB, boff, ks0, ks1); break;
            }
            if (half == 0 && tid == 0) tma_wait_read0();     // the stores have read Es / Tns long ago: no stall; S3 publishes it
        }
        __syncthreads();                                                               // S3: operand tile is free
    }

    // ---- partial Gram of this cluster (disjoint tiles per CTA) and ||Z||^2 of this CTA ---------------------------
    double* P = a.partial + (size_t)cl * (FN * FN);
    {
        const uint8_t* rt = p.tab.row[rank][warp];
        const uint8_t* ct = p.tab.cs[rank][warp];
#pragma unroll
        for (int s = 0; s < 9; ++s) {
            const int r0 = 32 * (int)rt[s] + g;
            const int cc = 8 * (int)ct[s] + 2 * t;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                P[(size_t)cc * FN + r0 + 8 * mi] = acc[s][mi][0];
                P[(size_t)(cc + 1) * FN + r0 + 8 * mi] = acc[s][mi][1];
            }
        }
    }
    zz = warp_sum(zz);
    if (lane == 0) red[warp] = zz;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) s += red[w8];
        a.zpart[blockIdx.x] = s;
    }
    if (tid == 0) tma_wait_all0();
    cluster_arrive();            // keep this CTA's shared memory alive until the peer is done with it
    cluster_wait();
}


// (A warp-specialised variant -- 8 MMA warps + 4 producer warps, setmaxnreg, mbarrier-only synchronisation -- was built and
// measured in round 1: 8.4 ms against 5.1 ms for this lock-step kernel, because the producers' 2-cycle FP64 instructions
// queue behind the 16-cycle DMMAs on the shared FP64 pipe.  It was removed in round 2; see DESIGN.md.)

// G[i,j] = G[j,i] = sum over the clusters (fixed order) of the upper-triangular partials; zz = sum of the CTA partials
__global__ void fused_reduce_kernel(const double* __restrict__ partial, int ncluster, const double* __restrict__ zpart,
                                    int ncta, double* __restrict__ G, double* __restrict__ zz_out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0 && zz_out) {
        double s = 0.0;
        for (int c = 0; c < ncta; ++c) s += zpart[c];
        *zz_out = s;
    }
    if (idx >= FN * FN) return;
    const int i = idx % FN, j = idx / FN;
    if (i > j) return;
    const double* p = partial + (size_t)j * FN + i;
    double s = 0.0;
    for (int c = 0; c < ncluster; ++c) s += p[(size_t)c * (FN * FN)];
    G[(size_t)j * FN + i] = s;
    G[(size_t)i * FN + j] = s;
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

bool encode_map(CUtensorMap* map, const double* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, int box_cols) {
    const cuuint64_t gdim[2] = {(cuuint64_t)rows, (cuuint64_t)cols};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * 8};
    const cuuint32_t box[2] = {(cuuint32_t)box_rows, (cuuint32_t)box_cols};
    const cuuint32_t estr[2] = {1, 1};
    return encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Strip table: CTA 0 owns Gram tiles (a, b), a <= 3, a <= b <= 5; CTA 1 owns (a, 6..7), a <= 3, and (a, b >= a), a >= 4.
// Strips (32 x 8) are enumerated tile row by tile row; warp w takes strips [9w, 9w + 9) -- at most two tile rows.
FusedStripTab make_tab() {
    FusedStripTab tb = {};
    for (int r = 0; r < 2; ++r) {
        int n = 0;
        for (int arow = 0; arow < 8; ++arow) {
            int lo, hi;                                    // strip columns [lo, hi) in units of 8 columns
            if (r == 0) { if (arow > 3) continue; lo = 4 * arow; hi = 24; }
            else if (arow <= 3) { lo = 24; hi = 32; }
            else { lo = 4 * arow; hi = 32; }
            for (int c = lo; c < hi; ++c, ++n) {
                tb.row[r][n / 9][n % 9] = (uint8_t)arow;
                tb.cs[r][n / 9][n % 9] = (uint8_t)c;
            }
        }
    }
    return tb;
}

template <int RP>
size_t smem_bytes() {
    return (size_t)W2_BYTES + 3 * (size_t)TILE_BYTES + 2 * (size_t)FH * RP * 8 + 2 * (size_t)RP * FR * 8 +
           2 * (size_t)RP * FR * 8 + (size_t)RP * 8 + 8 * 8 + 16;
}

struct Inst {
    int ncluster = -1;      // co-resident clusters (queried once)
};

template <class Kern>
int query_clusters(Kern kern, int threads, size_t smem, int sm_count) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(sm_count & ~1));
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nc = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&nc, kern, &cfg);
    if (e != cudaSuccess || nc < 1) { cudaGetLastError(); nc = sm_count / 2 - 2; }
    if (nc > sm_count / 2) nc = sm_count / 2;
    return nc < 1 ? 1 : nc;
}

template <int RP, bool HANKEL>
cudaError_t launch_inst(const CUtensorMap& mD, const CUtensorMap& mY, const CUtensorMap& mTp, const CUtensorMap& mTn,
                        const CUtensorMap& mYo, const CUtensorMap& mTo, FusedDev p, int sm_count, cudaStream_t st,
                        int* ncluster_out) {
    static Inst inst;
    auto kern = alm_fused_kernel<RP, HANKEL>;
    const size_t smem = smem_bytes<RP>();
    if (inst.ncluster < 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        inst.ncluster = query_clusters(kern, 256, smem, sm_count);
    }
    int nc = inst.ncluster;
    if (nc > p.ntiles) nc = p.ntiles > 0 ? p.ntiles : 1;
    p.ncluster = nc;
    *ncluster_out = nc;
    kern<<<2 * nc, 256, smem, st>>>(mD, mY, mTp, mTn, mYo, mTo, p);
    return cudaGetLastError();
}

template <int RP>
cudaError_t launch_rp(bool hankel, const CUtensorMap* m, const FusedDev& p, int sm_count, cudaStream_t st, int* nc) {
    return hankel ? launch_inst<RP, true>(m[0], m[1], m[2], m[3], m[4], m[5], p, sm_count, st, nc)
                  : launch_inst<RP, false>(m[0], m[1], m[2], m[3], m[4], m[5], p, sm_count, st, nc);
}

}  // namespace

FusedStripTab fused_strip_table() { return make_tab(); }

size_t fused_partial_doubles(int sm_count) {
    return (size_t)(sm_count / 2) * FN * FN + (size_t)sm_count + 8;
}

bool fused_eligible(const MatSrc& D, bool hankel, int64_t M, int64_t N) {
    if (N != FN || M < 4096 || M >= ((int64_t)1 << 31)) return false;
    if (hankel) { if (D.ld != 1) return false; }        // Y / T live in padded (even) leading dimensions: any M
    else if ((M & 1) || (D.ld & 1) || (reinterpret_cast<uintptr_t>(D.p) & 15)) return false;
    return encode_fn() != nullptr;
}

int fused_rank_pad(int svp, int svp_prev) {
    const int m = svp > svp_prev ? svp : svp_prev;
    return m <= 4 ? 4 : ((m + 3) & ~3);
}

cudaError_t launch_alm_fused(const FusedArgs& a, bool hankel, const double* Yp, const double* Tp, const double* Tn_given,
                             double* G, double* zz_out, int sm_count, cudaStream_t st, int64_t* launches) {
    static const FusedStripTab tab = make_tab();
    if (!encode_fn()) return cudaErrorNotSupported;
    const int rp = fused_rank_pad(a.svp, a.svp_prev);
    if (rp > kFusedMaxRank) return cudaErrorInvalidValue;
    FusedDev p = {};
    p.a = a;
    p.tab = tab;
    p.ntiles = (int)((a.M + FR - 1) / FR);
    p.has_d = hankel ? 0 : 1;
    p.has_y = (a.gram_of == FUSED_GRAM_D) ? 0 : 1;
    p.has_tp = (a.gram_of != FUSED_GRAM_D && a.svp_prev > 0 && Tp) ? 1 : 0;
    const bool needs_tk = (a.gram_of == FUSED_GRAM_WNEXT || a.gram_of == FUSED_GRAM_Z);
    p.has_tn = (needs_tk && !a.compute_T) ? 1 : 0;
    if (p.has_tn && !Tn_given) return cudaErrorInvalidValue;
    if (p.has_y && !Yp) return cudaErrorInvalidValue;
    // a valid (even if unused) tensor map for every slot
    const double* any = a.partial;      // cudaMalloc-aligned placeholder for the unused slots
    CUtensorMap m[6];      // D, Y_{k-1}, T_{k-1}, T_k (given), Y_k out, T_k out
    bool ok = true;
    ok &= hankel ? encode_map(&m[0], any, 32, 128, 32, FR, FH) : encode_map(&m[0], a.D.p, a.M, FN, a.D.ld, FR, FH);
    ok &= p.has_y ? encode_map(&m[1], Yp, a.M, FN, a.ldy, FR, FH) : encode_map(&m[1], any, 32, 128, 32, FR, FH);
    ok &= p.has_tp ? encode_map(&m[2], Tp, a.M, kStreamMaxRank, a.ldt, FR, rp) : encode_map(&m[2], any, 32, 128, 32, FR, rp);
    ok &= p.has_tn ? encode_map(&m[3], Tn_given, a.M, kStreamMaxRank, a.ldt, FR, rp) : encode_map(&m[3], any, 32, 128, 32, FR, rp);
    const bool y_out = needs_tk && a.write_Y && a.Yn;
    const bool t_out = needs_tk && a.compute_T && a.Tn;
    ok &= y_out ? encode_map(&m[4], a.Yn, a.M, FN, a.ldy, FR, FH) : encode_map(&m[4], any, 32, 128, 32, FR, FH);
    ok &= t_out ? encode_map(&m[5], a.Tn, a.M, kStreamMaxRank, a.ldt, FR, rp) : encode_map(&m[5], any, 32, 128, 32, FR, rp);
    if (!ok) return cudaErrorInvalidValue;
    if (needs_tk && a.write_Y && !a.Yn) return cudaErrorInvalidValue;
    p.a.VpT = nullptr;
    int nc = 0;
    cudaError_t e;
    switch (rp) {
        case 4:  e = launch_rp<4>(hankel, m, p, sm_count, st, &nc); break;
        case 8:  e = launch_rp<8>(hankel, m, p, sm_count, st, &nc); break;
        case 12: e = launch_rp<12>(hankel, m, p, sm_count, st, &nc); break;
        default: e = launch_rp<16>(hankel, m, p, sm_count, st, &nc); break;
    }
    if (e != cudaSuccess) return e;
    fused_reduce_kernel<<<(FN * FN + 255) / 256, 256, 0, st>>>(a.partial, nc, a.zpart, 2 * nc, G, zz_out);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

}  // namespace tlsq
