// eig.cu -- eigen-decomposition of the small symmetric PSD Gram matrix G = W'W (n <= 512) by one-sided
// (Hestenes) Jacobi with warp-shuffle rotations.  sigma_i = sqrt(lambda_i) and V are exactly what the reference
// takes from LAPACK dgesdd (src/robustPCA.jl:194) -- the left factor is never needed because
// A = U_r (S_r - 1/mu) V_r' = W V_r diag(1 - 1/(mu s_i)) V_r'.
//
// Invariant: X = G * V with V orthogonal.  Plane rotations are applied to column pairs of X (and V) until the
// columns of X are mutually orthogonal; then X = V * Lambda.  Warm start: V0 = eigenvectors of the previous ALM
// iteration, X0 = G * V0 is already nearly orthogonal, so 1-3 sweeps suffice instead of 6-10.
//
// Engines:
//  * jacobi_cluster_block_kernel (n <= 256): ONE thread-block cluster of up to 16 CTAs holds all columns (X and V parts)
//    in distributed shared memory; hierarchical tournament: every CTA rotates the cross pairs of its two half-blocks in
//    place, then the half-blocks move one circle-method position through DSMEM (one cluster barrier per outer round).
//  * jacobi_coop_block_kernel (256 < n <= 512): the same tournament on a cooperative grid, half-blocks in shared memory,
//    exchange through a double-buffered staging area in L2 (one grid barrier per outer round).
//  * jacobi_global_kernel / jacobi_global_loop_kernel (fallback / n > 512): cooperative grid, columns stay in L2.
// svd mode: the same kernels orthogonalise the columns of a GENERAL square matrix K (K V = U S) -- used by the
// CholeskyQR2-style refinement of the returned SVD (solver.cu); chol_upper_kernel is the Cholesky factor it needs.
#include <cooperative_groups.h>
#include "kernels.h"

namespace cg = cooperative_groups;

namespace tlsq {

namespace {

// ---------------------------------------------------------------------------------------------------
// X0 = G * V  (n x n x n, plain FP64 FMA with 32x32 shared tiles; ~17 MFMA at n=256 -> microseconds)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gemm_small_kernel(const double* __restrict__ G, const double* __restrict__ V, int n, double* __restrict__ X) {
    __shared__ double Gs[32][33];
    __shared__ double Vsm[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // ty in 0..7
    const int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = 0; k0 < n; k0 += 32) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int kk = ty + 8 * r;
            // Gs[kk][tx] = G[i0+tx, k0+kk]   (column-major, symmetric)
            Gs[kk][tx] = (i0 + tx < n && k0 + kk < n) ? G[(int64_t)(k0 + kk) * n + i0 + tx] : 0.0;
            // Vsm[kk][tx] = V[k0+tx, j0+kk]
            Vsm[kk][tx] = (k0 + tx < n && j0 + kk < n) ? V[(int64_t)(j0 + kk) * n + k0 + tx] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int jj = ty + 8 * r;
            double a = acc[r];
#pragma unroll
            for (int kk = 0; kk < 32; ++kk) a = fma(Gs[kk][tx], Vsm[jj][kk], a);
            acc[r] = a;
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int jj = ty + 8 * r;
        if (i0 + tx < n && j0 + jj < n) X[(int64_t)(j0 + jj) * n + i0 + tx] = acc[r];
    }
}

// ---------------------------------------------------------------------------------------------------
// rotation of one column pair held in registers (E doubles per lane per column part)
// returns true if a rotation was applied
// ---------------------------------------------------------------------------------------------------
template <int E>
__device__ __forceinline__ bool jacobi_rotate(double (&xp)[E], double (&xq)[E], double (&vp)[E], double (&vq)[E],
                                              double tol) {
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
    if (!jacobi_cs(alpha, beta, gamma, tol, c, s)) return false;       // already orthogonal (or a null column)
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

// ---------------------------------------------------------------------------------------------------
// Cluster engine, hierarchical tournament (the flat one-barrier-per-round tournament of round 1 was 5.8 ms vs 4.2 ms).  Every CTA holds two HALF-BLOCKS of spc columns (top / bottom).
// One sweep = 2C-1 outer rounds; in an outer round a CTA rotates all spc x spc cross pairs of its two half-blocks in
// spc inner rounds (pair (T[w], B[(w+r) % spc]) on warp w, in place in shared memory, __syncthreads between rounds),
// then the half-blocks move one position of the circle method (top[0] fixed, top[c] -> top[c+1], top[C-1] -> bot[C-1],
// bot[c] -> bot[c-1], bot[0] -> top[1]) through DSMEM and the cluster synchronises ONCE.  The pairs inside a
// half-block are rotated in the first outer round of every sweep.  Every column pair is visited exactly once per
// sweep like in the flat tournament, but with 2C-1 = 31 cluster barriers per sweep instead of 255 (n = 256).
// ---------------------------------------------------------------------------------------------------
template <int E>
__global__ void __launch_bounds__(256)
jacobi_cluster_block_kernel(const double* __restrict__ X0, const double* __restrict__ V0, int n, int spc,
                            double tol, int max_sweeps, double* __restrict__ Xo, double* __restrict__ Vo,
                            int* __restrict__ info, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;      // fast path succeeded: nothing to do (uniform over the cluster)
    constexpr int LEN = 32 * E;
    extern __shared__ double smem[];
    __shared__ int counters[64];
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int c = (int)cluster.block_rank();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot_doubles = 2 * LEN;               // [X part | V part]
    const int buf_doubles = 2 * spc * slot_doubles; // slots 0..spc-1 = top half-block, spc..2spc-1 = bottom
    double* buf0 = smem;
    double* buf1 = smem + buf_doubles;
    if (threadIdx.x < 64) counters[threadIdx.x] = 0;

    // initial load: column j -> CTA j / (2 spc), slot j % (2 spc).  Columns >= n are zero dummies.
    for (int sl = warp; sl < 2 * spc; sl += 8) {
        const int j = c * 2 * spc + sl;
        double* dst = buf0 + sl * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = lane + 32 * e;
            double xv = 0.0, vv = 0.0;
            if (j < n && i < n) {
                xv = X0[(int64_t)j * n + i];
                vv = V0 ? V0[(int64_t)j * n + i] : (i == j ? 1.0 : 0.0);
            }
            dst[i] = xv;
            dst[LEN + i] = vv;
        }
    }
    cluster.sync();

    int* counters0 = cluster.map_shared_rank(counters, 0);
    double* cur = buf0;
    double* nxt = buf1;
    const int spe = spc + (spc & 1);                // even size of the in-block tournament
    const int outer = 2 * C - 1;
    int sweep = 0;

    auto rotate_slots = [&](int sa, int sb) -> bool {
        double xp[E], xq[E], vp[E], vq[E];
        double* pa = cur + sa * slot_doubles;
        double* pb = cur + sb * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            xp[e] = pa[lane + 32 * e];
            vp[e] = pa[LEN + lane + 32 * e];
            xq[e] = pb[lane + 32 * e];
            vq[e] = pb[LEN + lane + 32 * e];
        }
        if (!jacobi_rotate<E>(xp, xq, vp, vq, tol)) return false;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            pa[lane + 32 * e] = xp[e];
            pa[LEN + lane + 32 * e] = vp[e];
            pb[lane + 32 * e] = xq[e];
            pb[LEN + lane + 32 * e] = vq[e];
        }
        return true;
    };

    for (; sweep < max_sweeps; ++sweep) {
        bool rotated = false;
        for (int orow = 0; orow < outer; ++orow) {
            if (orow == 0 && spc > 1) {
                // pairs inside the two half-blocks: circle method on spe columns, warps [0, spe/2) on top, next on bottom
                for (int r = 0; r < spe - 1; ++r) {
                    const int half = warp / (spe / 2), pi = warp % (spe / 2);
                    if (half < 2) {
                        int p, q;
                        if (pi == 0) { p = spe - 1; q = r; }
                        else { p = (r + pi) % (spe - 1); q = (r - pi + (spe - 1)) % (spe - 1); }
                        if (p < spc && q < spc) rotated |= rotate_slots(half * spc + p, half * spc + q);
                    }
                    __syncthreads();
                }
            }
            for (int r = 0; r < spc; ++r) {
                if (warp < spc) rotated |= rotate_slots(warp, spc + (warp + r) % spc);
                __syncthreads();
            }
            // move the half-blocks (every column is copied into the next buffer of its destination CTA)
            for (int sl = warp; sl < 2 * spc; sl += 8) {
                const int top = sl < spc ? 1 : 0, l = top ? sl : sl - spc;
                int dc, dtop;
                if (C == 1) { dc = 0; dtop = top; }
                else if (top) {
                    if (c == 0) { dc = 0; dtop = 1; }
                    else if (c == C - 1) { dc = C - 1; dtop = 0; }
                    else { dc = c + 1; dtop = 1; }
                } else {
                    if (c == 0) { dc = 1; dtop = 1; }
                    else { dc = c - 1; dtop = 0; }
                }
                const double* src = cur + sl * slot_doubles;
                double* base = (dc == c) ? nxt : cluster.map_shared_rank(nxt, dc);
                double* dst = base + ((dtop ? 0 : spc) + l) * slot_doubles;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    dst[lane + 32 * e] = src[lane + 32 * e];
                    dst[LEN + lane + 32 * e] = src[LEN + lane + 32 * e];
                }
            }
            cluster.sync();
            double* tmp = cur; cur = nxt; nxt = tmp;
        }
        if (rotated && lane == 0) atomicAdd(counters0 + sweep, 1);
        cluster.sync();
        const int cnt = *((volatile int*)(counters0 + sweep));
        if (cnt == 0) { ++sweep; break; }
    }
    cluster.sync();   // nobody may exit while a peer still reads counters0 / writes DSMEM

    for (int sl = warp; sl < 2 * spc; sl += 8) {   // write back (order is irrelevant; eig_post sorts)
        const int j = c * 2 * spc + sl;
        const double* src = cur + sl * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = lane + 32 * e;
            if (i < n) {
                Xo[(int64_t)j * n + i] = src[i];
                Vo[(int64_t)j * n + i] = src[LEN + i];
            }
        }
    }
    if (c == 0 && threadIdx.x == 0) info[0] = sweep;
}

// ---------------------------------------------------------------------------------------------------
// Global-memory engine (cooperative launch): columns live in Xo / Vo (L2 resident), one warp per pair.
// ---------------------------------------------------------------------------------------------------
template <int E>
__global__ void __launch_bounds__(256)
jacobi_global_kernel(int n, int np, double tol, int max_sweeps, double* __restrict__ Xo, double* __restrict__ Vo,
                     int* __restrict__ info, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    cg::grid_group grid = cg::this_grid();
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const int npairs = np / 2;
    int* counters = info + 2;
    int sweep = 0;
    for (; sweep < max_sweeps; ++sweep) {
        bool rotated = false;
        for (int round = 0; round < np - 1; ++round) {
            for (int pi = gw; pi < npairs; pi += nw) {
                int p, q;
                if (pi == 0) { p = np - 1; q = round; }
                else { p = (round + pi) % (np - 1); q = (round - pi + (np - 1)) % (np - 1); }
                if (p >= n || q >= n) continue;
                double xp[E], xq[E], vp[E], vq[E];
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int i = lane + 32 * e;
                    const bool ok = i < n;
                    xp[e] = ok ? __ldcg(Xo + (int64_t)p * n + i) : 0.0;
                    xq[e] = ok ? __ldcg(Xo + (int64_t)q * n + i) : 0.0;
                    vp[e] = ok ? __ldcg(Vo + (int64_t)p * n + i) : 0.0;
                    vq[e] = ok ? __ldcg(Vo + (int64_t)q * n + i) : 0.0;
                }
                if (jacobi_rotate<E>(xp, xq, vp, vq, tol)) {
                    rotated = true;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const int i = lane + 32 * e;
                        if (i < n) {
                            __stcg(Xo + (int64_t)p * n + i, xp[e]);
                            __stcg(Xo + (int64_t)q * n + i, xq[e]);
                            __stcg(Vo + (int64_t)p * n + i, vp[e]);
                            __stcg(Vo + (int64_t)q * n + i, vq[e]);
                        }
                    }
                }
            }
            grid.sync();
        }
        if (rotated && lane == 0) atomicAdd(counters + sweep, 1);
        grid.sync();
        const int cnt = *((volatile int*)(counters + sweep));
        if (cnt == 0) { ++sweep; break; }
    }
    if (gw == 0 && lane == 0) info[0] = sweep;
}


// Same engine for large n (> 512): a column no longer fits a lane's registers, so every pair makes two passes over its
// columns (dot products, then the rotation) out of L2.  Slow (O(100 ms) per sweep at n = 2048) but it is only the
// fallback of the large-n fast path and the once-per-solve full spectrum of the returned SVD.
__global__ void __launch_bounds__(256)
jacobi_global_loop_kernel(int n, int np, double tol, int max_sweeps, double* __restrict__ Xo, double* __restrict__ Vo,
                          int* __restrict__ info, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    cg::grid_group grid = cg::this_grid();
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const int npairs = np / 2;
    int* counters = info + 2;
    int sweep = 0;
    for (; sweep < max_sweeps; ++sweep) {
        bool rotated = false;
        for (int round = 0; round < np - 1; ++round) {
            for (int pi = gw; pi < npairs; pi += nw) {
                int p, q;
                if (pi == 0) { p = np - 1; q = round; }
                else { p = (round + pi) % (np - 1); q = (round - pi + (np - 1)) % (np - 1); }
                if (p >= n || q >= n) continue;
                double* xp = Xo + (int64_t)p * n;
                double* xq = Xo + (int64_t)q * n;
                double alpha = 0.0, beta = 0.0, gamma = 0.0;
                for (int i = lane; i < n; i += 32) {
                    const double a = __ldcg(xp + i), b = __ldcg(xq + i);
                    alpha = fma(a, a, alpha);
                    beta = fma(b, b, beta);
                    gamma = fma(a, b, gamma);
                }
                alpha = warp_sum(alpha); beta = warp_sum(beta); gamma = warp_sum(gamma);
                double c, s;
                if (!jacobi_cs(alpha, beta, gamma, tol, c, s)) continue;
                rotated = true;
                double* vp = Vo + (int64_t)p * n;
                double* vq = Vo + (int64_t)q * n;
                for (int i = lane; i < n; i += 32) {
                    const double a = __ldcg(xp + i), b = __ldcg(xq + i);
                    __stcg(xp + i, fma(c, a, -s * b));
                    __stcg(xq + i, fma(s, a, c * b));
                    const double va = __ldcg(vp + i), vb = __ldcg(vq + i);
                    __stcg(vp + i, fma(c, va, -s * vb));
                    __stcg(vq + i, fma(s, va, c * vb));
                }
            }
            grid.sync();
        }
        if (rotated && lane == 0) atomicAdd(counters + sweep, 1);
        grid.sync();
        const int cnt = *((volatile int*)(counters + sweep));
        if (cnt == 0) { ++sweep; break; }
    }
    if (gw == 0 && lane == 0) info[0] = sweep;
}


// ---------------------------------------------------------------------------------------------------------------------
// Cooperative-grid form of the hierarchical tournament for 256 < n <= 512: the columns no longer fit one cluster's
// shared memory (4 MB for X and V), so every CTA keeps its two half-blocks of `spc` columns in shared memory, rotates
// all their pairs there (__syncthreads only), and the half-blocks move one circle-method position through a
// double-buffered staging area in global memory (L2) with ONE grid barrier per outer round: 2C-1 = 63 grid barriers per
// sweep at n = 512 instead of the 511 of jacobi_global_kernel (which also went to L2 for every single rotation).
// ---------------------------------------------------------------------------------------------------------------------
template <int E>
__global__ void __launch_bounds__(256)
jacobi_coop_block_kernel(const double* __restrict__ X0, const double* __restrict__ V0, int n, int spc, double tol,
                         int max_sweeps, double* __restrict__ XoA, double* __restrict__ VoA, double* __restrict__ XoB,
                         double* __restrict__ VoB, int* __restrict__ info, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;      // fast path succeeded: nothing to do (uniform over the grid)
    constexpr int LEN = 32 * E;
    extern __shared__ double smem[];
    cg::grid_group grid = cg::this_grid();
    const int C = (int)gridDim.x;
    const int c = (int)blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot_doubles = 2 * LEN;               // [X part | V part]
    double* cur = smem;                             // slots 0..spc-1 = top half-block, spc..2spc-1 = bottom
    int* counters = info + 2;

    for (int sl = warp; sl < 2 * spc; sl += 8) {    // initial load: column j -> CTA j / (2 spc), slot j % (2 spc)
        const int j = c * 2 * spc + sl;
        double* dst = cur + sl * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = lane + 32 * e;
            double xv = 0.0, vv = 0.0;
            if (j < n && i < n) {
                xv = X0[(int64_t)j * n + i];
                vv = V0 ? V0[(int64_t)j * n + i] : (i == j ? 1.0 : 0.0);
            }
            dst[i] = xv;
            dst[LEN + i] = vv;
        }
    }
    __syncthreads();

    auto rotate_slots = [&](int sa, int sb) -> bool {
        double xp[E], xq[E], vp[E], vq[E];
        double* pa = cur + sa * slot_doubles;
        double* pb = cur + sb * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            xp[e] = pa[lane + 32 * e];
            vp[e] = pa[LEN + lane + 32 * e];
            xq[e] = pb[lane + 32 * e];
            vq[e] = pb[LEN + lane + 32 * e];
        }
        if (!jacobi_rotate<E>(xp, xq, vp, vq, tol)) return false;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            pa[lane + 32 * e] = xp[e];
            pa[LEN + lane + 32 * e] = vp[e];
            pb[lane + 32 * e] = xq[e];
            pb[LEN + lane + 32 * e] = vq[e];
        }
        return true;
    };

    const int spe = spc + (spc & 1);                // even size of the in-block tournament
    const int outer = 2 * C - 1;
    int sweep = 0, stage = 0;
    for (; sweep < max_sweeps; ++sweep) {
        bool rotated = false;
        for (int orow = 0; orow < outer; ++orow) {
            if (orow == 0 && spc > 1) {
                for (int r = 0; r < spe - 1; ++r) {         // pairs inside the two half-blocks
                    const int half = warp / (spe / 2), pi = warp % (spe / 2);
                    if (half < 2) {
                        int p, q;
                        if (pi == 0) { p = spe - 1; q = r; }
                        else { p = (r + pi) % (spe - 1); q = (r - pi + (spe - 1)) % (spe - 1); }
                        if (p < spc && q < spc) rotated |= rotate_slots(half * spc + p, half * spc + q);
                    }
                    __syncthreads();
                }
            }
            for (int r = 0; r < spc; ++r) {                 // all cross pairs of the two half-blocks
                if (warp < spc) rotated |= rotate_slots(warp, spc + (warp + r) % spc);
                __syncthreads();
            }
            if (C == 1) continue;
            // move the half-blocks one circle-method position through the staging area (ping-pong: a CTA that is still
            // reading round r never sees the writes of round r+1)
            double* Xs = stage ? XoB : XoA;
            double* Vs = stage ? VoB : VoA;
            for (int sl = warp; sl < 2 * spc; sl += 8) {
                const int top = sl < spc ? 1 : 0, l = top ? sl : sl - spc;
                int dc, dtop;
                if (top) {
                    if (c == 0) { dc = 0; dtop = 1; }
                    else if (c == C - 1) { dc = C - 1; dtop = 0; }
                    else { dc = c + 1; dtop = 1; }
                } else {
                    if (c == 0) { dc = 1; dtop = 1; }
                    else { dc = c - 1; dtop = 0; }
                }
                const double* src = cur + sl * slot_doubles;
                const int64_t g = (int64_t)(dc * 2 * spc + (dtop ? 0 : spc) + l) * LEN;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    __stcg(Xs + g + lane + 32 * e, src[lane + 32 * e]);
                    __stcg(Vs + g + lane + 32 * e, src[LEN + lane + 32 * e]);
                }
            }
            grid.sync();
            for (int sl = warp; sl < 2 * spc; sl += 8) {
                const int64_t g = (int64_t)(c * 2 * spc + sl) * LEN;
                double* dst = cur + sl * slot_doubles;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    dst[lane + 32 * e] = __ldcg(Xs + g + lane + 32 * e);
                    dst[LEN + lane + 32 * e] = __ldcg(Vs + g + lane + 32 * e);
                }
            }
            __syncthreads();
            stage ^= 1;
        }
        if (rotated && lane == 0) atomicAdd(counters + sweep, 1);
        grid.sync();
        const int cnt = *((volatile int*)(counters + sweep));
        if (cnt == 0) { ++sweep; break; }
    }
    grid.sync();      // nobody still reads the staging area: the result goes to buffer A with n-row columns
    for (int sl = warp; sl < 2 * spc; sl += 8) {
        const int j = c * 2 * spc + sl;
        const double* src = cur + sl * slot_doubles;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = lane + 32 * e;
            if (i < n) {
                XoA[(int64_t)j * n + i] = src[i];
                VoA[(int64_t)j * n + i] = src[LEN + i];
            }
        }
    }
    if (c == 0 && threadIdx.x == 0) info[0] = sweep;
}

// counters / sweep count of the cooperative engines
__global__ void jacobi_info_reset_kernel(int* __restrict__ info, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    if (threadIdx.x < 66) info[threadIdx.x] = 0;
}

// prepare Xo/Vo for the global engine: Xo = X0 (or G), Vo = V0 (or I)
__global__ void jacobi_global_init_kernel(const double* __restrict__ X0, const double* __restrict__ V0, int n,
                                          double* __restrict__ Xo, double* __restrict__ Vo, int* __restrict__ info,
                                          const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < 66) info[idx] = 0;
    if (idx >= (int64_t)n * n) return;
    const int i = (int)(idx % n), j = (int)(idx / n);
    Xo[idx] = X0[idx];
    Vo[idx] = V0 ? V0[idx] : (i == j ? 1.0 : 0.0);
}

// ---------------------------------------------------------------------------------------------------
// post-processing: lambda_j = v_j . x_j, rank (descending), perm; dummy columns (v == 0) are dropped
// single CTA, 256 threads
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
eig_post_kernel(const double* __restrict__ Xo, const double* __restrict__ Vo, int n, int ncols,
                double* __restrict__ lam_raw, double* __restrict__ lam_sorted, int* __restrict__ perm,
                const int* __restrict__ run_flag, int svd_mode) {
    if (run_flag && run_flag[1] == 0) return;
    extern __shared__ double sl[];          // ncols lam + ncols valid flags (as double)
    double* lam = sl;
    double* valid = sl + ncols;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = warp; j < ncols; j += 8) {
        double dot = 0.0, vv = 0.0;
        for (int i = lane; i < n; i += 32) {
            const double v = Vo[(int64_t)j * n + i];
            const double x = Xo[(int64_t)j * n + i];
            dot = fma(svd_mode ? x : v, x, dot);                   // svd mode: |x_j|^2 (X = K V, K general square)
            vv = fma(v, v, vv);
        }
        dot = warp_sum(dot);
        vv = warp_sum(vv);
        if (svd_mode) dot = sqrt(dot);                             // singular value of K
        if (lane == 0) {
            lam[j] = dot;
            valid[j] = (vv > 0.5) ? 1.0 : 0.0;
            lam_raw[j] = dot;
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < ncols; j += blockDim.x) {
        if (valid[j] == 0.0) continue;
        const double lj = lam[j];
        int rank = 0;
        for (int k = 0; k < ncols; ++k) {
            if (valid[k] == 0.0) continue;
            const double lk = lam[k];
            rank += (lk > lj) || (lk == lj && k < j);
        }
        if (rank < n) {
            perm[rank] = j;
            lam_sorted[rank] = lj;
        }
    }
}

// Vs[:, r] = Vo[:, perm[r]]
__global__ void permute_cols_kernel(const double* __restrict__ Vo, const int* __restrict__ perm, int n,
                                    double* __restrict__ Vs, const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    const int r = blockIdx.x;
    const int j = perm[r];
    for (int i = threadIdx.x; i < n; i += blockDim.x) Vs[(int64_t)r * n + i] = Vo[(int64_t)j * n + i];
}

__global__ void svt_post_kernel(const double* __restrict__ lam, int n, double tau, int nukeA,
                                double* __restrict__ sigma, double* __restrict__ fvec, int* __restrict__ svp,
                                const int* __restrict__ run_flag) {
    if (run_flag && run_flag[1] == 0) return;
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    int local = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double l = lam[i];
        const double sg = l > 0.0 ? sqrt(l) : 0.0;
        sigma[i] = sg;
        const bool keep = sg >= tau;                                   // s.S .>= 1/mu   (src/robustPCA.jl:198)
        local += keep ? 1 : 0;
        // A = U_r diag(S_r - 1/mu) V_r' = W V_r diag((S_r - 1/mu)/S_r) V_r'   (:207-208);  nukeA=false: factor 1
        fvec[i] = keep ? (nukeA ? (sg - tau) / sg : 1.0) : 0.0;
    }
    if (local) atomicAdd(&cnt, local);
    __syncthreads();
    if (threadIdx.x == 0) *svp = cnt;
}


// ---------------------------------------------------------------------------------------------------
// Upper Cholesky factor R (R'R = A) of a small SPD matrix, single CTA, right-looking, the matrix stays in global
// memory (L2 resident).  Used once per solve by the SVD refinement (solver.cu): A = C'C with C = W V diag(1/s) nearly
// orthonormal, so A is close to the identity.  A pivot that has lost all its digits (<= n eps times its original
// value: the column depends on the previous ones, e.g. an exactly rank-deficient W) deflates: its row of R is zero.
// R: n x n column-major, strictly lower part zeroed.  In place: R must hold A on entry.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
chol_upper_kernel(double* __restrict__ R, int n) {
    extern __shared__ double rowj[];            // [n] scaled row j, then [n] original diagonal
    double* d0 = rowj + n;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    for (int i = tid; i < n; i += blockDim.x) d0[i] = R[(int64_t)i * n + i];
    __syncthreads();
    const double epsn = 2.220446049250313e-16 * (double)n;
    for (int j = 0; j < n; ++j) {
        __syncthreads();                         // the trailing update of step j-1 is complete
        const double ajj = R[(int64_t)j * n + j];
        const bool ok = ajj > epsn * d0[j] && d0[j] > 0.0;
        const double piv = ok ? sqrt(ajj) : 0.0;
        const double ipiv = ok ? 1.0 / piv : 0.0;
        __syncthreads();                         // everybody has read the pivot before it is overwritten
        for (int k = j + tid; k < n; k += blockDim.x) {
            const double v = (k == j) ? piv : R[(int64_t)k * n + j] * ipiv;
            rowj[k] = v;
            R[(int64_t)k * n + j] = v;
        }
        __syncthreads();
        if (ok) {
            for (int k = j + 1 + warp; k < n; k += nw) {
                const double rjk = rowj[k];
                double* col = R + (int64_t)k * n;
                for (int i = j + 1 + lane; i <= k; i += 32) col[i] = fma(-rowj[i], rjk, col[i]);
            }
        }
    }
    __syncthreads();
    for (int64_t idx = tid; idx < (int64_t)n * n; idx += blockDim.x) {
        const int i = (int)(idx % n), k = (int)(idx / n);
        if (i > k) R[idx] = 0.0;
    }
}

// B[:, c] = V[:, c] / max(s_c, floor * s_0)   (st_out[c] = the clamped scale)
__global__ void scale_cols_floor_kernel(const double* __restrict__ V, const double* __restrict__ sigma, int n,
                                        double floor_rel, double* __restrict__ B, double* __restrict__ st_out) {
    const int c = blockIdx.x;
    double s = sigma[c];
    const double fl = floor_rel * sigma[0];
    if (!(s > fl)) s = fl;
    const double f = s > 0.0 ? 1.0 / s : 0.0;
    if (threadIdx.x == 0) st_out[c] = s;
    for (int i = threadIdx.x; i < n; i += blockDim.x) B[(int64_t)c * n + i] = V[(int64_t)c * n + i] * f;
}
// B[:, c] = V[:, c] * f[c] for the first `cols` columns (n rows)
__global__ void scale_cols_mulvec_kernel(const double* __restrict__ V, const double* __restrict__ f, int n,
                                         double* __restrict__ B) {
    const int c = blockIdx.x;
    const double s = f[c];
    for (int i = threadIdx.x; i < n; i += blockDim.x) B[(int64_t)c * n + i] = V[(int64_t)c * n + i] * s;
}
// K[:, c] = R[:, c] * st[c]
__global__ void scale_cols_mul_kernel(const double* __restrict__ R, const double* __restrict__ st, int n,
                                      double* __restrict__ K) {
    const int c = blockIdx.x;
    const double s = st[c];
    for (int i = threadIdx.x; i < n; i += blockDim.x) K[(int64_t)c * n + i] = R[(int64_t)c * n + i] * s;
}

template <int E>
cudaError_t launch_cluster(const double* X0, const double* V0, int n, int C, int spc, double tol, int max_sweeps,
                           double* Xo, double* Vo, int* info, const int* run_flag, cudaStream_t st) {
    constexpr int LEN = 32 * E;
    const size_t smem = (size_t)2 * 2 * spc * 2 * LEN * sizeof(double);
    auto kern = jacobi_cluster_block_kernel<E>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (C > 8) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, X0, V0, n, spc, tol, max_sweeps, Xo, Vo, info, run_flag);
}

template <int E>
cudaError_t launch_global(int n, int np, double tol, int max_sweeps, double* Xo, double* Vo, int* info,
                          const int* run_flag, int sm_count, cudaStream_t st) {
    int npairs = np / 2;
    int blocks = (npairs + 7) / 8;
    if (blocks > sm_count) blocks = sm_count;
    if (blocks < 1) blocks = 1;
    void* args[] = {&n, &np, &tol, &max_sweeps, &Xo, &Vo, &info, &run_flag};
    if (n > 32 * E) return cudaLaunchCooperativeKernel((void*)jacobi_global_loop_kernel, dim3(blocks), dim3(256), args, 0, st);
    return cudaLaunchCooperativeKernel((void*)jacobi_global_kernel<E>, dim3(blocks), dim3(256), args, 0, st);
}

}  // namespace

size_t eig_work_doubles(int n) {
    const size_t np = (size_t)n + 34;          // padded column count upper bound
    // X0 (n*n) + Xo (np*n) + Vo (np*n) + lam_raw (np) + perm (n ints -> n doubles) + info (66 ints -> 64 doubles)
    // 256 < n <= 512: + four staging buffers of np slots x 512 doubles for the cooperative block tournament
    const size_t stagew = (n > 256 && n <= 512) ? 4 * ((size_t)n + 64) * 512 : 0;       // up to n + 63 padded columns
    return (size_t)n * n + 2 * np * n + np + n + 64 + 16 + stagew;
}

cudaError_t launch_eigh(const double* G, int n, const double* V0, EigWork w, double* lam, double* Vs,
                        int sm_count, cudaStream_t st, int64_t* launches, const int* run_flag, int svd_mode) {
    cudaError_t e;
    const double tol = 1.0e-15 * (n < 16 ? 4.0 : sqrt((double)n));   // relative orthogonality threshold
    const int max_sweeps = 30;
    const double* X0 = G;
    if (V0) {
        dim3 grid((n + 31) / 32, (n + 31) / 32);
        gemm_small_kernel<<<grid, 256, 0, st>>>(G, V0, n, w.X0);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (launches) *launches += 1;
        X0 = w.X0;
    }
    int ncols;
    if (n <= 256) {
        // seats m >= ceil(n/2); cluster size C in {1,2,4,8,16}, seats per CTA spc <= 8
        const int mneed = (n + 1) / 2;
        int C = 1;
        while (C < 16 && (mneed + C - 1) / C > 8) C *= 2;
        const int spc = (mneed + C - 1) / C;
        ncols = 2 * C * spc;
        if (n <= 32) e = launch_cluster<1>(X0, V0, n, C, spc, tol, max_sweeps, w.Xo, w.Vo, w.info, run_flag, st);
        else if (n <= 64) e = launch_cluster<2>(X0, V0, n, C, spc, tol, max_sweeps, w.Xo, w.Vo, w.info, run_flag, st);
        else if (n <= 128) e = launch_cluster<4>(X0, V0, n, C, spc, tol, max_sweeps, w.Xo, w.Vo, w.info, run_flag, st);
        else e = launch_cluster<8>(X0, V0, n, C, spc, tol, max_sweeps, w.Xo, w.Vo, w.info, run_flag, st);
        if (e != cudaSuccess) return e;
        if (launches) *launches += 1;
    } else if (n <= 512) {
        // cooperative block tournament: C CTAs x 2 half-blocks of spc columns, C * 2 * spc >= n, spc <= 8
        const int mneed = (n + 1) / 2;
        int C = 16;
        while ((mneed + C - 1) / C > 8) C *= 2;
        if (C > sm_count) C = sm_count;
        const int spc = (mneed + C - 1) / C;
        ncols = 2 * C * spc;
        constexpr int LEN = 512;
        const size_t smem = (size_t)2 * spc * 2 * LEN * sizeof(double);
        auto kern = jacobi_coop_block_kernel<16>;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        jacobi_info_reset_kernel<<<1, 96, 0, st>>>(w.info, run_flag);
        // staging buffers live behind the regular work area (eig_work_doubles)
        const size_t nps = (size_t)n + 64;
        double* stg = reinterpret_cast<double*>(w.info) + 64 + 16;
        double* XoA = stg, *VoA = stg + nps * LEN, *XoB = stg + 2 * nps * LEN, *VoB = stg + 3 * nps * LEN;
        double tolv = tol;
        int ms = max_sweeps, nn = n, sp = spc;
        void* args[] = {&X0, &V0, &nn, &sp, &tolv, &ms, &XoA, &VoA, &XoB, &VoB, &w.info, &run_flag};
        if ((e = cudaLaunchCooperativeKernel((void*)kern, dim3(C), dim3(256), args, smem, st)) != cudaSuccess) return e;
        if (launches) *launches += 2;
        // eig_post / permute read n-row columns from XoA / VoA
        eig_post_kernel<<<1, 256, 2 * ncols * sizeof(double), st>>>(XoA, VoA, n, ncols, w.lam_raw, lam, w.perm, run_flag,
                                                                     svd_mode);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        permute_cols_kernel<<<n, 128, 0, st>>>(VoA, w.perm, n, Vs, run_flag);
        if (launches) *launches += 2;
        return cudaGetLastError();
    } else {
        const int np = (n + 1) & ~1;
        ncols = n;
        jacobi_global_init_kernel<<<(unsigned)(((int64_t)n * n + 255) / 256), 256, 0, st>>>(X0, V0, n, w.Xo, w.Vo,
                                                                                           w.info, run_flag);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        e = launch_global<16>(n, np, tol, max_sweeps, w.Xo, w.Vo, w.info, run_flag, sm_count, st);
        if (e != cudaSuccess) return e;
        if (launches) *launches += 2;
    }
    eig_post_kernel<<<1, 256, 2 * ncols * sizeof(double), st>>>(w.Xo, w.Vo, n, ncols, w.lam_raw, lam, w.perm, run_flag,
                                                                 svd_mode);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    permute_cols_kernel<<<n, 128, 0, st>>>(w.Vo, w.perm, n, Vs, run_flag);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

cudaError_t launch_chol_upper(double* R, int n, cudaStream_t st, int64_t* launches) {
    chol_upper_kernel<<<1, 1024, 2 * (size_t)n * sizeof(double), st>>>(R, n);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_scale_cols_floor(const double* V, const double* sigma, int n, double floor_rel, double* B,
                                    double* st_out, cudaStream_t st, int64_t* launches) {
    scale_cols_floor_kernel<<<n, 128, 0, st>>>(V, sigma, n, floor_rel, B, st_out);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_scale_cols_mul(const double* R, const double* sc, int n, double* K, cudaStream_t st,
                                  int64_t* launches) {
    scale_cols_mul_kernel<<<n, 128, 0, st>>>(R, sc, n, K);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_scale_cols_mulvec(const double* V, const double* f, int n, int cols, double* B, cudaStream_t st,
                                     int64_t* launches) {
    if (cols < 1) return cudaSuccess;
    scale_cols_mulvec_kernel<<<cols, 128, 0, st>>>(V, f, n, B);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_gemm_nn(const double* A, const double* B, int n, double* C, cudaStream_t st, int64_t* launches) {
    dim3 grid((n + 31) / 32, (n + 31) / 32);
    gemm_small_kernel<<<grid, 256, 0, st>>>(A, B, n, C);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_svt_post(const double* lam, int n, double tau, int nukeA, double* sigma, double* fvec,
                            int* svp, cudaStream_t st, int64_t* launches, const int* run_flag) {
    svt_post_kernel<<<1, 256, 0, st>>>(lam, n, tau, nukeA, sigma, fvec, svp, run_flag);
    if (launches) *launches += 1;
    return cudaGetLastError();
}

}  // namespace tlsq
