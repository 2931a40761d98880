// stream.cu -- the ALM epilogue as two streaming kernels (used when the SVT input W_k is materialised and svp <= 32):
//
//   alm_stream_kernel  every thread owns one matrix row (FACT: the iterate A is kept FACTORED, A_k = clamp(T_k V_k'),
//                      T: M x 32 -- the dense A is neither read nor written inside the loop):
//                      loop 1  T[i,:] = (W_k[i,:] V_r) .* f      streaming read of W, svp FMAs per element
//                      loop 2  one coalesced pass over D, A_{k-1}, Y_{k-1}:
//                        A_k = clamp(sum_c T[i,c] V[j,c])                         src/robustPCA.jl:205-219
//                        E_k = soft_th((D - A_{k-1}) + Y_{k-1}/mu, lambda/mu)     :188-191
//                        Z = (D - A_k) - E_k ;  Y_k = Y_{k-1} + mu Z ;  ||Z||_F^2 :221-222, 225
//                        W_{k+1} = (D - E_{k+1}) + Y_k/mu_{k+1}                   :188-192 of the NEXT iteration
//                      and writes A_k, Y_k, W_{k+1} (E_k only on request).
// Compared with the fused tile kernel (epilogue.cu) this moves one extra S of traffic (W is read by tproj) but both
// kernels are pure streams with every thread owning one row: 128-byte coalesced column segments, no shared-memory
// staging of the data, no intra-CTA phases -- the memory system sees a STREAM-like access pattern.
// The low-rank reconstruction costs svp FP64 FMAs per element, which the otherwise idle FP64 pipe absorbs.
#include "kernels.h"

namespace tlsq {

namespace {

// sum_c t[c] * v[c] with v read from shared memory as 16-byte vectors (RP is a multiple of 8, v is 16-byte aligned)
template <int RP>
__device__ __forceinline__ double dot_rp(const double (&t)[RP > 0 ? RP : 1], const double* __restrict__ v) {
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < RP; c += 2) {
        const double2 vv = *reinterpret_cast<const double2*>(v + c);
        acc = fma(t[c], vv.x, acc);
        acc = fma(t[c + 1], vv.y, acc);
    }
    return acc;
}

// PH: 0 = both loops in one kernel; 1 = only T = (W V_r) .* f (written to a.Tn); 2 = only the element-wise pass (T_k read
// back from a.Tn).  FACT at a rank above 0 always runs the split form (1 then 2): each loop at a higher occupancy.
template <int RP, bool HANKEL, bool FACT, int PH>
__global__ void __launch_bounds__(128)
alm_stream_kernel(const EpiArgs a, const double* __restrict__ W, int svp_host, const int* __restrict__ svp_dev) {
    static_assert(!(FACT && PH == 0 && RP > 0), "FACT at a rank above 0 runs the split form (T_{k-1} is loaded by PH 2)");
    // Rank of this iteration: either known on the host, or (speculative launch, solver.cu) read from the device scalar
    // the eigen step just wrote.  The launch was specialised on a GUESS of the rank; if the actual rank does not fit
    // the guess the whole grid returns before touching anything and the host relaunches with the right RP.
    const int svp = svp_dev ? __ldg(svp_dev) : svp_host;
    if (svp > RP) return;
    extern __shared__ double Vsm[];            // [NC][RP]  (+ [NC][RP] of V_{k-1} when FACT)
    __shared__ double fsm[RP > 0 ? RP : 1];
    const int N = (int)a.N;
    // column range of this launch: all N columns, or (PH == 2 only, large N: the V rows of all columns do not fit in
    // shared memory) the chunk [c0, c1)
    const int cb = a.c1 > 0 ? a.c0 : 0, ce = a.c1 > 0 ? a.c1 : N, NC = ce - cb;
    double* Vpm = Vsm + (size_t)NC * RP;
    if (threadIdx.x < RP) fsm[threadIdx.x] = (int)threadIdx.x < svp ? __ldg(a.fvec + threadIdx.x) : 0.0;
    for (int idx = threadIdx.x; idx < NC * RP; idx += blockDim.x) {
        const int j = idx % NC, c = idx / NC;
        Vsm[j * RP + c] = c < svp ? __ldg(a.Vs + (int64_t)c * N + cb + j) : 0.0;
        if (FACT && PH != 1) Vpm[j * RP + c] = c < a.svp_prev ? __ldg(a.Vp + (int64_t)c * N + cb + j) : 0.0;
    }
    __syncthreads();
    double zz = 0.0;
    constexpr int UB = 4;                      // columns whose loads are issued together
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < a.M;
         row += (int64_t)gridDim.x * blockDim.x) {
        // ---- T[row, :] = f .* (W[row, :] V_r): one streaming read of the materialised SVT input ----------------
        // (software pipelined: the loads of the next column batch are in flight while the current one is consumed)
        double tr[RP > 0 ? RP : 1];
        double tp[RP > 0 ? RP : 1];
#pragma unroll
        for (int c = 0; c < RP; ++c) tr[c] = 0.0;
        if (RP > 0 && PH == 2) {
#pragma unroll
            for (int c = 0; c < RP; ++c) {
                tr[c] = c < svp ? __ldg(a.Tn + (int64_t)c * a.M + row) : 0.0;
                tp[c] = c < a.svp_prev ? __ldg(a.Tp + (int64_t)c * a.M + row) : 0.0;
            }
        }
        if (RP > 0 && PH != 2) {
            constexpr int UW = 8;
            double wv[UW], wn[UW];
#pragma unroll
            for (int u = 0; u < UW; ++u) wv[u] = u < N ? __ldg(W + (int64_t)u * a.ldw + row) : 0.0;
            for (int j0 = 0; j0 < N; j0 += UW) {
#pragma unroll
                for (int u = 0; u < UW; ++u) {
                    const int j = j0 + UW + u;
                    wn[u] = j < N ? __ldg(W + (int64_t)j * a.ldw + row) : 0.0;
                }
#pragma unroll
                for (int u = 0; u < UW; ++u) {
                    const int j = j0 + u < N ? j0 + u : N - 1;
                    const double* v = Vsm + j * RP;
#pragma unroll
                    for (int c = 0; c < RP; c += 2) {
                        const double2 vv = *reinterpret_cast<const double2*>(v + c);
                        tr[c] = fma(wv[u], vv.x, tr[c]);
                        tr[c + 1] = fma(wv[u], vv.y, tr[c + 1]);
                    }
                }
#pragma unroll
                for (int u = 0; u < UW; ++u) wv[u] = wn[u];
            }
#pragma unroll
            for (int c = 0; c < RP; ++c) tr[c] *= fsm[c];
            if (FACT) {
#pragma unroll
                for (int c = 0; c < RP; ++c) a.Tn[(int64_t)c * a.M + row] = tr[c];
            }
        }
        if (PH == 1) continue;
        double dv[UB], av[UB], yv[UB], dn[UB], an_[UB], yn_[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            dv[u] = av[u] = yv[u] = 0.0;
            if (cb + u < ce) {
                const int64_t off = (int64_t)(cb + u) * a.ldw + row;
                dv[u] = src_at<HANKEL>(a.D, row, cb + u);
                if (!FACT) av[u] = __ldg(a.Ap + off);
                yv[u] = __ldg(a.Yp + off);
            }
        }
        for (int j0 = cb; j0 < ce; j0 += UB) {
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int j = j0 + UB + u;
                dn[u] = an_[u] = yn_[u] = 0.0;
                if (j < ce) {
                    const int64_t off = (int64_t)j * a.ldw + row;
                    dn[u] = src_at<HANKEL>(a.D, row, j);
                    if (!FACT) an_[u] = __ldg(a.Ap + off);
                    yn_[u] = __ldg(a.Yp + off);
                }
            }
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int j = j0 + u;
                if (j < ce) {
                    const int64_t off = (int64_t)j * a.ldw + row;
                    const double d = dv[u], yp = yv[u];
                    double an = 0.0, ap = 0.0;
                    if (RP > 0) an = dot_rp<RP>(tr, Vsm + (j - cb) * RP);
                    if (a.nonnegA) an = (__double_as_longlong(an) > 0) ? an : 0.0;   // A .= max.(A, 0)   :218
                    if (FACT) {                                                       // A_{k-1} from its factors
                        if (RP > 0) ap = dot_rp<RP>(tp, Vpm + (j - cb) * RP);
                        if (a.nonnegA) ap = (__double_as_longlong(ap) > 0) ? ap : 0.0;
                    } else {
                        ap = av[u];
                    }
                    double e, w;
                    alm_ew(d, ap, yp, a.im, a.eps, a.nonnegE, e, w);
                    const double z = __dsub_rn(__dsub_rn(d, an), e);                  // @. Z = D - A - E  :221
                    const double yn = __dadd_rn(yp, __dmul_rn(a.mu, z));              // @. Y = Y + mu*Z   :222
                    zz = fma(z, z, zz);
                    if (!FACT) a.An[off] = an;
                    a.Yn[off] = yn;
                    if (a.Eout) a.Eout[off] = e;
                    if (a.Zout) a.Zout[off] = z;
                    double e2, w2;
                    alm_ew(d, an, yn, a.im_next, a.eps_next, a.nonnegE, e2, w2);      // SVT input of iteration k+1
                    a.Wn[off] = w2;
                }
            }
#pragma unroll
            for (int u = 0; u < UB; ++u) { dv[u] = dn[u]; av[u] = an_[u]; yv[u] = yn_[u]; }
        }
    }
    __shared__ double red[4];
    zz = warp_sum(zz);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = zz;
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(a.zz, red[0] + red[1] + red[2] + red[3]);
}

// A = clamp(T V')  /  Z = (D - A_k) - E_k with both iterates factored (rare paths: outputs, missed Z prediction)
template <int RP, bool HANKEL, int ZMODE>
__global__ void __launch_bounds__(128)
fact_dense_kernel(const EpiArgs a, const double* __restrict__ T, const double* __restrict__ V, int svp,
                  double* __restrict__ out) {
    extern __shared__ double Vsm[];
    const int N = (int)a.N;
    const int cb = a.c1 > 0 ? a.c0 : 0, ce = a.c1 > 0 ? a.c1 : N, NC = ce - cb;      // column chunk of this launch
    double* Vpm = Vsm + (size_t)NC * RP;
    for (int idx = threadIdx.x; idx < NC * RP; idx += blockDim.x) {
        const int j = idx % NC, c = idx / NC;
        Vsm[j * RP + c] = c < svp ? __ldg(V + (int64_t)c * N + cb + j) : 0.0;
        if (ZMODE) Vpm[j * RP + c] = c < a.svp_prev ? __ldg(a.Vp + (int64_t)c * N + cb + j) : 0.0;
    }
    __syncthreads();
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < a.M;
         row += (int64_t)gridDim.x * blockDim.x) {
        double tr[RP > 0 ? RP : 1], tp[(ZMODE && RP > 0) ? RP : 1];
#pragma unroll
        for (int c = 0; c < RP; ++c) {
            tr[c] = c < svp ? __ldg(T + (int64_t)c * a.M + row) : 0.0;
            if (ZMODE) tp[c] = c < a.svp_prev ? __ldg(a.Tp + (int64_t)c * a.M + row) : 0.0;
        }
        for (int j = cb; j < ce; ++j) {
            const int64_t off = (int64_t)j * a.ldw + row;
            double an = 0.0;
            const double* v = Vsm + (j - cb) * RP;
#pragma unroll
            for (int c = 0; c < RP; ++c) an = fma(tr[c], v[c], an);
            if (a.nonnegA) an = (__double_as_longlong(an) > 0) ? an : 0.0;
            if (ZMODE == 0) { out[off] = an; continue; }
            double ap = 0.0;
            const double* vp = Vpm + (j - cb) * RP;
#pragma unroll
            for (int c = 0; c < RP; ++c) ap = fma(tp[c], vp[c], ap);
            if (a.nonnegA) ap = (__double_as_longlong(ap) > 0) ? ap : 0.0;
            const double d = src_at<HANKEL>(a.D, row, j);
            double e, w;
            alm_ew(d, ap, __ldg(a.Yp + off), a.im, a.eps, a.nonnegE, e, w);
            if (ZMODE == 1) {
                out[off] = __dsub_rn(__dsub_rn(d, an), e);
            } else {                                    // final outputs of the solve (:238): A_k, E_k and the last W
                if (a.An) a.An[off] = an;
                if (a.Eout) a.Eout[off] = e;
                if (out) out[off] = w;
            }
        }
    }
}

// padded rank of the specialised kernels: 0, 4, 8, 12, 16, 24, 32
inline int rp_of(int svp) { return svp <= 16 ? ((svp + 3) & ~3) : ((svp + 7) & ~7); }

// columns per launch so that `copies` blocks of [NC][RP] doubles fit in shared memory (all N when they do)
inline int chunk_cols(int64_t N, int rp, int copies) {
    if (rp == 0) return (int)N;
    const int64_t fit = ((int64_t)200 * 1024 / ((int64_t)rp * 8 * copies)) & ~(int64_t)7;
    return (int)(N <= fit ? N : fit);
}

// B (N x RP) = V_r diag(f): the right factor of T = (W V_r) .* f as a GEMM operand (rank read from the device)
__global__ void __launch_bounds__(256)
build_vf_kernel(const double* __restrict__ Vs, const double* __restrict__ fvec, const int* __restrict__ svp_dev,
                int svp_host, int N, int RP, double* __restrict__ B) {
    const int svp = svp_dev ? __ldg(svp_dev) : svp_host;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < N * RP; idx += gridDim.x * blockDim.x) {
        const int c = idx / N;
        B[idx] = (c < svp && svp <= RP) ? __ldg(Vs + idx) * __ldg(fvec + c) : 0.0;
    }
}

template <int RP>
cudaError_t launch_stream_rp(const EpiArgs& a, const double* W, int svp, const int* svp_dev, bool hankel, int sm_count,
                             cudaStream_t st) {
    const bool fact = a.Tn != nullptr;
    int64_t blocks = (a.M + 127) / 128;
    int64_t cap = (int64_t)sm_count * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    cudaError_t e = cudaSuccess;
#define TLSQ_STREAM_LAUNCH(H, F, PH, SM)                                                                          \
    do {                                                                                                          \
        auto kern = alm_stream_kernel<RP, H, F, PH>;                                                              \
        const size_t smem_ = (SM);                                                                                \
        if (smem_ > 32 * 1024) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_); \
        if (e == cudaSuccess) kern<<<(unsigned)blocks, 128, smem_, st>>>(a, W, svp, svp_dev);                     \
    } while (0)
    // TMA-staged kernels (stream_tma.cu) whenever the shape allows them; the register-prefetch kernels below remain for
    // small / oddly aligned problems, the dense iterate and the column-chunked large-N form
    if (fact && RP >= 4 && stream_tma_eligible(a, W, RP, hankel))
        return launch_stream_tma(a, W, RP, svp, svp_dev, hankel, sm_count, st);
    const int nc = chunk_cols(a.N, RP, fact ? 2 : 1);
    if (nc < a.N) {
        // large N: T = W (V_r diag(f)) as a DMMA GEMM (a.vf_work: N x 32 scratch), then the element-wise pass per
        // column chunk with the chunk's rows of V_{k-1}, V_k in shared memory
        if (!fact || !a.vf_work) return cudaErrorInvalidValue;
        build_vf_kernel<<<64, 256, 0, st>>>(a.Vs, a.fvec, svp_dev, svp, (int)a.N, RP, a.vf_work);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if ((e = launch_gemm_any(W, a.M, (int)a.N, a.ldw, a.vf_work, RP, a.Tn, st, nullptr)) != cudaSuccess) return e;
        for (int c0 = 0; c0 < a.N && e == cudaSuccess; c0 += nc) {
            EpiArgs ac = a;
            ac.c0 = c0;
            ac.c1 = (int)(c0 + nc < a.N ? c0 + nc : a.N);
            const size_t smc = (size_t)2 * (ac.c1 - ac.c0) * RP * sizeof(double);
            auto kern_h = alm_stream_kernel<RP, true, true, 2>;
            auto kern_d = alm_stream_kernel<RP, false, true, 2>;
            if (smc > 32 * 1024)
                e = cudaFuncSetAttribute(hankel ? kern_h : kern_d, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smc);
            if (e != cudaSuccess) break;
            if (hankel) kern_h<<<(unsigned)blocks, 128, smc, st>>>(ac, W, svp, svp_dev);
            else kern_d<<<(unsigned)blocks, 128, smc, st>>>(ac, W, svp, svp_dev);
        }
        if (e != cudaSuccess) return e;
        return cudaGetLastError();
    }
    const size_t sm1 = (size_t)a.N * RP * sizeof(double);
    if (!fact) {
        if (hankel) TLSQ_STREAM_LAUNCH(true, false, 0, sm1); else TLSQ_STREAM_LAUNCH(false, false, 0, sm1);
    } else if constexpr (RP == 0) {
        if (hankel) TLSQ_STREAM_LAUNCH(true, true, 0, 2 * sm1); else TLSQ_STREAM_LAUNCH(false, true, 0, 2 * sm1);
    } else {
        if (hankel) { TLSQ_STREAM_LAUNCH(true, true, 1, sm1); if (e == cudaSuccess) TLSQ_STREAM_LAUNCH(true, true, 2, 2 * sm1); }
        else        { TLSQ_STREAM_LAUNCH(false, true, 1, sm1); if (e == cudaSuccess) TLSQ_STREAM_LAUNCH(false, true, 2, 2 * sm1); }
    }
#undef TLSQ_STREAM_LAUNCH
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

template <int RP, int ZMODE>
cudaError_t launch_fact_rp(const EpiArgs& a, const double* T, const double* V, int svp, bool hankel, double* out,
                           int sm_count, cudaStream_t st) {
    int64_t blocks = (a.M + 127) / 128;
    int64_t cap = (int64_t)sm_count * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    cudaError_t e = cudaSuccess;
    const int nc = chunk_cols(a.N, RP, ZMODE ? 2 : 1);           // all N columns unless V does not fit in shared memory
    for (int c0 = 0; c0 < a.N && e == cudaSuccess; c0 += nc) {
        EpiArgs ac = a;
        if (nc < a.N) { ac.c0 = c0; ac.c1 = (int)(c0 + nc < a.N ? c0 + nc : a.N); }
        const size_t smem = (size_t)(nc < a.N ? ac.c1 - ac.c0 : a.N) * RP * sizeof(double) * (ZMODE ? 2 : 1);
        if (hankel) {
            auto kern = fact_dense_kernel<RP, true, ZMODE>;
            if (smem > 32 * 1024) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) kern<<<(unsigned)blocks, 128, smem, st>>>(ac, T, V, svp, out);
        } else {
            auto kern = fact_dense_kernel<RP, false, ZMODE>;
            if (smem > 32 * 1024) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) kern<<<(unsigned)blocks, 128, smem, st>>>(ac, T, V, svp, out);
        }
    }
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

}  // namespace

bool stream_factored_fits(int64_t N, int svp, int svp_prev) {
    (void)N;        // any N: when the V blocks do not fit in shared memory the element-wise pass runs per column chunk
    return svp <= kStreamMaxRank && svp_prev <= kStreamMaxRank;
}

int stream_rank_pad(int svp, int svp_prev, bool fact) { return rp_of(fact && svp_prev > svp ? svp_prev : svp); }

cudaError_t launch_stream_epilogue(const EpiArgs& a, const double* W, int svp, bool hankel, int sm_count,
                                   cudaStream_t st, int64_t* launches, bool svp_on_device) {
    cudaError_t e;
    const bool fact = a.Tn != nullptr;
    const int rp = rp_of(fact && a.svp_prev > svp ? a.svp_prev : svp);
    const int* svp_dev = svp_on_device ? a.svp : nullptr;
    switch (rp) {
        case 0:  e = launch_stream_rp<0>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        case 4:  e = launch_stream_rp<4>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        case 8:  e = launch_stream_rp<8>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        case 12: e = launch_stream_rp<12>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        case 16: e = launch_stream_rp<16>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        case 24: e = launch_stream_rp<24>(a, W, svp, svp_dev, hankel, sm_count, st); break;
        default: e = launch_stream_rp<32>(a, W, svp, svp_dev, hankel, sm_count, st); break;
    }
    if (launches) *launches += (fact && rp > 0) ? 2 : 1;
    return e;
}

cudaError_t launch_fact_to_dense(const double* T, const double* V, int svp, int64_t M, int64_t N, int nonnegA,
                                 double* A, int sm_count, cudaStream_t st, int64_t* launches) {
    EpiArgs a = {};
    a.M = M; a.N = N; a.ldw = M; a.nonnegA = nonnegA;
    cudaError_t e;
    switch (rp_of(svp)) {
        case 0:  e = launch_fact_rp<0, 0>(a, T, V, svp, false, A, sm_count, st); break;
        case 4:  e = launch_fact_rp<4, 0>(a, T, V, svp, false, A, sm_count, st); break;
        case 8:  e = launch_fact_rp<8, 0>(a, T, V, svp, false, A, sm_count, st); break;
        case 12: e = launch_fact_rp<12, 0>(a, T, V, svp, false, A, sm_count, st); break;
        case 16: e = launch_fact_rp<16, 0>(a, T, V, svp, false, A, sm_count, st); break;
        case 24: e = launch_fact_rp<24, 0>(a, T, V, svp, false, A, sm_count, st); break;
        default: e = launch_fact_rp<32, 0>(a, T, V, svp, false, A, sm_count, st); break;
    }
    if (launches) *launches += 1;
    return e;
}

// a.{D, Yp, Tp, Vp, svp_prev, im, eps, nonnegA, nonnegE, M, N, ldw} describe iteration k's inputs; (a.Tn, a.Vs, svp) = A_k
cudaError_t launch_z_from_factors(const EpiArgs& a, bool hankel, int svp, double* Z, int sm_count, cudaStream_t st,
                                  int64_t* launches) {
    cudaError_t e;
    const int rp = rp_of(a.svp_prev > svp ? a.svp_prev : svp);
    switch (rp) {
        case 0:  e = launch_fact_rp<0, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        case 4:  e = launch_fact_rp<4, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        case 8:  e = launch_fact_rp<8, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        case 12: e = launch_fact_rp<12, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        case 16: e = launch_fact_rp<16, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        case 24: e = launch_fact_rp<24, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
        default: e = launch_fact_rp<32, 1>(a, a.Tn, a.Vs, svp, hankel, Z, sm_count, st); break;
    }
    if (launches) *launches += 1;
    return e;
}

// final outputs from the factored iterates in ONE pass: a.An <- A_k (a.Tn, a.Vs, svp), a.Eout <- E_k, Wout <- W_k (the
// last SVT input, for U); a.{Tp, Vp, svp_prev, Yp, im, eps} describe iteration k's inputs.  Null outputs are skipped.
cudaError_t launch_final_from_factors(const EpiArgs& a, bool hankel, int svp, double* Wout, int sm_count,
                                      cudaStream_t st, int64_t* launches) {
    cudaError_t e;
    const int rp = rp_of(a.svp_prev > svp ? a.svp_prev : svp);
    switch (rp) {
        case 0:  e = launch_fact_rp<0, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        case 4:  e = launch_fact_rp<4, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        case 8:  e = launch_fact_rp<8, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        case 12: e = launch_fact_rp<12, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        case 16: e = launch_fact_rp<16, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        case 24: e = launch_fact_rp<24, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
        default: e = launch_fact_rp<32, 2>(a, a.Tn, a.Vs, svp, hankel, Wout, sm_count, st); break;
    }
    if (launches) *launches += 1;
    return e;
}

}  // namespace tlsq
